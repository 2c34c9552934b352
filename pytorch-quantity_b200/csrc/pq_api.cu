// pq_api.cu -- library identity and error strings.
#include "pq_common.cuh"

extern "C" int pq_version(void) { return PQ_VERSION; }

extern "C" const char *pq_error_string(int code)
{
    switch (code) {
        case PQ_OK: return "ok";
        case PQ_EINVAL: return "PQ_EINVAL: invalid argument (null pointer, bad size or aliasing)";
        case PQ_EUNSUPPORTED: return "PQ_EUNSUPPORTED: shape or parameter not implemented by the sm_100a kernels";
        case PQ_EALIGN: return "PQ_EALIGN: pointer alignment";
        case PQ_ETOOMANY: return "PQ_ETOOMANY: more than PQ_MAX_SEGMENTS tensors in one call";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "unknown pq error";
}
