// pq_stats.cu -- C-ABI entry points for the statistics kernels (SURVEY.md 8 rows a1, a3).
#include "pq_stats_kernels.cuh"

namespace {

constexpr int kHistCopies = 1;   // privatised sub-histograms per CTA (see DESIGN.md, histogram)

int build_table(pq::SegTable &t, const float *const *xs, const uint64_t *ns, const float *params, int k)
{
    if (k < 0 || (k > 0 && (!xs || !ns))) return PQ_EINVAL;
    if (k > PQ_MAX_SEGMENTS) return PQ_ETOOMANY;
    unsigned long long total = 0;
    for (int i = 0; i < k; ++i) {
        if (ns[i] && !xs[i]) return PQ_EINVAL;
        if (((unsigned long long)xs[i] & 3ull) != 0) return PQ_EALIGN;
        t.ptr[i] = xs[i];
        t.n[i] = ns[i];
        t.param[i] = params ? params[i] : 0.0f;
        total += pq::seg_num_chunks(xs[i], ns[i]);
        if (total > 0xffffffffull) return PQ_EUNSUPPORTED;
        t.chunk_end[i] = (unsigned int)total;
    }
    t.k = k;
    t.total_chunks = (unsigned int)total;
    return PQ_OK;
}

unsigned int grid_for(unsigned int total_chunks, int ctas_per_sm)
{
    unsigned int g = (unsigned int)(pq::kNumSMs * ctas_per_sm);
    return total_chunks < g ? total_chunks : g;
}

}  // namespace

extern "C" int pq_absmax_multi_f32(const float *const *xs_host, const uint64_t *ns_host, int k,
                                   uint32_t *max_bits, pq_stream_t stream)
{
    if (k == 0) return PQ_OK;
    if (!max_bits) return PQ_EINVAL;
    pq::SegTable t;
    int rc = build_table(t, xs_host, ns_host, nullptr, k);
    if (rc != PQ_OK) return rc;
    pq::absmax_multi_kernel<<<grid_for(t.total_chunks, 8), pq::kStatThreads, 0, (cudaStream_t)stream>>>(
        t, max_bits);
    return (int)cudaGetLastError();
}

namespace {
// m = ceil(2^(31+l) / d), l = ceil(log2 d): floor(n * m / 2^(31+l)) == n / d for every n < 2^31
void magic31(unsigned int d, unsigned int *m, int *s)
{
    int l = 0;
    while ((1ull << l) < d) ++l;
    *s = 31 + l;
    *m = (unsigned int)(((1ull << *s) + d - 1) / d);
}
}  // namespace

extern "C" int pq_absmax_per_channel_f32(const float *x, uint64_t outer, int channels, uint64_t inner,
                                         uint32_t *max_bits, pq_stream_t stream)
{
    if (channels < 0) return PQ_EINVAL;
    if (outer == 0 || channels == 0 || inner == 0) return PQ_OK;
    if (!x || !max_bits) return PQ_EINVAL;
    if (((unsigned long long)x & 3ull) != 0) return PQ_EALIGN;
    if (channels > 8192 || inner >= (1ull << 31) - (1ull << 14) || outer * (uint64_t)channels >= (1ull << 31))
        return PQ_EUNSUPPORTED;
    // small planes, many images: the periodic variant (one float4 column per thread, see the kernel)
    const uint64_t per_img = (uint64_t)channels * inner;
    if (inner < 784 && outer >= 16 && (per_img & 3) == 0 && per_img / 4 < (1ull << 31) && outer < (1ull << 31) &&
        ((unsigned long long)x & 15ull) == 0) {
        const unsigned int vec_per_img = (unsigned int)(per_img / 4);
        const unsigned int gx = (vec_per_img + pq::kStatThreads - 1) / pq::kStatThreads;
        unsigned long long gy = ((unsigned long long)pq::kNumSMs * 8 + gx - 1) / gx;        // ~8 CTAs per SM in total
        if (gy > outer / 2) gy = outer / 2;                                               // >= 2 images per thread
        if (gy > 65535) gy = 65535;
        if (gy < 1) gy = 1;
        pq::absmax_periodic_kernel<<<dim3(gx, (unsigned int)gy), pq::kStatThreads, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const float4 *>(x), vec_per_img, (unsigned int)outer, (unsigned int)inner, max_bits);
        return (int)cudaGetLastError();
    }
    pq::ChannelGeom g;
    g.total = outer * (uint64_t)channels * inner;
    g.inner = (unsigned int)inner;
    g.channels = (unsigned int)channels;
    magic31(g.inner, &g.m_inner, &g.s_inner);
    magic31(g.channels, &g.m_chan, &g.s_chan);
    unsigned long long head = ((16ull - ((unsigned long long)x & 15ull)) & 15ull) >> 2;
    if (head > g.total) head = g.total;
    const unsigned long long nvec = (g.total - head) >> 2;
    const unsigned int tail = (unsigned int)(g.total - head - (nvec << 2));
    unsigned long long chunks = (nvec + pq::kChunkVecs - 1) / pq::kChunkVecs;
    if (chunks == 0) chunks = 1;
    if (chunks > 0xffffffffull) return PQ_EUNSUPPORTED;
    pq::absmax_per_channel_kernel<<<grid_for((unsigned int)chunks, 8), pq::kStatThreads, (size_t)channels * 4,
                                    (cudaStream_t)stream>>>(x, g, (unsigned int)head, nvec, tail,
                                                            (unsigned int)chunks, max_bits);
    return (int)cudaGetLastError();
}

namespace {
bool aligned16(const void *p) { return (((unsigned long long)p) & 15ull) == 0; }

int launch_epilogue(pq::EpiArgs &p, int mode, cudaStream_t stream)
{
    const unsigned long long nvec = p.n >> 2;
    if (nvec >= (1ull << 31) || (mode == pq::EPI_BIAS1 && p.n >= (1ull << 31))) return PQ_EUNSUPPORTED;
    magic31(p.hw, &p.m_hw, &p.s_hw);
    magic31(p.channels, &p.m_chan, &p.s_chan);
    unsigned long long blocks = (nvec / pq::kEpiUnroll + pq::kStatThreads - 1) / pq::kStatThreads;
    if (blocks > (unsigned long long)pq::kNumSMs * 8) blocks = (unsigned long long)pq::kNumSMs * 8;
    if (blocks == 0) blocks = 1;
    const unsigned int g = (unsigned int)blocks;
    if (mode == pq::EPI_BIAS4) pq::epilogue_kernel<pq::EPI_BIAS4><<<g, pq::kStatThreads, 0, stream>>>(p);
    else if (mode == pq::EPI_BIAS1) pq::epilogue_kernel<pq::EPI_BIAS1><<<g, pq::kStatThreads, 0, stream>>>(p);
    else pq::epilogue_kernel<pq::EPI_ADD><<<g, pq::kStatThreads, 0, stream>>>(p);
    return (int)cudaGetLastError();
}
}  // namespace

extern "C" int pq_conv_epilogue_f32(float *y, const float *bias, int N, int C, uint64_t hw, float *relu_out,
                                    uint32_t *max_slot, pq_stream_t stream)
{
    if (N < 0 || C <= 0) return PQ_EINVAL;
    if (N == 0 || hw == 0) return PQ_OK;
    if (!y || !bias || relu_out == y) return PQ_EINVAL;
    if (!aligned16(y) || !aligned16(relu_out) || (((unsigned long long)bias) & 3ull)) return PQ_EALIGN;
    if (hw >= (1ull << 31) || (uint64_t)N * (uint64_t)C >= (1ull << 31)) return PQ_EUNSUPPORTED;
    pq::EpiArgs p = {};
    p.a = y;
    p.b = bias;
    p.out = y;
    p.relu_out = relu_out;
    p.max_slot = max_slot;
    p.n = (uint64_t)N * (uint64_t)C * hw;
    p.channels = (unsigned int)C;
    const int mode = (hw & 3) == 0 ? pq::EPI_BIAS4 : pq::EPI_BIAS1;
    p.hw = (unsigned int)(mode == pq::EPI_BIAS4 ? hw / 4 : hw);
    return launch_epilogue(p, mode, (cudaStream_t)stream);
}

extern "C" int pq_eltwise_add_f32(const float *a, const float *b, float *z, size_t n, float *relu_out,
                                  uint32_t *max_slot, pq_stream_t stream)
{
    if (n == 0) return PQ_OK;
    if (!a || !b || !z || z == a || z == b || relu_out == a || relu_out == b || relu_out == z) return PQ_EINVAL;
    if (!aligned16(a) || !aligned16(b) || !aligned16(z) || !aligned16(relu_out)) return PQ_EALIGN;
    pq::EpiArgs p = {};
    p.a = a;
    p.b = b;
    p.out = z;
    p.relu_out = relu_out;
    p.max_slot = max_slot;
    p.n = n;
    p.hw = 1;
    p.channels = 1;
    return launch_epilogue(p, pq::EPI_ADD, (cudaStream_t)stream);
}

extern "C" int pq_hist2048_multi_f32(const float *const *xs_host, const uint64_t *ns_host,
                                     const float *intervals_host, int k, long long *hist,
                                     pq_stream_t stream)
{
    if (k == 0) return PQ_OK;
    if (!hist || !intervals_host) return PQ_EINVAL;
    for (int i = 0; i < k; ++i)
        if (!(intervals_host[i] > 0.0f)) return PQ_EINVAL;   // also rejects NaN
    pq::SegTable t;
    int rc = build_table(t, xs_host, ns_host, intervals_host, k);
    if (rc != PQ_OK) return rc;
    constexpr size_t smem = pq::hist_smem_bytes(kHistCopies);
    auto kern = pq::hist_multi_kernel<kHistCopies>;
    static bool attr_set = false;
    if (!attr_set) {
        PQ_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    const int ctas_per_sm = (int)((200 * 1024) / smem) < 8 ? (int)((200 * 1024) / smem) : 8;
    kern<<<grid_for(t.total_chunks, ctas_per_sm), pq::kStatThreads, smem, (cudaStream_t)stream>>>(
        t, reinterpret_cast<unsigned long long *>(hist));
    return (int)cudaGetLastError();
}

extern "C" int pq_hist_multi_f32(const float *const *xs_host, const uint64_t *ns_host, const float *intervals_host,
                                 int k, int nbins, long long *hist, pq_stream_t stream)
{
    if (nbins == PQ_HIST_BINS) return pq_hist2048_multi_f32(xs_host, ns_host, intervals_host, k, hist, stream);
    if (nbins < 1) return PQ_EINVAL;
    if (nbins > PQ_HIST_BINS_MAX) return PQ_EUNSUPPORTED;
    if (k == 0) return PQ_OK;
    if (!hist || !intervals_host) return PQ_EINVAL;
    for (int i = 0; i < k; ++i)
        if (!(intervals_host[i] > 0.0f)) return PQ_EINVAL;
    pq::SegTable t;
    int rc = build_table(t, xs_host, ns_host, intervals_host, k);
    if (rc != PQ_OK) return rc;
    const size_t smem = (size_t)nbins * 4;
    static bool attr_set = false;
    if (!attr_set) {
        PQ_CUDA_TRY(cudaFuncSetAttribute(pq::hist_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         PQ_HIST_BINS_MAX * 4));
        attr_set = true;
    }
    int ctas_per_sm = (int)((200 * 1024) / (smem + 1024));
    ctas_per_sm = ctas_per_sm < 1 ? 1 : (ctas_per_sm > 8 ? 8 : ctas_per_sm);
    pq::hist_generic_kernel<<<grid_for(t.total_chunks, ctas_per_sm), pq::kStatThreads, smem, (cudaStream_t)stream>>>(
        t, nbins, reinterpret_cast<unsigned long long *>(hist));
    return (int)cudaGetLastError();
}
