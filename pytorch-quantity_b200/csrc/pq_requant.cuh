// pq_requant.cuh -- the int8 epilogue arithmetic and launch plumbing shared by the convolution kernels of
// pq_gemm_s8.cu (tensor-core GEMM / implicit GEMM) and pq_depthwise.cu (depthwise stencil):
//   RightShift -> BiasAdd -> Sp (new_quantity_op.py:11-44, 71-101) on int32 accumulators, the saturating int8
//   pack, and programmatic dependent launch.
#pragma once
#include <cstdlib>

#include "pq_common.cuh"

namespace pq {

// Programmatic dependent launch: every kernel here is launched with programmaticStreamSerializationAllowed, lets its
// successor start as soon as this grid's CTAs have been scheduled (launch_dependents) and touches global memory only
// after its predecessor has completed and flushed (wait).  A CTA of the next kernel lands on an SM as soon as this
// kernel's CTA there has exited (one CTA per SM: shared memory), so its barrier / TMEM / tensor-map set-up overlaps the
// tail of this kernel instead of following the launch latency.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// sat_s8(y0) | sat_s8(y1) << 8 | sat_s8(y2) << 16 | sat_s8(y3) << 24   (two I2IP.S8.S32.SAT)
__device__ __forceinline__ uint32_t pack4_sat_s8(int y0, int y1, int y2, int y3)
{
    uint32_t t, w;
    asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(y3), "r"(y2), "r"(0));
    asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(w) : "r"(y1), "r"(y0), "r"(t));
    return w;
}
// byte permute with sign replication (selector nibble bit 3): sign-extends one packed int8 / int16 lane
__device__ __forceinline__ int prmt_sx(uint32_t w, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(0u), "r"(sel));
    return (int)d;
}

// RightShift (round half away from zero, saturate) + BiasAdd + Sp, all in integers, branch-free:
//   rs >= 1:  round_half_away(acc / 2^rs) = (acc + 2^(rs-1) - (acc < 0)) >> rs   (arithmetic shift)
//   rs <= 0:  acc * 2^-rs, saturated first (the shift is monotone)
struct Requant {
    int half, sh, mul, lo;     // rs >= 1: half = 2^(rs-1), sh = rs, mul unused; rs <= 0: mul = 2^-rs
    bool pos;
};
__device__ __forceinline__ Requant make_requant(int rs, int relu)
{
    Requant q;
    q.lo = relu ? 0 : -128;
    q.pos = rs >= 1;
    q.half = rs >= 1 ? (1 << (rs - 1)) : 0;
    q.sh = rs >= 1 ? rs : 0;
    q.mul = rs >= 1 ? 1 : (1 << (-rs));
    return q;
}
// result is saturated from below (q.lo = -128, or 0 when a ReLU is fused) but NOT from above: callers
// finish with min(., 127) or with the saturating pack
__device__ __forceinline__ int requant_nohi(int acc, const Requant &q, int bias)
{
    int r;
    if (q.pos) r = (acc + q.half + (acc >> 31)) >> q.sh;
    else r = max(-128, min(127, acc)) * q.mul;
    r = max(-128, min(127, r));
    return __viaddmax_s32(r, bias, q.lo);           // max(r + bias, lo) in one VIADDMNMX
}
__device__ __forceinline__ int requant(int acc, const Requant &q, int bias)
{
    return min(127, requant_nohi(acc, q, bias));
}

// The same chain with the sign of rs a compile-time constant (the epilogue loops are instantiated for both).
template <bool POS>
__device__ __forceinline__ int requant_t(int acc, const Requant &q, int bias)
{
    int r;
    if (POS) r = (acc + q.half + (acc >> 31)) >> q.sh;        // VIADD, LEA.HI.SX32, SHF
    else r = max(-128, min(127, acc)) * q.mul;
    r = max(-128, min(127, r));                               // first saturation (RightShift)
    return __viaddmax_s32(r, bias, q.lo);                     // max(r + bias, lo); callers saturate from above
}

// The same chain with BiasAdd folded into the rounding add (PQ_FLAG_BIAS_FOLDED, rs >= 1): b << rs is a multiple
// of 2^rs, so with the per-channel constant c = 2^(rs-1) + (b << rs)
//   (acc + c + (acc >> 31)) >> rs  ==  round_half_away(acc / 2^rs) + b,
// and because the rounding is monotone the first saturation can be applied to the accumulator instead, with
// channel-independent bounds:  clamp(r, -128, 127) == r(clamp(acc, -128 * 2^rs - 2^(rs-1) + 1, 127 * 2^rs + 2^(rs-1) - 1)).
// The second saturation is the packing instruction's.  With a fused ReLU the lower bound is redundant (anything
// below it ends at 0 either way).  5 ALU operations per element instead of 6, with the same single per-channel
// constant vector as the classic chain; the CPU test suite checks the identities over every (rs, b) and the
// accumulators around both bounds.
template <bool RELU>
__device__ __forceinline__ int requant_folded(int acc, int sh, int a_lo, int a_hi, int c)
{
    const int a = RELU ? min(acc, a_hi) : max(min(acc, a_hi), a_lo);
    const int t = (a + c + (a >> 31)) >> sh;
    return RELU ? max(t, 0) : t;
}

}  // namespace pq

namespace {
// cudaLaunchKernelEx with programmatic stream serialisation (see pdl_wait); PQ_NO_PDL=1 in the environment turns the
// attribute off (the kernels' griddepcontrol instructions are then no-ops)
template <typename... KArgs, typename... Args>
int launch_pdl(void (*kern)(KArgs...), dim3 grid, int threads, size_t smem, cudaStream_t s, Args &&...args)
{
    static const bool no_pdl = [] { const char *e = getenv("PQ_NO_PDL"); return e && e[0] == '1'; }();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = no_pdl ? 0 : 1;
    return (int)cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
}  // namespace
