// pq_gemm_s8.cu -- ReconModel integer simulation (subsystem 4; SURVEY.md 8 rows a13, a14):
// int8 x int8 -> int32 GEMM and implicit-GEMM convolution on the 5th-generation tensor cores
// (tcgen05.mma kind::i8, accumulators in TMEM), operands staged by TMA, with the reference's
//   RightShift -> BiasAdd -> Sp -> DeQuantity        (new_quantity_op.py:11-44, 61-101, 124-133)
// chain fused into the epilogue.
//
// Persistent kernel, one CTA per SM, looping over 128 x BN output tiles (n fastest, so consecutive
// tiles reuse the same activation rows out of L2):
//   warp 0   : TMA producer.  A tile = 128 output pixels x BK input channels of ONE filter tap,
//              fetched by a single im2col-mode TMA (padding = hardware zero fill, stride =
//              traversal stride), or a plain 2-D tile for GEMMs / 1x1 stride-1 convolutions.
//              B tile = BN filters x the same BK-byte slice of the [K][R*S*C] weight matrix.
//   warp 1   : allocates TMEM (two accumulators of BN columns), issues tcgen05.mma (one elected
//              lane), commits to mbarriers.
//   warps 2-17: epilogue, four warps per TMEM lane quadrant, each taking a quarter of the columns,
//              TMEM loads software-pipelined against the arithmetic and the stores:
//              tcgen05.ld the int32 accumulators (lane = output pixel, column = output channel),
//              shift / round-half-away / saturate, + bias, saturate, then de-quantise to fp32 NCHW
//              (the module boundary of the reference) and / or store int8 NHWC.
// A STAGES-deep smem ring (full/empty mbarriers) decouples TMA from MMA; the two TMEM accumulators
// (tmem_full/tmem_empty mbarriers) let the epilogue of tile i overlap the main loop of tile i+1.
// Round 2: separate A / B producer warps (warp 18 = B), 2-4 accumulator stages with one warp group per tile in
// flight, the fused NewAdd epilogue (epilogue_add), resident weights and "patch windows" for short-K 3x3 layers
// (GemmParams::win_*: one TMA box per tile, nine shifted descriptors), programmatic dependent launch.
#include <cuda.h>
#include <cstdlib>

#include "pq_common.cuh"
#include "pq_requant.cuh"

namespace pq {

constexpr int kBM = 128;               // UMMA M (cta_group::1): one TMEM lane per output row
constexpr int kEpiWarps = 16;           // four per TMEM lane quadrant
constexpr int kGemmThreads = 64 + 32 * kEpiWarps + 32;   // A-operand TMA warp, MMA warp, epilogue warps, B-operand TMA warp
constexpr int kWarpB = 2 + kEpiWarps;   // the B-operand producer is the last warp (the epilogue keeps warps 2..17)

// ------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
// One leader lane per warp (deterministic for a given member mask).  The producer and MMA loops are
// executed by the WHOLE warp with only the asynchronous instructions predicated on the leader, so that
// tile / stage / coordinate arithmetic stays warp-uniform (uniform datapath, no R2UR waterfall loops):
// a single-lane loop needed ~100 dependent instructions per K block and bounded the short-K layers.
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap *map, uint64_t *bar, void *dst, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// variants taking precomputed shared-window addresses
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d_a(const CUtensorMap *map, uint32_t bar, uint32_t dst, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d_a(const CUtensorMap *map, uint32_t bar, uint32_t dst, int c0, int c1, int c2)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_a(const CUtensorMap *map, uint32_t bar, uint32_t dst, int c0, int c1, int c2,
                                              int c3)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_5d_a(const CUtensorMap *map, uint32_t bar, uint32_t dst, int c0, int c1, int c2,
                                              int c3, int c4)
{
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void tma_load_im2col_4d_a(const CUtensorMap *map, uint32_t bar, uint32_t dst, int c, int w,
                                                     int h, int n, uint16_t off_w, uint16_t off_h)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
        : "memory");
}
__device__ __forceinline__ void bulk_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_load_1d_a(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tma_load_5d(const CUtensorMap *map, uint64_t *bar, void *dst, int c0, int c1, int c2,
                                            int c3, int c4)
{
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void tma_load_im2col_4d(const CUtensorMap *map, uint64_t *bar, void *dst, int c, int w,
                                                   int h, int n, uint16_t off_w, uint16_t off_h)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
        : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, const void *src, int c0, int c1)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap *map, const void *src, int c0, int c1, int c2, int c3)
{
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(map),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
// variants on shared-window addresses + a value the optimiser cannot re-derive: under register pressure ptxas
// rematerialises shared addresses (S2UR SR_CgaCtaId / SR_SWINHI, the 1024-byte alignment of the dynamic segment: ~20
// instructions each time) and the lane id (S2R + its ~20-cycle latency) at every use inside the epilogue's slab
// loop -- 150 of ~550 instructions per slab in the fused-add epilogue (ncu source view).
__device__ __forceinline__ uint32_t keep_u32(uint32_t x)
{
    uint32_t y;
    asm volatile("mov.u32 %0, %1;" : "=r"(y) : "r"(x));
    return y;
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_store_2d_a(const CUtensorMap *map, uint32_t src, int c0, int c1)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(src),
                 "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_4d_a(const CUtensorMap *map, uint32_t src, int c0, int c1, int c2, int c3)
{
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(map),
                 "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ uint4 lds_u4(uint32_t addr)
{
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ void sts_u4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync(int threads)
{
    asm volatile("bar.sync 1, %0;" ::"r"(threads) : "memory");
}
__device__ __forceinline__ uint4 ldg_nc_u4(const void *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t cols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void umma_commit_a(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], int8 operands, int32 accumulate
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                        uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[16])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major shared-memory operand descriptor (cute::UMMA::SmemDescriptor): rows of BK bytes, swizzle
// span == BK, 8-row groups SBO = 8*BK bytes apart; version 1 (Blackwell).
template <int BK>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr)
{
    constexpr uint64_t layout = BK == 128 ? 2 : (BK == 64 ? 4 : 6);      // SWIZZLE_128B / 64B / 32B
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);                          // start address
    d |= (uint64_t)1 << 16;                                              // LBO (unused for swizzled K-major)
    d |= (uint64_t)((8 * BK) >> 4) << 32;                                // SBO
    d |= (uint64_t)1 << 46;                                              // descriptor version
    d |= layout << 61;
    return d;
}

// cute::UMMA::InstrDescriptor for kind::i8: S32 accumulate, signed A and B, both K-major.
__host__ __device__ constexpr uint32_t make_idesc_i8(int m, int n)
{
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct GemmParams {
    int M, N;                  // output rows (pixels) and columns (channels)
    int num_kb;                // K blocks of BK bytes
    int a_im2col;              // 0: A is a 2-D [M][K] tile source; 1: im2col over NHWC; 2: row windows (below)
    int R, S, cblocks;         // filter taps and BK-blocks per tap (im2col mode)
    int b_resident;            // the whole B operand of the CTA (one n tile, num_kb <= ring slots) is loaded ONCE into the
                               // ring's B slots and stays there: short-K 3x3 layers are bound by L2 -> SM traffic (the
                               // im2col gather re-reads every input byte R*S times), of which the per-tile weight
                               // re-fetch was a third
    int tps;                   // K blocks per pipeline stage (im2col mode): one mbarrier round trip moves tps A tiles and tps
                               // B tiles (3 for short-K 3x3 layers, whose K block holds only ~70 cycles of tensor work)
    int C;                     // padded channels (bytes per pixel)
    int P, Q;                  // output height / width (im2col mode)
    int stride_h, stride_w, pad_h, pad_w;
    int dil_h, dil_w;          // filter dilation (im2col mode): tap (r, s) reads pixel offset (r * dil_h, s * dil_w)
    int rs, ob;                // RightShift amount, output fractional bit
    int hw;                    // pixels per image for the fp32 NCHW store (1: plain [M][N])
    int relu;                  // int8 pipeline: apply max(y, 0) in the epilogue (a following nn.ReLU)
    int stage_s8;              // int8 output leaves through a swizzled smem tile + TMA store (N % 16 == 0)
    // a_im2col == 2, convolutions with <= 8 input channels (the ResNet stem): the input is a zero-padded
    // NHWC image with 8-byte pixels, so the S taps of one filter row are BK contiguous bytes and an
    // overlapping-stride tensor map (pixel step = stride_w * 8 bytes) fetches them for a TH x TW patch of
    // output pixels in one tiled TMA; K loop = the R filter rows.
    // Fused NewAdd (int8 pipeline): the epilogue adds a shortcut tensor of the output's [M][N] geometry,
    //   num = clamp(y * 2^add_cshift + shortcut * 2^add_sshift, add_lo, add_hi)        (units of 2^-o_bit)
    // and writes num as int16 (out16) and round_half_even(num * 2^add_qshift) saturated as int8 (out_s8).
    const void *add_sc;        // shortcut, int8 or int16 (add_is16); NULL: no fused add
    int add_is16, add_sc_relu, add_cshift, add_sshift, add_lo, add_hi, add_qshift;
    int16_t *out16;
    int tw_shift, TW, TH;      // output patch of one tile: TH x TW = 128 pixels, TW = 1 << tw_shift
    int tiles_p, tiles_q;      // patches per image
    // a_im2col == 3, "patch windows" (3x3, stride 1, pad 1, C == BK, one n tile, resident weights): the A operand of
    // a tile is ONE tiled TMA box [TH + 2 input rows][TW pixels from column -1][C] (hardware zero fill = the padding),
    // and the nine taps are nine shared-memory descriptors into it: GEMM row i = pixel (i / TW, i % TW) of the patch
    // reads box pixel i + r * TW + s, i.e. the same K-major rows C bytes apart, start address shifted by
    // (r * TW + s) * C bytes.  Patch columns >= Q (at least two of the TW) read the neighbouring box row: those GEMM
    // rows are junk and never stored.  L2 -> SM traffic per tile: (TH + 2) / TH input tiles instead of nine.
    int win_slot_bytes, win_slots;
    const int32_t *bias;       // [N] quantised bias (already saturated to int8 range)
    const int32_t *bias_c;     // PQ_FLAG_BIAS_FOLDED (1 <= rs <= 20): [N] 2^(rs-1) + (bias << rs), see requant_folded
    const uint32_t *bias_hl;   // PQ_FLAG_BIAS_FOLDED: [N/2] s16x2 pairs 127 + min(b, 0), then [N/2] pairs -128 + max(b, 0)
    float *out_f32;            // optional
    int8_t *out_s8;            // optional, [M][N]
    // Grouped convolution (modes 0 and 1): n tile t reads the input channels [(t / g_tpg) * g_wb, + g_wb), the
    // channel window of the groups it covers; the weights are stored block-diagonally over that window, so the K loop
    // is over g_wb bytes.  g_wb = 0: a dense layer (window origin 0).
    int g_wb, g_tpg;
};

// Accumulator stages in TMEM (<= 512 columns) == groups of epilogue warps working on different tiles.
// FAST (int8-only, staged) epilogues are instruction-bound: 2-4 tiles in flight, one warp per (tile, lane
// quadrant[, column half]).  The generic epilogue (fp32 NCHW stores, unstaged int8) is store-bound and
// does best when all 16 warps drain ONE tile at a time (its 128 x BN x 4 bytes leave as one burst).
// (the RightShift -> BiasAdd -> Sp chain itself, Requant / requant_t / requant_folded, is in pq_requant.cuh: the
// depthwise kernel of pq_depthwise.cu shares it)
template <int BN, bool FAST = true> struct EpiCfg {
    static constexpr int kAcc = (FAST && BN < 256) ? 4 : 2;            // TMEM accumulator stages
    static constexpr int kGroups = FAST ? kAcc : (BN >= 64 ? 1 : 2);   // warp groups on different tiles
    static constexpr int kWarpsPerAcc = kEpiWarps / kGroups;           // arrivals that release an accumulator
    static constexpr int kColSplit = kWarpsPerAcc / 4;                 // warps sharing the columns of one 32-row block
    static constexpr int kCols = BN / kColSplit;                       // columns per warp and tile
    static constexpr int kSlab = FAST ? (kCols < 64 ? kCols : 64) : kCols;   // bytes per staged row (FAST only)
    static constexpr int kSlabBytes = 32 * kSlab;                      // warp-private staging buffer
    static constexpr uint32_t kTmemCols = kAcc * BN < 32 ? 32 : kAcc * BN;
    static_assert(kCols % 16 == 0 && kCols >= 16, "16-column chunks");
    static_assert(!FAST || kSlab >= 32, "staged rows of >= 32 bytes");
};

// fused NewAdd epilogue (ADDK kernels): per epilogue warp one int8 output slab [32 rows][32 B] and two buffers
// [32 rows][64 B] that receive the shortcut slab by TMA and are overwritten in place with the int16 sum
constexpr int kAddSlab = 32;                                   // output channels per staged slab
constexpr int kAddO8Bytes = 32 * kAddSlab;                     // 1 KB
constexpr int kAddS16Bytes = 32 * kAddSlab * 2;                // 2 KB
constexpr int kAddWarpBytes = kAddO8Bytes + 2 * kAddS16Bytes;  // 5 KB

// BSLOTS: B-operand ring slots.  Normally one per A slot; the "deep A" configuration of short-K 3x3 layers keeps the
// whole B operand resident in 9 slots and spends the rest of shared memory on A slots (bytes in flight: these layers
// are bound by the latency of the im2col gather, 72 KB in flight per SM moved only one tile per TMA round trip).
template <int BN, int BK, int STAGES, bool ADDK = false, int BSLOTS = STAGES>
struct GemmSmem {
    static constexpr int kABytes = kBM * BK;
    static constexpr int kBBytes = BN * BK;
    static constexpr int kRingBytes = STAGES * kABytes + BSLOTS * kBBytes;
    static constexpr int kOutBytes = ADDK ? kEpiWarps * kAddWarpBytes
                                          : kEpiWarps * EpiCfg<BN, true>::kSlabBytes;   // warp-private int8 staging slabs (FAST is the larger)
    static constexpr size_t kTotal = 1024 /*align slack*/ + (size_t)kRingBytes + kOutBytes + 768 /*barriers*/;
};


// ---------------------------------------------------------------------------------------- epilogue
// Executed by warps 2..17: four warps per TMEM lane quadrant, each taking a quarter of the tile's columns;
// TMEM loads are software-pipelined against the arithmetic.  tcgen05.ld hands every lane the int32
// accumulators of its own output row (pixel); then shift / round-half-away / saturate, + bias, saturate,
// and either de-quantise to fp32 NCHW (the module boundary of the reference, lanes = consecutive pixels)
// and / or pack to int8 and leave through a swizzled shared-memory tile + TMA store (full 128-byte lines;
// the TMA clips rows >= M and columns >= N).
// Round 2: the saturations of the folded chain move BEHIND the shift, onto packed 16-bit pairs.  With
//   t = (acc + c + (acc >> 31)) >> rs = r + b        (r = round_half_away(acc / 2^rs), NOT saturated)
// the reference's  Sp(Sp(r) + b)  is  clamp(t, l, h)  with the per-channel bounds  h = 127 + min(b, 0),
// l = -128 + max(b, 0): the function r -> Sp(Sp(r) + b) is monotone, equals r + b in between and is constant h
// (l) above (below) the int8 range of r; under a fused ReLU l <= 0 is redundant.  Two accumulators are packed with
// signed saturation (I2IP.S16.S32.SAT: monotone, and |l|, |h| <= 255), clamped as a pair (VIMNMX.S16x2[.RELU]) and
// their low bytes gathered by one PRMT per four -- the pre-shift clamps on the 32-bit accumulator are gone.  h / l
// travel as s16x2 pairs in the third row of the folded bias buffer (pq_bias_fold_s32): two LDG.128 each per 16
// channels, warp-uniform.  Used by the fused-add epilogue (16 launches of ResNet-50: 2.85 -> 2.75 ms), NOT by the
// plain int8 epilogue, where the extra loads cost more than the arithmetic saves (measured, see below).
template <bool RELU>
__device__ __forceinline__ void requant_packed16(const uint32_t (&a)[16], int sh, const int32_t *c_row,
                                                 const uint32_t *h_row, const uint32_t *l_row, uint32_t (&w)[8])
{
    int c[16];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int4 c4 = __ldg(reinterpret_cast<const int4 *>(c_row) + j);
        c[4 * j] = c4.x; c[4 * j + 1] = c4.y; c[4 * j + 2] = c4.z; c[4 * j + 3] = c4.w;
    }
    uint32_t h[8], l[8];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const uint4 h4 = __ldg(reinterpret_cast<const uint4 *>(h_row) + j);
        h[4 * j] = h4.x; h[4 * j + 1] = h4.y; h[4 * j + 2] = h4.z; h[4 * j + 3] = h4.w;
        if (!RELU) {
            const uint4 l4 = __ldg(reinterpret_cast<const uint4 *>(l_row) + j);
            l[4 * j] = l4.x; l[4 * j + 1] = l4.y; l[4 * j + 2] = l4.z; l[4 * j + 3] = l4.w;
        }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int a0 = (int)a[2 * q], a1 = (int)a[2 * q + 1];
        const int t0 = (a0 + c[2 * q] + (a0 >> 31)) >> sh, t1 = (a1 + c[2 * q + 1] + (a1 >> 31)) >> sh;
        uint32_t d;
        asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(d) : "r"(t1), "r"(t0));
        w[q] = RELU ? __vimin_s16x2_relu(d, h[q]) : __vmaxs2(__vmins2(d, h[q]), l[q]);
    }
}

// FOLD: 0 = classic chain, 1 = folded bias, 2 = folded bias + fused ReLU (FAST, POS only)
template <int BN, bool POS, bool FAST, int FOLD = 0>
__device__ __forceinline__ void epilogue(const GemmParams &p, const CUtensorMap *tmap_o, uint8_t *smem_o,
                                         uint64_t *tmem_full_bar, uint64_t *tmem_empty_bar, uint32_t tmem_base,
                                         int total_tiles, int n_tiles)
{
    using E = EpiCfg<BN, FAST>;
    const int warp = (int)keep_u32(threadIdx.x >> 5), lane = (int)keep_u32(threadIdx.x & 31);   // (see keep_u32)
    const int quad = warp & 3;                     // TMEM lane quadrant this warp may access
    const int idx = (warp - 2) >> 2;               // 0..3
    const int group = idx / E::kColSplit;          // which tiles (and which accumulator stage) this warp serves
    const int part = idx % E::kColSplit;           // which column part of those tiles
    constexpr int kCols = E::kCols, kSlab = E::kSlab;
    constexpr int kChunksPerSlab = kSlab / 16, kSlabs = kCols / kSlab;
    constexpr uint32_t kSwzMask = kSlab == 64 ? 3u : 1u;
    const uint32_t stage_addr = keep_u32(smem_u32(smem_o + (warp - 2) * E::kSlabBytes));
    const uint32_t tfull_base = keep_u32(smem_u32(tmem_full_bar)), tempty_base = tfull_base + 32u;   // [4] + [4] mbarriers
    const int row = quad * 32 + lane;
    const Requant rq = make_requant(p.rs, p.relu);
    const float dq = __int_as_float((127 - p.ob) << 23);        // 2^-ob, exact
    const bool staged = FAST;                                    // TMA-stored int8 slabs exist only here
    int it = 0;                                                  // position in this CTA's tile sequence
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        if ((it & (E::kGroups - 1)) != group) continue;
        const int acc = it & (E::kAcc - 1);                      // TMEM accumulator stage of this tile
        const uint32_t acc_phase = (uint32_t)(it / E::kAcc) & 1u;
        const int m0 = (tile / n_tiles) * kBM, nt0 = (tile % n_tiles) * BN, n0 = nt0 + part * kCols;
        int m = m0 + row, p_img = 0, p_row = 0, p_col = 0;
        bool row_ok = m < p.M;
        if (p.a_im2col >= 2) {                     // tile row -> pixel of the TH x TW output patch
            const int mt = tile / n_tiles, per_img = p.tiles_p * p.tiles_q;
            p_img = mt / per_img;
            const int rem = mt - p_img * per_img;
            p_row = (rem / p.tiles_q) * p.TH;
            p_col = (rem % p.tiles_q) * p.TW;
            const int pr = p_row + (row >> p.tw_shift), pc = p_col + (row & (p.TW - 1));
            row_ok = pr < p.P && pc < p.Q;
            m = (p_img * p.P + pr) * p.Q + pc;
        }
        float *of = nullptr;
        size_t cstride = 1;
        int8_t *o8 = nullptr;
        if (!FAST) {
            if (p.out_f32) {
                if (p.hw > 1) {                    // NCHW: lanes of a warp write consecutive pixels
                    const int img = m / p.hw, pix = m - img * p.hw;
                    of = p.out_f32 + ((size_t)img * p.N + n0) * p.hw + pix;
                    cstride = (size_t)p.hw;
                } else {
                    of = p.out_f32 + (size_t)m * p.N + n0;
                }
            }
            if (p.out_s8) o8 = p.out_s8 + (size_t)m * p.N + n0;     // generic path: direct int8 stores
        }
        mbar_wait_a(tfull_base + 8u * (uint32_t)acc, acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + part * kCols);

        // one chunk of 16 columns held in registers -> packed int8 (4 words) [+ fp32 / unstaged int8 stores]
        auto emit = [&](const uint32_t (&a)[16], int c0, uint32_t (&packed)[4]) {
            if (FAST) {
                // N % 16 == 0 here, so a chunk is entirely inside or outside N (outside: the TMA store clips
                // it); bias is 64-byte aligned: 4 x LDG.128, warp-uniform
                if (n0 + c0 >= p.N) return;
                if (FOLD != 0) {
                    // (the packed post-shift saturation of requant_packed16 was measured here too: no gain with a
                    // fused ReLU, 4-10 % SLOWER without -- the two extra bound vectors cost more than the two ALU
                    // operations they save; it pays only in the fused-add epilogue, whose tail is packed anyway)
                    const int4 *cp = reinterpret_cast<const int4 *>(p.bias_c + n0 + c0);
                    const int a_hi = 127 * (1 << rq.sh) + rq.half - 1, a_lo = -128 * (1 << rq.sh) - rq.half + 1;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int4 c4 = __ldg(cp + j);
                        packed[j] = pack4_sat_s8(requant_folded<FOLD == 2>((int)a[4 * j], rq.sh, a_lo, a_hi, c4.x),
                                                 requant_folded<FOLD == 2>((int)a[4 * j + 1], rq.sh, a_lo, a_hi, c4.y),
                                                 requant_folded<FOLD == 2>((int)a[4 * j + 2], rq.sh, a_lo, a_hi, c4.z),
                                                 requant_folded<FOLD == 2>((int)a[4 * j + 3], rq.sh, a_lo, a_hi, c4.w));
                    }
                    return;
                }
                const int4 *bp = reinterpret_cast<const int4 *>(p.bias + n0 + c0);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int4 b4 = __ldg(bp + j);
                    packed[j] = pack4_sat_s8(requant_t<POS>((int)a[4 * j], rq, b4.x), requant_t<POS>((int)a[4 * j + 1], rq, b4.y),
                                             requant_t<POS>((int)a[4 * j + 2], rq, b4.z), requant_t<POS>((int)a[4 * j + 3], rq, b4.w));
                }
                return;
            }
            // generic path, kept compact (the loop body of four chunks must stay I-cache sized): one bias
            // gather, one requantisation, one strided fp32 store loop that serves NCHW (stride = pixels per
            // image, lanes = consecutive pixels) and plain [M][N] (stride 1) alike.
            const int nvalid = p.N - (n0 + c0);            // columns of this chunk inside N (may be <= 0 or > 16)
            if (nvalid <= 0) return;
            int y[16];
            if (nvalid >= 16) {
                const int4 *bp = reinterpret_cast<const int4 *>(p.bias + n0 + c0);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int4 b4 = __ldg(bp + j);
                    y[4 * j] = b4.x; y[4 * j + 1] = b4.y; y[4 * j + 2] = b4.z; y[4 * j + 3] = b4.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) y[j] = j < nvalid ? __ldg(p.bias + n0 + c0 + j) : 0;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) y[j] = min(127, requant_t<POS>((int)a[j], rq, y[j]));
#pragma unroll
            for (int j = 0; j < 4; ++j)
                packed[j] = pack4_sat_s8(y[4 * j], y[4 * j + 1], y[4 * j + 2], y[4 * j + 3]);
            if (!row_ok) return;
            if (of) {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (j < nvalid) of[(size_t)(c0 + j) * cstride] = __fmul_rn((float)y[j], dq);
            }
            if (o8) {                                  // unstaged fall-back (N % 16 != 0): direct stores
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (j < nvalid) o8[c0 + j] = (int8_t)y[j];
            }
        };

        // software pipeline over the chunks of the tile: the TMEM load of chunk i+1 is in flight while chunk
        // i is processed; after each slab (kSlab columns) the warp stages and TMA-stores its 32 rows.  The
        // slab loop is NOT unrolled: four warp groups run different tiles, so the code must stay I-cache sized.
        uint32_t a0[16], a1[16];
        uint32_t packed[kChunksPerSlab][4];
        constexpr int kChunks = kCols / 16;
        static_assert(kChunksPerSlab % 2 == 0 || kSlabs == 1, "chunk parity selects the TMEM register buffer");
        tmem_ld16(taddr, a0);
#pragma unroll 1
        for (int slab = 0; slab < kSlabs; ++slab) {
#pragma unroll
            for (int j = 0; j < kChunksPerSlab; ++j) {
                const int ch = slab * kChunksPerSlab + j;
                tmem_ld_wait();
                if (ch + 1 < kChunks) {
                    if (j & 1) tmem_ld16(taddr + (uint32_t)((ch + 1) * 16), a0);
                    else tmem_ld16(taddr + (uint32_t)((ch + 1) * 16), a1);
                } else {
                    // every TMEM read of this accumulator has completed: hand it back to the MMA warp
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_a(tempty_base + 8u * (uint32_t)acc);
                }
                if (j & 1) emit(a1, ch * 16, packed[j]);
                else emit(a0, ch * 16, packed[j]);
            }
            const int colb = n0 + slab * kSlab;                         // first output channel of the slab
            if (staged && colb < p.N) {                                 // warp-uniform
                // the previous TMA store of this warp must have finished reading the staging buffer
                if (lane == 0) bulk_wait_read0();
                __syncwarp();
#pragma unroll
                for (int j = 0; j < kChunksPerSlab; ++j) {
                    const uint32_t o = (uint32_t)(lane * kSlab + 16 * j);
                    sts_u4(stage_addr + (o ^ (((o >> 7) & kSwzMask) << 4)), packed[j][0], packed[j][1], packed[j][2],
                           packed[j][3]);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    if (p.a_im2col >= 2) {         // 32 tile rows = a (32 / TW) x min(TW, 32) piece of the patch
                        const int r0 = quad * 32;
                        tma_store_4d_a(tmap_o, stage_addr, colb, p_col + (r0 & (p.TW - 1)), p_row + (r0 >> p.tw_shift), p_img);
                    } else {
                        tma_store_2d_a(tmap_o, stage_addr, colb, m0 + quad * 32);
                    }
                    bulk_commit();
                }
            }
        }
    }
    if (staged && lane == 0) bulk_wait_read0();
}


// ------------------------------------------------------------------- fused NewConv2d + NewAdd epilogue
// NewAdd (new_quantity_op.py:166-174) and the nn.ReLU after it, evaluated on the accumulators of the producing
// convolution while they are still in registers, in the SAME lane-owns-row mapping as the TMEM load (lane =
// output pixel, 16 consecutive channels per chunk):
//   y    = RightShift / BiasAdd / Sp of the accumulator (int8 range, bit ob)              32-bit, as above
//   sum  = clamp(y * 2^cshift + shortcut * 2^sshift, lo, hi)   at bit o = max(ob, shortcut bit)   packed s16x2
//   out16 = sum (the exact Eltwise output, for the next identity shortcut)
//   out8  = Quantity(q_bit)(sum)  (ties-to-even shift, saturated; what the next convolution reads)
// The shortcut slab [32 rows][32 channels] of the warp arrives by TMA one slab AHEAD (two buffers per warp, own
// mbarriers) into swizzled shared memory, the lane reads its own row from there (conflict-free LDS.128), the
// int16 sum overwrites the shortcut in place and leaves by a second TMA store next to the int8 slab.  No lane
// ever touches global memory, every global transaction is a full 64-byte / 32-byte row segment, and the
// arithmetic after the shift runs on packed 16-bit pairs (VIADDMNMX.S16x2, VIMNMX.S16x2): ~7 ALU operations per
// element instead of the 27 of the former second pass over the staged slab.
__device__ __forceinline__ uint32_t pack2_sat_s16(int hi, int lo)
{
    uint32_t d;
    asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(d) : "r"(hi), "r"(lo));
    return d;
}


// One 16-column chunk of the fused add once the convolution result (pk) and the shortcut (sc) are in registers as
// packed s16x2 pairs.  OUT_RELU / FASTQ are compile-time so that the common case (ReLU after the Eltwise, Eltwise bit ==
// sum bit) is a straight line of 1.25 packed instructions per element; everything else takes the general 32-bit
// requantisation.
template <bool OUT_RELU, bool FASTQ>
__device__ __forceinline__ void add_chunk(const uint32_t (&pk)[8], const uint32_t (&sc)[8], uint32_t s_hi2, uint32_t s_lo2,
                                          int qshift, int d, int rc, uint32_t (&sum)[8], uint32_t (&o)[4])
{
#pragma unroll
    for (int q = 0; q < 8; ++q)
        sum[q] = OUT_RELU ? __viaddmin_s16x2_relu(pk[q], sc[q], s_hi2)
                          : __vmaxs2(__viaddmin_s16x2(pk[q], sc[q], s_hi2), s_lo2);
    if (FASTQ) {                                       // same bit: saturate the pairs, keep the low bytes
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t w0 = __vmins2(sum[2 * q], 0x007f007fu), w1 = __vmins2(sum[2 * q + 1], 0x007f007fu);
            if (!OUT_RELU) { w0 = __vmaxs2(w0, 0xff80ff80u); w1 = __vmaxs2(w1, 0xff80ff80u); }
            o[q] = __byte_perm(w0, w1, 0x6420);
        }
    } else {                                           // general requantisation in 32 bits (ties to even / left shift)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            int e[4] = {(int)(short)(sum[2 * q] & 0xffffu), (int)sum[2 * q] >> 16,
                        (int)(short)(sum[2 * q + 1] & 0xffffu), (int)sum[2 * q + 1] >> 16};
#pragma unroll
            for (int u = 0; u < 4; ++u)
                e[u] = d ? (e[u] + rc + ((e[u] >> d) & 1)) >> d : max(-128, min(127, e[u])) << qshift;
            o[q] = pack4_sat_s8(e[0], e[1], e[2], e[3]);
        }
    }
}

template <int BN, bool POS, bool FOLD>
__device__ __forceinline__ void epilogue_add(const GemmParams &p, const CUtensorMap *tmap_o, const CUtensorMap *tmap_sc,
                                             const CUtensorMap *tmap_o16, uint8_t *smem_o, uint64_t *sc_bar_all,
                                             uint64_t *tmem_full_bar, uint64_t *tmem_empty_bar, uint32_t tmem_base,
                                             int total_tiles, int n_tiles)
{
    using E = EpiCfg<BN, true>;
    const int warp = (int)keep_u32(threadIdx.x >> 5), lane = (int)keep_u32(threadIdx.x & 31);
    const int quad = warp & 3;
    const int idx = (warp - 2) >> 2;
    const int group = idx / E::kColSplit;
    const int part = idx % E::kColSplit;
    constexpr int kCols = E::kCols, kSlabs = kCols / kAddSlab;
    const uint32_t wbase = keep_u32(smem_u32(smem_o + (warp - 2) * kAddWarpBytes));
    const uint32_t o8_base = wbase, s16_base = wbase + kAddO8Bytes;
    const uint32_t bar_base = keep_u32(smem_u32(sc_bar_all + 2 * (warp - 2)));
    const uint32_t tfull_base = keep_u32(smem_u32(tmem_full_bar)), tempty_base = tfull_base + 32u;   // [4] + [4] mbarriers
    const Requant rq = make_requant(p.rs, 0);
    const bool sc16 = p.add_is16 != 0;
    const uint32_t sc_bytes = sc16 ? (uint32_t)kAddS16Bytes : (uint32_t)kAddO8Bytes;
    // constants of the packed arithmetic
    const int cmul = 1 << p.add_cshift;                // (bounds of the scaled conv result; the scaling itself is a shift)
    const uint32_t y_hi2 = (uint32_t)(127 * cmul) * 0x10001u, y_lo2 = ((uint32_t)(-128 * cmul) & 0xffffu) * 0x10001u;
    const uint32_t s_hi2 = (uint32_t)p.add_hi * 0x10001u, s_lo2 = ((uint32_t)p.add_lo & 0xffffu) * 0x10001u;
    const bool out_relu = p.add_lo == 0;
    const int d = p.add_qshift < 0 ? -p.add_qshift : 0, rc = d ? (1 << (d - 1)) - 1 : 0;
    const int a_hi = 127 * (1 << rq.sh) + rq.half - 1, a_lo = -128 * (1 << rq.sh) - rq.half + 1;
    // swizzled shared-memory offsets of this lane's row: 64-byte rows (int16) and 32-byte rows (int8)
    auto off16 = [&](int chunk16) { return (uint32_t)(lane * 64 + ((chunk16 ^ ((lane >> 1) & 3)) << 4)); };
    auto off8 = [&](int chunk16) { return (uint32_t)(lane * 32 + ((chunk16 ^ ((lane >> 2) & 1)) << 4)); };

    // this warp's tiles: it = group, group + kGroups, ...; a tile counts only if its first column is inside N
    auto tile_of = [&](int it) { return blockIdx.x + it * (int)gridDim.x; };
    auto n0_of = [&](int tile) { return (n_tiles == 1 ? 0 : tile % n_tiles) * BN + part * kCols; };
    auto next_loaded_it = [&](int it) {              // first it' >= it whose tile exists and has columns for this warp
        for (;; it += E::kGroups) {
            const int t = tile_of(it);
            if (t >= total_tiles) return -1;
            if (n0_of(t) < p.N) return it;
        }
    };
    // (row, column) of a slab are passed in: the tile -> coordinate divisions are done once per TILE, not per slab
    // (ncu source view: a MUFU.RCP division sequence per slab, ~10 % of the epilogue's instructions)
    auto issue_load = [&](int buf, int m0r, int colb) {      // leader lane only
        const uint32_t bar = bar_base + 8u * (uint32_t)buf;
        mbar_expect_tx_a(bar, sc_bytes);
        tma_load_2d_a(tmap_sc, bar, s16_base + (uint32_t)buf * kAddS16Bytes, sc16 ? colb * 2 : colb, m0r);
    };
    auto row0_of = [&](int tile) { return (n_tiles == 1 ? tile : tile / n_tiles) * kBM + quad * 32; };

    uint32_t ph0 = 0u, ph1 = 0u;                       // parity of the next completion of either buffer's barrier
    int cur = 0;                                       // buffer that holds (or will hold) the current slab's shortcut
    {
        const int it0 = next_loaded_it(group);
        if (it0 >= 0 && lane == 0) issue_load(0, row0_of(tile_of(it0)), n0_of(tile_of(it0)));
    }
    for (int it = group;; it += E::kGroups) {
        const int tile = tile_of(it);
        if (tile >= total_tiles) break;
        const int acc = it & (E::kAcc - 1);
        const uint32_t acc_phase = (uint32_t)(it / E::kAcc) & 1u;
        const int m0r = row0_of(tile), n0 = n0_of(tile);
        int nslab = (p.N - n0 + kAddSlab - 1) / kAddSlab;             // slabs of this warp inside N
        nslab = nslab < 0 ? 0 : (nslab > kSlabs ? kSlabs : nslab);
        mbar_wait_a(tfull_base + 8u * (uint32_t)acc, acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + part * kCols);
        if (nslab == 0) {                              // nothing to do here, but the accumulator must be released
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_a(tempty_base + 8u * (uint32_t)acc);
            continue;
        }
        uint32_t a0[16], a1[16];
        tmem_ld16(taddr, a0);
#pragma unroll 1
        for (int slab = 0; slab < nslab; ++slab) {
            const int colb = n0 + slab * kAddSlab;
            uint32_t pk[2][8];                         // conv result of the slab's two chunks as packed s16x2, x 2^cshift
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int ch = slab * 2 + j;
                tmem_ld_wait();
                if (ch + 1 < nslab * 2) {
                    if (j & 1) tmem_ld16(taddr + (uint32_t)((ch + 1) * 16), a0);
                    else tmem_ld16(taddr + (uint32_t)((ch + 1) * 16), a1);
                } else {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_a(tempty_base + 8u * (uint32_t)acc);
                }
                const uint32_t (&a)[16] = (j & 1) ? a1 : a0;
                if (colb + 16 * j < p.N) {
                    if (FOLD && p.add_cshift == 0) {       // y directly as clamped s16x2 pairs (see requant_packed16)
                        const uint32_t *hrow = p.bias_hl + ((colb + 16 * j) >> 1);
                        requant_packed16<false>(a, rq.sh, p.bias_c + colb + 16 * j, hrow, hrow + (p.N >> 1), pk[j]);
                        continue;
                    }
                    int y[16];
                    if (FOLD) {
                        const int4 *cp = reinterpret_cast<const int4 *>(p.bias_c + colb + 16 * j);
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int4 c4 = __ldg(cp + q);
                            y[4 * q] = requant_folded<false>((int)a[4 * q], rq.sh, a_lo, a_hi, c4.x);
                            y[4 * q + 1] = requant_folded<false>((int)a[4 * q + 1], rq.sh, a_lo, a_hi, c4.y);
                            y[4 * q + 2] = requant_folded<false>((int)a[4 * q + 2], rq.sh, a_lo, a_hi, c4.z);
                            y[4 * q + 3] = requant_folded<false>((int)a[4 * q + 3], rq.sh, a_lo, a_hi, c4.w);
                        }
                    } else {
                        const int4 *bp = reinterpret_cast<const int4 *>(p.bias + colb + 16 * j);
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int4 b4 = __ldg(bp + q);
                            y[4 * q] = requant_t<POS>((int)a[4 * q], rq, b4.x);
                            y[4 * q + 1] = requant_t<POS>((int)a[4 * q + 1], rq, b4.y);
                            y[4 * q + 2] = requant_t<POS>((int)a[4 * q + 2], rq, b4.z);
                            y[4 * q + 3] = requant_t<POS>((int)a[4 * q + 3], rq, b4.w);
                        }
                    }
                    // (r + b) is within [-256, 254]: scale (only when the sum lives at a finer bit), pack, then the
                    // second saturation on the packed pairs
                    if (p.add_cshift == 0) {
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            pk[j][q] = __vmaxs2(__vmins2(pack2_sat_s16(y[2 * q + 1], y[2 * q]), y_hi2), y_lo2);
                    } else {
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            pk[j][q] = __vmaxs2(__vmins2(pack2_sat_s16(y[2 * q + 1] << p.add_cshift, y[2 * q] << p.add_cshift),
                                                         y_hi2), y_lo2);
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < 8; ++q) pk[j][q] = 0u;
                }
            }
            // ---- the shortcut of this slab has been on its way since the previous slab
            const uint32_t sbuf = s16_base + (uint32_t)cur * kAddS16Bytes;
            mbar_wait_a(bar_base + 8u * (uint32_t)cur, cur ? ph1 : ph0);
            if (cur) ph1 ^= 1u; else ph0 ^= 1u;
            uint32_t sc[2][8];
            if (sc16) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const uint4 lo = lds_u4(sbuf + off16(2 * j)), hi = lds_u4(sbuf + off16(2 * j + 1));
                    sc[j][0] = lo.x; sc[j][1] = lo.y; sc[j][2] = lo.z; sc[j][3] = lo.w;
                    sc[j][4] = hi.x; sc[j][5] = hi.y; sc[j][6] = hi.z; sc[j][7] = hi.w;
                }
            } else {                                   // int8 shortcut: sign-extend byte pairs to s16x2
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const uint4 v = lds_u4(sbuf + off8(j));
                    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        sc[j][2 * q] = (uint32_t)prmt_sx(w[q], 0x9180u);
                        sc[j][2 * q + 1] = (uint32_t)prmt_sx(w[q], 0xb3a2u);
                    }
                }
            }
            // every lane has its shortcut in registers: the buffers may now be rewritten.  The stores of the previous
            // slab must have finished READING the int8 slab and the other int16 buffer before either is reused.
            if (lane == 0) bulk_wait_read0();
            __syncwarp();
            {                                          // prefetch the next slab's shortcut into the other buffer
                int nrow = m0r, ncol = colb + kAddSlab;
                bool more = true;
                if (slab + 1 == nslab) {               // the first slab of this warp's next tile (divisions: once per tile)
                    const int itn = next_loaded_it(it + E::kGroups);
                    more = itn >= 0;
                    if (more) { nrow = row0_of(tile_of(itn)); ncol = n0_of(tile_of(itn)); }
                }
                if (more && lane == 0) issue_load(cur ^ 1, nrow, ncol);
            }
            if (p.add_sc_relu) {                       // a pending nn.ReLU on the shortcut operand
#pragma unroll
                for (int j = 0; j < 2; ++j)
#pragma unroll
                    for (int q = 0; q < 8; ++q) sc[j][q] = __vmaxs2(sc[j][q], 0u);
            }
            if (p.add_sshift) {                        // rare: shortcut at a coarser bit than the sum
#pragma unroll
                for (int j = 0; j < 2; ++j)
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const int lo16 = (int)(short)(sc[j][q] & 0xffffu), hi16 = (int)sc[j][q] >> 16;
                        sc[j][q] = pack2_sat_s16(hi16 << p.add_sshift, lo16 << p.add_sshift);
                    }
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                if (colb + 16 * j >= p.N) continue;
                uint32_t sum[8], o[4];
                if (p.add_qshift == 0) {
                    if (out_relu) add_chunk<true, true>(pk[j], sc[j], s_hi2, s_lo2, 0, 0, 0, sum, o);
                    else add_chunk<false, true>(pk[j], sc[j], s_hi2, s_lo2, 0, 0, 0, sum, o);
                } else {
                    if (out_relu) add_chunk<true, false>(pk[j], sc[j], s_hi2, s_lo2, p.add_qshift, d, rc, sum, o);
                    else add_chunk<false, false>(pk[j], sc[j], s_hi2, s_lo2, p.add_qshift, d, rc, sum, o);
                }
                if (p.out16) {
                    sts_u4(sbuf + off16(2 * j), sum[0], sum[1], sum[2], sum[3]);
                    sts_u4(sbuf + off16(2 * j + 1), sum[4], sum[5], sum[6], sum[7]);
                }
                sts_u4(o8_base + off8(j), o[0], o[1], o[2], o[3]);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                tma_store_2d_a(tmap_o, o8_base, colb, m0r);
                if (p.out16) tma_store_2d_a(tmap_o16, sbuf, colb * 2, m0r);
                bulk_commit();
            }
            cur ^= 1;
        }
    }
    if (lane == 0) bulk_wait_read0();
}

// A-operand producer loop, specialised per addressing mode (0: 2-D [M][K] tiles, 1: im2col over NHWC,
// 2: overlapping-stride 5-D windows for <= 8 input channels).  Runs on a whole warp; only the leader
// lane issues.  Arrives on full_bar with the A bytes of the stage (the B producer adds its own).
template <int MODE, int BK, int STAGES>
__device__ __forceinline__ void produce_a(const GemmParams &p, const CUtensorMap *tmap_a, uint8_t *smem_a,
                                          uint64_t *full_bar, uint64_t *empty_bar, int total_tiles, int n_tiles)
{
    constexpr uint32_t kABytes = kBM * BK;
    const bool leader = elect_one();
    const int lane = threadIdx.x & 31;
    int stage = 0; uint32_t phase = 0;
    const int pq = p.P * p.Q;
    const uint32_t a_base = smem_u32(smem_a), full_base = smem_u32(full_bar);
    // Tile -> coordinate divisions are done 32 tiles at a time, one tile per lane, and handed to the
    // (warp-uniform) issue loop with shuffles: the divisions were 40 % of this warp's instruction stream.
    int l_m0 = 0, l_nb = 0, l_hp = 0, l_wq = 0, l_c0 = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        if ((it & 31) == 0) {
            const int t = tile + lane * (int)gridDim.x;            // tiles beyond the end are never fetched
            const int mt = n_tiles == 1 ? t : t / n_tiles;
            l_m0 = mt * kBM;
            if (MODE != 2 && p.g_wb) l_c0 = ((t - mt * n_tiles) / p.g_tpg) * p.g_wb;   // grouped: channel window
            if (MODE == 1) {                   // first output pixel of the tile -> input coords
                l_nb = l_m0 / pq;
                const int rem = l_m0 - l_nb * pq;
                l_hp = rem / p.Q;
                l_wq = rem - l_hp * p.Q;
            }
            if (MODE == 2) {                   // patch -> (image, first output row, first output column)
                const int per_img = p.tiles_p * p.tiles_q;
                l_nb = mt / per_img;
                const int rem = mt - l_nb * per_img;
                l_hp = (rem / p.tiles_q) * p.TH;
                l_wq = (rem % p.tiles_q) * p.TW;
            }
        }
        const int m0 = __shfl_sync(0xffffffffu, l_m0, it & 31);
        const int c0 = (MODE != 2 && p.g_wb) ? __shfl_sync(0xffffffffu, l_c0, it & 31) : 0;
        int wq = 0, hp = 0, nb = 0;
        if (MODE != 0) {
            nb = __shfl_sync(0xffffffffu, l_nb, it & 31);
            hp = __shfl_sync(0xffffffffu, l_hp, it & 31);
            wq = __shfl_sync(0xffffffffu, l_wq, it & 31);
        }
        const int w0 = wq * p.stride_w - p.pad_w, h0 = hp * p.stride_h - p.pad_h;
        int r = 0, s = 0, cb = 0;
        const int tps = MODE == 1 ? p.tps : 1, nss = STAGES / tps;       // stages of tps consecutive ring slots
        for (int kb = 0; kb < p.num_kb; kb += tps) {
            mbar_wait(empty_bar + stage, phase ^ 1);
            const uint32_t bar = full_base + (uint32_t)stage * 8u;
            if (leader) mbar_expect_tx_a(bar, kABytes * (uint32_t)tps);
            for (int t = 0; t < tps; ++t) {
                if (leader) {
                    const uint32_t dst = a_base + (uint32_t)(stage * tps + t) * kABytes;
                    if (MODE == 2)             // filter row kb: padded input row = p * stride_h + kb
                        tma_load_5d_a(tmap_a, bar, dst, 0, wq, hp + kb / p.stride_h, kb % p.stride_h, nb);
                    else if (MODE == 1)
                        tma_load_im2col_4d_a(tmap_a, bar, dst, c0 + cb * BK, w0, h0, nb, (uint16_t)(s * p.dil_w),
                                             (uint16_t)(r * p.dil_h));
                    else
                        tma_load_2d_a(tmap_a, bar, dst, c0 + kb * BK, m0);
                }
                if (MODE == 1) { if (++cb == p.cblocks) { cb = 0; if (++s == p.S) { s = 0; ++r; } } }
            }
            if (++stage == nss) { stage = 0; phase ^= 1; }
        }
    }
}

// ---- a_im2col == 3 (patch windows, see GemmParams): one box per tile, nine descriptors per box
template <int BK>
__device__ __forceinline__ void produce_windows(const GemmParams &p, const CUtensorMap *tmap_a, uint8_t *smem_a,
                                                uint64_t *full_bar, uint64_t *empty_bar, int total_tiles)
{
    const bool leader = elect_one();
    const uint32_t a_base = smem_u32(smem_a), full_base = smem_u32(full_bar);
    const uint32_t bytes = (uint32_t)((p.TH + 2) * p.TW * BK);
    int slot = 0; uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {      // one n tile: tile == patch
        const int img = tile / p.tiles_p, h0 = (tile - img * p.tiles_p) * p.TH;
        mbar_wait(empty_bar + slot, phase ^ 1);
        if (leader) {
            const uint32_t bar = full_base + (uint32_t)slot * 8u;
            mbar_expect_tx_a(bar, bytes);
            tma_load_4d_a(tmap_a, bar, a_base + (uint32_t)(slot * p.win_slot_bytes), 0, -p.pad_w, h0 - p.pad_h, img);
        }
        __syncwarp();
        if (++slot == p.win_slots) { slot = 0; phase ^= 1; }
    }
}

template <int BN, int BK>
__device__ __forceinline__ void mma_windows(const GemmParams &p, uint8_t *smem_a, uint8_t *smem_b, uint64_t *full_bar,
                                            uint64_t *empty_bar, uint64_t *tmem_full_bar, uint64_t *tmem_empty_bar,
                                            uint64_t *bres_bar, uint32_t tmem_base, int total_tiles, int kAcc)
{
    constexpr uint32_t idesc = make_idesc_i8(kBM, BN < 16 ? 16 : BN);
    constexpr uint32_t kBBytes = BN * BK;
    const bool leader = elect_one();
    const uint64_t da0 = make_smem_desc<BK>(smem_u32(smem_a)), db0 = make_smem_desc<BK>(smem_u32(smem_b));
    const uint32_t empty_base = smem_u32(empty_bar), tfull_base = smem_u32(tmem_full_bar);
    const uint32_t row_step = (uint32_t)(p.TW * BK) >> 4;                 // one filter row down, in descriptor units
    int slot = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    mbar_wait(bres_bar, 0);                                               // the weights: nine [BN][BK] tiles, tap-major
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        mbar_wait(tmem_empty_bar + acc, acc_phase ^ 1);
        mbar_wait(full_bar + slot, phase);
        tc_fence_after();
        if (leader) {
            const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
            uint64_t da_r = da0 + (uint64_t)((uint32_t)(slot * p.win_slot_bytes) >> 4);
            uint64_t db = db0;
#pragma unroll 1
            for (int r = 0; r < 3; ++r) {
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const uint64_t da = da_r + (uint64_t)((uint32_t)(s * BK) >> 4);
#pragma unroll
                    for (int k = 0; k < BK / 32; ++k)
                        umma_i8(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (r | s | k) != 0);
                    db += kBBytes >> 4;
                }
                da_r += row_step;
            }
            umma_commit_a(empty_base + (uint32_t)slot * 8u);
            umma_commit_a(tfull_base + (uint32_t)acc * 8u);
        }
        __syncwarp();
        if (++slot == p.win_slots) { slot = 0; phase ^= 1; }
        if (++acc == kAcc) { acc = 0; acc_phase ^= 1; }
    }
}

template <int BN, int BK, int STAGES, bool ADDK = false, int BSLOTS = STAGES>
__global__ void __launch_bounds__(kGemmThreads, 1)     // 19 warps = 5 on one SM sub-partition: <= 104 registers / thread
gemm_s8_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_o, const __grid_constant__ CUtensorMap tmap_sc,
               const __grid_constant__ CUtensorMap tmap_o16, const GemmParams p)
{
    using Cfg = GemmSmem<BN, BK, STAGES, ADDK, BSLOTS>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *smem_a = smem;
    uint8_t *smem_b = smem + (size_t)STAGES * Cfg::kABytes;
    uint8_t *smem_o = smem + (size_t)Cfg::kRingBytes;                    // 1024-byte aligned
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem_o + Cfg::kOutBytes);
    uint64_t *empty_bar = full_bar + STAGES;
    uint64_t *tmem_full_bar = empty_bar + STAGES;      // [kAcc]
    uint64_t *tmem_empty_bar = tmem_full_bar + 4;      // [kAcc]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty_bar + 4);
    uint64_t *sc_bar = tmem_empty_bar + 5;             // [kEpiWarps][2] shortcut-slab barriers (ADDK kernels only)
    uint64_t *bres_bar = sc_bar + 2 * kEpiWarps;       // resident-B arrival
    const bool fast_epi = ADDK || (p.stage_s8 && !p.out_f32);          // which epilogue configuration runs
    const int kAcc = fast_epi ? EpiCfg<BN, true>::kAcc : EpiCfg<BN, false>::kAcc;

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform
    constexpr uint32_t kTmemCols = EpiCfg<BN, true>::kTmemCols;
    const int n_tiles = (p.N + BN - 1) / BN;
    const int total_tiles = (p.a_im2col >= 2 ? p.M / kBM : (p.M + kBM - 1) / kBM) * n_tiles;   // modes 2, 3: M = patches * 128

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_b) : "memory");
        if (p.stage_s8) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_o) : "memory");
        for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar + s, p.b_resident ? 1 : 2); mbar_init(empty_bar + s, 1); }   // A and B producers
        mbar_init(bres_bar, 1);
        const int arrivals = fast_epi ? EpiCfg<BN, true>::kWarpsPerAcc : EpiCfg<BN, false>::kWarpsPerAcc;
        for (int s = 0; s < kAcc; ++s) { mbar_init(tmem_full_bar + s, 1); mbar_init(tmem_empty_bar + s, arrivals); }
        if (ADDK) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_sc) : "memory");
            if (p.out16) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_o16) : "memory");
            for (int s = 0; s < 2 * kEpiWarps; ++s) mbar_init(sc_bar + s, 1);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
    pdl_launch_dependents();
    pdl_wait();                                        // operands / shortcut come from the preceding kernel

    if (warp == 0) {
        // ===================== A-operand TMA producer (whole warp, leader lane issues) =====================
        // One warp per operand: a single warp's dependent uniform-datapath chain costs ~8 cycles per
        // instruction (ncu: ~50 instructions = 410 cycles per K block with both operands in one warp),
        // which bounded every layer whose K block holds less than ~400 cycles of tensor work.
        if (p.a_im2col == 3) { if (!ADDK) produce_windows<BK>(p, &tmap_a, smem_a, full_bar, empty_bar, total_tiles); }
        else if (p.a_im2col == 1) produce_a<1, BK, STAGES>(p, &tmap_a, smem_a, full_bar, empty_bar, total_tiles, n_tiles);
        else if (p.a_im2col == 2) produce_a<2, BK, STAGES>(p, &tmap_a, smem_a, full_bar, empty_bar, total_tiles, n_tiles);
        else produce_a<0, BK, STAGES>(p, &tmap_a, smem_a, full_bar, empty_bar, total_tiles, n_tiles);
    } else if (warp == kWarpB) {
        // ===================== B-operand TMA producer =====================
        // weights [N][R*S*C]: the K offset of tap (r, s), channel block cb is kb * BK (C == cblocks * BK)
        const bool leader = elect_one();
        int stage = 0; uint32_t phase = 0;
        const uint32_t b_base = smem_u32(smem_b), full_base = smem_u32(full_bar);
        if (p.b_resident) {                            // all K blocks of the (single) n tile, once; slot == K block
            if (leader) {
                const uint32_t bar = smem_u32(bres_bar);
                const int tps = p.a_im2col == 1 ? p.tps : 1;
                mbar_expect_tx_a(bar, (uint32_t)Cfg::kBBytes * (uint32_t)p.num_kb);
                for (int kb = 0; kb < p.num_kb; kb += tps) {
                    const uint32_t dst = b_base + (uint32_t)kb * (uint32_t)Cfg::kBBytes;
                    if (tps == 1) tma_load_2d_a(&tmap_b, bar, dst, kb * BK, 0);
                    else tma_load_3d_a(&tmap_b, bar, dst, 0, 0, kb);
                }
            }
            __syncwarp();
        }
        for (int tile = blockIdx.x; tile < total_tiles && !p.b_resident; tile += gridDim.x) {
            const int n0 = (n_tiles == 1 ? 0 : tile % n_tiles) * BN;
            const int tps = p.a_im2col == 1 ? p.tps : 1, nss = STAGES / tps;
            for (int kb = 0; kb < p.num_kb; kb += tps) {
                mbar_wait(empty_bar + stage, phase ^ 1);
                if (leader) {
                    const uint32_t bar = full_base + (uint32_t)stage * 8u;
                    const uint32_t dst = b_base + (uint32_t)(stage * tps) * (uint32_t)Cfg::kBBytes;
                    mbar_expect_tx_a(bar, (uint32_t)Cfg::kBBytes * (uint32_t)tps);
                    // tps > 1: the map is [K block][N][BK] and one box brings tps consecutive K blocks, each as its
                    // own [BN][BK] tile in consecutive ring slots
                    if (tps == 1) tma_load_2d_a(&tmap_b, bar, dst, kb * BK, n0);
                    else tma_load_3d_a(&tmap_b, bar, dst, 0, n0, kb);
                }
                if (++stage == nss) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1 && !ADDK && p.a_im2col == 3) {
        mma_windows<BN, BK>(p, smem_a, smem_b, full_bar, empty_bar, tmem_full_bar, tmem_empty_bar, bres_bar, tmem_base,
                            total_tiles, kAcc);
    } else if (warp == 1) {
        // ===================== MMA issuer (whole warp, leader lane issues) =====================
        constexpr uint32_t idesc = make_idesc_i8(kBM, BN < 16 ? 16 : BN);
        const bool leader = elect_one();
        const uint64_t da0 = make_smem_desc<BK>(smem_u32(smem_a)), db0 = make_smem_desc<BK>(smem_u32(smem_b));
        const uint32_t empty_base = smem_u32(empty_bar), tfull_base = smem_u32(tmem_full_bar);
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        if (p.b_resident) mbar_wait(bres_bar, 0);
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            mbar_wait(tmem_empty_bar + acc, acc_phase ^ 1);      // epilogue has drained this accumulator
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
            const int tps = p.a_im2col == 1 ? p.tps : 1, nss = STAGES / tps;
            for (int kb = 0; kb < p.num_kb; kb += tps) {
                mbar_wait(full_bar + stage, phase);
                tc_fence_after();
                if (leader) {
                    for (int t = 0; t < tps; ++t) {
                        // the 14-bit start-address field advances by bytes / 16 (shared addresses stay below 2^18)
                        const uint64_t da = da0 + (uint64_t)(uint32_t)((stage * tps + t) * (Cfg::kABytes >> 4));
                        const uint64_t db = db0 + (uint64_t)(uint32_t)((p.b_resident ? kb + t : stage * tps + t) * (Cfg::kBBytes >> 4));
#pragma unroll
                        for (int k = 0; k < BK / 32; ++k)  // UMMA_K = 32 int8: advance 32 B inside the swizzle span
                            umma_i8(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | t | k) != 0);
                    }
                    umma_commit_a(empty_base + (uint32_t)stage * 8u);    // frees the smem slots when these MMAs retire
                }
                __syncwarp();
                if (++stage == nss) { stage = 0; phase ^= 1; }
            }
            if (leader) umma_commit_a(tfull_base + (uint32_t)acc * 8u);  // accumulator complete
            __syncwarp();
            if (++acc == kAcc) { acc = 0; acc_phase ^= 1; }
        }
    } else if (warp < kWarpB) {
        // ===================== epilogue (warps 2..17) =====================
        // compile-time variants: POS = right shift by rs >= 1 (the usual case), FAST = int8 output only,
        // leaving through the staged TMA store (the int8 pipeline); anything else takes the generic body
        const bool fast = fast_epi;
        if (p.rs >= 1) {
            if (ADDK) {
                if (p.bias_c) epilogue_add<BN, true, true>(p, &tmap_o, &tmap_sc, &tmap_o16, smem_o, sc_bar, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
                else epilogue_add<BN, true, false>(p, &tmap_o, &tmap_sc, &tmap_o16, smem_o, sc_bar, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            }
            else if (fast && p.bias_c && p.relu) epilogue<BN, true, true, 2>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            else if (fast && p.bias_c) epilogue<BN, true, true, 1>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            else if (fast) epilogue<BN, true, true>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            else epilogue<BN, true, false>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
        } else {
            if (ADDK) epilogue_add<BN, false, false>(p, &tmap_o, &tmap_sc, &tmap_o16, smem_o, sc_bar, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            else if (fast) epilogue<BN, false, true>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            else epilogue<BN, false, false>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

// ------------------------------------------------------------------------ small-channel "row" kernel
// Convolutions with <= 8 input channels, stride_w == 2 and S <= 8 (the ResNet stem) over the zero-padded
// 8-byte-pixel NHWC image.  One tile = 128 consecutive output columns of ONE output row; its A operand for
// filter row r is the padded input row p*stride_h + r itself: output column q reads the 64 bytes that
// start 16*q bytes into that row, so consecutive GEMM rows are 16 bytes apart -- exactly the row pitch of
// an un-swizzled K-major core matrix.  A shared-memory descriptor with LBO = 16 B (next 16-byte K chunk)
// and SBO = 128 B (next 8 rows) therefore lets the tensor core read the overlapping windows straight out
// of the raw rows: per tile ONE contiguous bulk copy of R input rows (12.9 KB for the 7x7 stem) replaces
// 7 x 128 window fetches (56 KB), and the weights stay resident in shared memory for the whole kernel.
struct RowsParams {
    const int8_t *xp;          // [N][Hp][pitch] bytes
    int pitch, Hp;             // bytes per padded row, padded rows per image
    int a_stage, stages;       // bytes per A ring slot (R rows + over-read slack), ring depth
};

__device__ __forceinline__ uint64_t make_smem_desc_interleave(uint32_t smem_addr)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);          // start address
    d |= (uint64_t)(16 >> 4) << 16;                      // LBO: next 16-byte chunk along K
    d |= (uint64_t)(128 >> 4) << 32;                     // SBO: next group of 8 rows
    d |= (uint64_t)1 << 46;                              // descriptor version (layout type 0 = no swizzle)
    return d;
}

__global__ void __launch_bounds__(kGemmThreads, 1)
conv_rows_s8_kernel(const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_o,
                    const GemmParams p, const RowsParams rp)
{
    constexpr int BN = 64, BK = 64, kMaxStages = 8;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int n_tiles = (p.N + BN - 1) / BN;
    uint8_t *smem_b = smem;                                              // [n_tiles][R][64 filters][64 B], 64B swizzle
    uint8_t *smem_o = smem_b + (size_t)n_tiles * p.R * (BN * BK);       // warp-private output slabs, 1024-byte aligned
    uint8_t *smem_a = smem_o + kEpiWarps * EpiCfg<BN, true>::kSlabBytes; // ring of raw input rows
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem_a + (size_t)rp.stages * rp.a_stage);
    uint64_t *empty_bar = full_bar + kMaxStages;
    uint64_t *tmem_full_bar = empty_bar + kMaxStages;
    uint64_t *tmem_empty_bar = tmem_full_bar + 4;
    uint64_t *b_bar = tmem_empty_bar + 4;
    const bool fast_epi = p.stage_s8 && !p.out_f32;
    const int kAcc = fast_epi ? EpiCfg<BN, true>::kAcc : EpiCfg<BN, false>::kAcc;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(b_bar + 1);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform
    constexpr uint32_t kTmemCols = EpiCfg<BN, true>::kTmemCols;
    const int total_tiles = (p.M / kBM) * n_tiles;
    const int per_img = p.tiles_p * p.tiles_q;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_b) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_o) : "memory");
        for (int s = 0; s < rp.stages; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
        const int arrivals = fast_epi ? EpiCfg<BN, true>::kWarpsPerAcc : EpiCfg<BN, false>::kWarpsPerAcc;
        for (int s = 0; s < kAcc; ++s) { mbar_init(tmem_full_bar + s, 1); mbar_init(tmem_empty_bar + s, arrivals); }
        mbar_init(b_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
    pdl_launch_dependents();
    pdl_wait();

    // Both loops below run on the whole warp with the asynchronous instructions predicated on one leader
    // lane, and walk the tiles incrementally (no per-tile division): the single-lane version spent ~390
    // dependent instructions per tile in the MMA warp and starved the epilogue (ncu: 60 % of all stall
    // samples were epilogue warps waiting for an accumulator).
    if (warp == 0) {
        const bool leader = elect_one();
        if (leader) {                                  // weights: resident for the whole kernel
            mbar_expect_tx(b_bar, (uint32_t)(n_tiles * p.R * BN * BK));
            for (int nt = 0; nt < n_tiles; ++nt)
                for (int r = 0; r < p.R; ++r)
                    tma_load_2d(&tmap_b, b_bar, smem_b + (size_t)(nt * p.R + r) * (BN * BK), r * BK, nt * BN);
        }
        __syncwarp();
        int stage = 0; uint32_t phase = 0;
        const uint32_t bytes = (uint32_t)(p.R * rp.pitch);
        const uint32_t a_base = smem_u32(smem_a), full_base = smem_u32(full_bar);
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int mt = n_tiles == 1 ? tile : tile / n_tiles;
            const int img = mt / per_img, prow = (mt - img * per_img) / p.tiles_q;
            mbar_wait(empty_bar + stage, phase ^ 1);
            if (leader) {
                const uint32_t bar = full_base + (uint32_t)stage * 8u;
                mbar_expect_tx_a(bar, bytes);
                bulk_load_1d_a(a_base + (uint32_t)(stage * rp.a_stage),
                               rp.xp + ((size_t)img * rp.Hp + (size_t)prow * p.stride_h) * rp.pitch, bytes, bar);
            }
            __syncwarp();
            if (++stage == rp.stages) { stage = 0; phase ^= 1; }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = make_idesc_i8(kBM, BN);
        const bool leader = elect_one();
        mbar_wait(b_bar, 0);
        const uint64_t da0 = make_smem_desc_interleave(smem_u32(smem_a));
        const uint64_t db0 = make_smem_desc<BK>(smem_u32(smem_b));
        const uint32_t a_step = (uint32_t)(rp.pitch >> 4);           // one filter row down (pitch % 16 == 0)
        const uint32_t empty_base = smem_u32(empty_bar), tfull_base = smem_u32(tmem_full_bar);
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            int nt = 0, q0 = 0;
            if (n_tiles != 1 || p.tiles_q != 1) {                    // (the ResNet stem has one tile per output row)
                const int mt = tile / n_tiles;
                nt = tile - mt * n_tiles;
                q0 = ((mt % per_img) % p.tiles_q) * kBM;
            }
            mbar_wait(tmem_empty_bar + acc, acc_phase ^ 1);
            mbar_wait(full_bar + stage, phase);
            tc_fence_after();
            if (leader) {
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
                uint64_t da = da0 + (uint64_t)(uint32_t)((stage * rp.a_stage + q0 * 16) >> 4);
                uint64_t db = db0 + (uint64_t)(uint32_t)((nt * p.R * (BN * BK)) >> 4);
                for (int r = 0; r < p.R; ++r) {
#pragma unroll
                    for (int k = 0; k < BK / 32; ++k)
                        umma_i8(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (r | k) != 0);
                    da += a_step;
                    db += (BN * BK) >> 4;
                }
                umma_commit_a(empty_base + (uint32_t)stage * 8u);
                umma_commit_a(tfull_base + (uint32_t)acc * 8u);
            }
            __syncwarp();
            if (++stage == rp.stages) { stage = 0; phase ^= 1; }
            if (++acc == kAcc) { acc = 0; acc_phase ^= 1; }
        }
    } else if (warp < kWarpB) {                        // (warp kWarpB idles: the weights are resident here)
        const bool fast = fast_epi;
        if (p.rs >= 1) {
            if (fast && p.bias_c && p.relu) epilogue<BN, true, true, 2>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            else if (fast && p.bias_c) epilogue<BN, true, true, 1>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            else if (fast) epilogue<BN, true, true>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            else epilogue<BN, true, false>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
        } else {
            if (fast) epilogue<BN, false, true>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
            else epilogue<BN, false, false>(p, &tmap_o, smem_o, tmem_full_bar, tmem_empty_bar, tmem_base, total_tiles, n_tiles);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

}  // namespace pq

// ------------------------------------------------------------------------------------ host side
namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                   const cuuint64_t *, const int *, const int *, cuuint32_t, cuuint32_t,
                                   const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn g_encode_tiled = nullptr;
EncodeIm2colFn g_encode_im2col = nullptr;

int load_driver_entry_points()
{
    if (g_encode_tiled && g_encode_im2col) return PQ_OK;
    cudaDriverEntryPointQueryResult q;
    void *fn = nullptr;
    PQ_CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !fn) return PQ_EUNSUPPORTED;
    g_encode_tiled = (EncodeTiledFn)fn;
    PQ_CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !fn) return PQ_EUNSUPPORTED;
    g_encode_im2col = (EncodeIm2colFn)fn;
    return PQ_OK;
}

CUtensorMapSwizzle swizzle_for(int bk)
{
    return bk == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (bk == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

// 2-D K-major int8 matrix [rows][k_bytes] (row pitch `pitch` bytes) -> box [box_rows][bk]
int encode_2d(CUtensorMap *map, const void *base, uint64_t k_bytes, uint64_t rows, uint64_t pitch, int bk,
              int box_rows)
{
    cuuint64_t dims[2] = {k_bytes, rows};
    cuuint64_t strides[1] = {pitch};
    cuuint32_t box[2] = {(cuuint32_t)bk, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), dims, strides, box,
                                estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk),
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? PQ_OK : PQ_EUNSUPPORTED;
}

// rank-N tiled map over bytes: dims / box innermost first, strides[i] = byte pitch of dimension i + 1
int encode_nd(CUtensorMap *map, const void *base, int rank, const cuuint64_t *dims, const cuuint64_t *strides,
              const cuuint32_t *box, int swizzle_bytes)
{
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, (cuuint32_t)rank, const_cast<void *>(base), dims,
                                strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(swizzle_bytes),
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? PQ_OK : PQ_EUNSUPPORTED;
}

int encode_im2col(CUtensorMap *map, const void *base, const pq_conv_desc &d, int bk)
{
    cuuint64_t dims[4] = {(cuuint64_t)d.C, (cuuint64_t)d.W, (cuuint64_t)d.H, (cuuint64_t)d.N};
    cuuint64_t strides[3] = {(cuuint64_t)d.C, (cuuint64_t)d.W * d.C, (cuuint64_t)d.H * d.W * d.C};
    int lower[2] = {-d.pad_w, -d.pad_h};
    int upper[2] = {d.pad_w - (d.S - 1) * d.dil_w, d.pad_h - (d.R - 1) * d.dil_h};
    cuuint32_t estr[4] = {1, (cuuint32_t)d.stride_w, (cuuint32_t)d.stride_h, 1};
    CUresult r = g_encode_im2col(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void *>(base), dims, strides,
                                 lower, upper, (cuuint32_t)bk, (cuuint32_t)pq::kBM, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return PQ_EUNSUPPORTED;
    // Same work-around CUTLASS applies (cute/atom/copy_traits_sm90_im2col.hpp) for drivers <= 13.1:
    // small tensors must not carry the bit the encoder sets for them.
    int drv = 0;
    cudaDriverGetVersion(&drv);
    if (drv <= 13010 && (uint64_t)d.N * d.H * d.W * d.C < 131072) reinterpret_cast<uint64_t *>(map)[1] &= ~(1ull << 21);
    return PQ_OK;
}

int num_sms()
{
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = pq::kNumSMs;
    }
    return n;
}

// one gemm_s8_kernel instance (opted in to its shared memory on first use) on a persistent grid: one CTA per SM
template <int BN, int BK, int STAGES, bool ADDK, int BSLOTS>
int launch_gemm(const CUtensorMap &ta, const CUtensorMap &tb, const CUtensorMap &to, const CUtensorMap &tsc,
                const CUtensorMap &to16, const pq::GemmParams &p, cudaStream_t s)
{
    using Cfg = pq::GemmSmem<BN, BK, STAGES, ADDK, BSLOTS>;
    static_assert(Cfg::kTotal <= 227 * 1024, "shared memory budget");
    auto kern = pq::gemm_s8_kernel<BN, BK, STAGES, ADDK, BSLOTS>;
    static bool attr = false;
    if (!attr) {
        PQ_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kTotal));
        attr = true;
    }
    const long long tiles = (long long)((p.M + pq::kBM - 1) / pq::kBM) * ((p.N + BN - 1) / BN);
    const int grid = (int)(tiles < num_sms() ? tiles : num_sms());
    return launch_pdl(kern, dim3((unsigned)grid), pq::kGemmThreads, Cfg::kTotal, s, ta, tb, to, tsc, to16, p);
}

template <int BN, int BK, int STAGES, int BSLOTS = STAGES>
int launch_cfg(const CUtensorMap &ta, const CUtensorMap &tb, pq::GemmParams &p, cudaStream_t s)
{
    p.b_resident = (p.a_im2col != 2 && p.N <= BN && p.num_kb <= BSLOTS) ? 1 : 0;
    if (BSLOTS != STAGES && !p.b_resident) return PQ_EUNSUPPORTED;      // deep-A configurations need the resident B
    // int8 output tile: [128 rows][min(BN, 128) bytes] boxes of the row-major [M][N] result
    CUtensorMap to = {};
    p.stage_s8 = 0;
    if (p.out_s8 && !p.out_f32 && (p.N & 15) == 0 && (((uintptr_t)p.out_s8) & 15) == 0) {
        constexpr int kSlab = pq::EpiCfg<BN, true>::kSlab;     // each epilogue warp stores [32 rows][kSlab bytes] boxes
        int rc;
        if (p.a_im2col >= 2) {                     // NHWC output addressed by (channel, q, p, image): TH x TW patches
            const cuuint64_t dims[4] = {(cuuint64_t)p.N, (cuuint64_t)p.Q, (cuuint64_t)p.P,
                                        (cuuint64_t)(p.M / pq::kBM / (p.tiles_p * p.tiles_q))};
            const cuuint64_t strides[3] = {(cuuint64_t)p.N, (cuuint64_t)p.N * p.Q, (cuuint64_t)p.N * p.Q * p.P};
            const cuuint32_t box[4] = {(cuuint32_t)kSlab, (cuuint32_t)(p.TW < 32 ? p.TW : 32),
                                       (cuuint32_t)(p.TW < 32 ? 32 / p.TW : 1), 1};
            rc = encode_nd(&to, p.out_s8, 4, dims, strides, box, kSlab);
        } else {
            rc = encode_2d(&to, p.out_s8, (uint64_t)p.N, (uint64_t)p.M, (uint64_t)p.N, kSlab, 32);
        }
        if (rc != PQ_OK) return rc;
        p.stage_s8 = 1;
    }
    const CUtensorMap none = {};
    return launch_gemm<BN, BK, STAGES, false, BSLOTS>(ta, tb, to, none, none, p, s);
}

// fused NewConv2d + NewAdd kernels (ADDK): int8 result, shortcut and int16 sum travel as [32 rows][32 channels]
// boxes per epilogue warp (see epilogue_add); fewer operand stages because the epilogue stages 80 KB
template <int BN, int BK, int STAGES>
int launch_cfg_add(const CUtensorMap &ta, const CUtensorMap &tb, pq::GemmParams &p, cudaStream_t s)
{
    p.b_resident = (p.N <= BN && p.num_kb <= STAGES) ? 1 : 0;
    CUtensorMap to = {}, tsc = {}, to16 = {};
    int rc;
    const uint64_t N = (uint64_t)p.N, M = (uint64_t)p.M;
    if ((rc = encode_2d(&to, p.out_s8, N, M, N, pq::kAddSlab, 32)) != PQ_OK) return rc;
    if (p.add_is16) rc = encode_2d(&tsc, p.add_sc, 2 * N, M, 2 * N, 2 * pq::kAddSlab, 32);
    else rc = encode_2d(&tsc, p.add_sc, N, M, N, pq::kAddSlab, 32);
    if (rc != PQ_OK) return rc;
    if (p.out16 && (rc = encode_2d(&to16, p.out16, 2 * N, M, 2 * N, 2 * pq::kAddSlab, 32)) != PQ_OK) return rc;
    p.stage_s8 = 1;
    return launch_gemm<BN, BK, STAGES, true, STAGES>(ta, tb, to, tsc, to16, p, s);
}

// stage counts: fill ~192 KB of shared memory, at most 8 stages
template <int BK>
int launch_bn(const CUtensorMap &ta, const CUtensorMap &tb, pq::GemmParams &p, int bn, cudaStream_t s)
{
    if (p.add_sc) {                                // 80 KB of epilogue staging: <= 144 KB of operand stages
        switch (bn) {
            case 256: return launch_cfg_add<256, BK, (BK == 128 ? 3 : (BK == 64 ? 6 : 8))>(ta, tb, p, s);
            case 128: return launch_cfg_add<128, BK, (BK == 128 ? 4 : 8)>(ta, tb, p, s);
            default: return launch_cfg_add<64, BK, (BK == 128 ? 6 : 8)>(ta, tb, p, s);
        }
    }
    // ring slots; for BK <= 64 a multiple of three where it fits (stages of three K blocks, GemmParams::tps)
    constexpr int S256 = BK == 128 ? 4 : (BK == 64 ? 8 : 9);
    constexpr int S128 = BK == 128 ? 6 : 9;
    constexpr int S64 = BK == 128 ? 8 : 9;
    // short-K 3x3 layers (C = 64, N <= 64: ResNet's first stage): resident weights, 18 A slots = 144 KB in flight
    if (BK == 64 && bn == 64 && p.a_im2col == 1 && p.N <= 64 && p.num_kb <= 9 && p.tps == 3)
        return launch_cfg<64, 64, 18, 9>(ta, tb, p, s);
    switch (bn) {
        case 256: return launch_cfg<256, BK, S256>(ta, tb, p, s);
        case 128: return launch_cfg<128, BK, S128>(ta, tb, p, s);
        case 64: return launch_cfg<64, BK, S64>(ta, tb, p, s);
        default: return launch_cfg<32, BK, S64>(ta, tb, p, s);
    }
}

// widest tile that still leaves every SM at least two tiles; never wider than N needs
int pick_bn(long long m, int n)
{
    const long long m_tiles = (m + pq::kBM - 1) / pq::kBM;
    const int cap = n > 128 ? 256 : (n > 64 ? 128 : (n > 32 ? 64 : 32));
    for (int bn = cap; bn > 32; bn >>= 1)
        if (m_tiles * ((n + bn - 1) / bn) >= 2LL * num_sms()) return bn;
    return 32 < cap && m_tiles * ((n + 63) / 64) >= num_sms() ? 64 : 32;
}

int launch(const CUtensorMap &ta, const CUtensorMap &tb, pq::GemmParams &p, int bk, int bn, cudaStream_t s)
{
    switch (bk) {
        case 128: return launch_bn<128>(ta, tb, p, bn, s);
        case 64: return launch_bn<64>(ta, tb, p, bn, s);
        default: return launch_bn<32>(ta, tb, p, bn, s);
    }
}

}  // namespace

namespace {
// the epilogue half of GemmParams (RightShift, BiasAdd, Sp, DeQuantity, the fused ReLU and the outputs); p.N must be set.
// PQ_FLAG_BIAS_FOLDED: bias_q is int32 [3][N] as written by pq_bias_fold_s32
void set_epilogue(pq::GemmParams &p, const int32_t *bias_q, int rs, int ob, int hw, int flags, float *out_f32,
                  int8_t *out_s8)
{
    p.rs = rs; p.ob = ob; p.hw = hw; p.bias = bias_q; p.out_f32 = out_f32; p.out_s8 = out_s8;
    p.relu = flags & PQ_FLAG_RELU;
    p.bias_c = ((flags & PQ_FLAG_BIAS_FOLDED) && rs >= 1 && rs <= 20 && (p.N & 15) == 0) ? bias_q + p.N : nullptr;
    p.bias_hl = p.bias_c ? reinterpret_cast<const uint32_t *>(bias_q + 2 * p.N) : nullptr;
}

// validates a fused-add request and copies it into the kernel parameters
int apply_add(pq::GemmParams &p, const pq_add_desc *add, int conv_ob)
{
    if (!add) return PQ_OK;
    if (!add->shortcut || !add->out8 || p.out_f32 || p.relu) return PQ_EINVAL;
    if ((p.N & 15) || (((uintptr_t)add->shortcut | (uintptr_t)add->out8 | (uintptr_t)add->out16) & 15)) return PQ_EALIGN;
    const int o_bit = conv_ob > add->shortcut_bit ? conv_ob : add->shortcut_bit;
    const int span = o_bit - (conv_ob < add->shortcut_bit ? conv_ob : add->shortcut_bit);
    if (span > 7 || o_bit < 0 || o_bit > 7 || add->q_bit - o_bit > 15 || o_bit - add->q_bit > 15) return PQ_EUNSUPPORTED;
    p.add_sc = add->shortcut; p.add_is16 = add->shortcut_is16; p.add_sc_relu = add->shortcut_relu;
    p.add_cshift = o_bit - conv_ob; p.add_sshift = o_bit - add->shortcut_bit;
    p.add_lo = add->out_relu ? 0 : -128 * (1 << o_bit); p.add_hi = 127 * (1 << o_bit);
    p.add_qshift = add->q_bit - o_bit;
    p.out16 = add->out16; p.out_s8 = add->out8;
    return PQ_OK;
}

// a grouped layer, validated by conv_impl: K loop over wb bytes (the weights' row length), n tiles of `block` output
// channels, tile t reading the input channels [(t / tpg) * wb, + wb) (GemmParams::g_wb)
struct Grouping {
    int wb, tpg, block;
};

int gemm_impl(const int8_t *a, const int8_t *w, const int32_t *bias_q, int M, int N, int K, int rs, int ob, int hw,
              int flags, float *out_f32, int8_t *out_s8, const pq_add_desc *add, pq_stream_t stream,
              const Grouping *grp = nullptr)
{
    if (M <= 0 || N <= 0 || K <= 0 || hw <= 0) return PQ_EINVAL;
    if (!a || !w || !bias_q || (!out_f32 && !out_s8)) return PQ_EINVAL;
    if ((K & 15) || (((uintptr_t)a | (uintptr_t)w) & 15)) return PQ_EALIGN;
    if (ob < -100 || ob > 100 || rs > 24 || rs < -24 || (hw > 1 && M % hw)) return PQ_EUNSUPPORTED;
    if ((uintptr_t)bias_q & 15) return PQ_EALIGN;
    int rc = load_driver_entry_points();
    if (rc != PQ_OK) return rc;
    // grouped: the K tail of a window is zero-filled in the weights' map only; the A bytes it reads (the next group's
    // channels) meet zero weights
    const int kw = grp ? grp->wb : K;
    const int bk = kw >= 128 ? 128 : (kw >= 64 ? 64 : 32);
    int bn = grp ? grp->block : pick_bn(M, N);
    if (add && bn < 64) bn = 64;                 // the fused-add pass works on 64-column slabs
    CUtensorMap ta, tb;
    if ((rc = encode_2d(&ta, a, K, M, K, bk, pq::kBM)) != PQ_OK) return rc;
    if ((rc = encode_2d(&tb, w, kw, N, kw, bk, bn)) != PQ_OK) return rc;
    pq::GemmParams p = {};
    p.M = M; p.N = N; p.num_kb = (kw + bk - 1) / bk; p.a_im2col = 0;
    if (grp) { p.g_wb = grp->wb; p.g_tpg = grp->tpg; }
    set_epilogue(p, bias_q, rs, ob, hw, flags, out_f32, out_s8);
    if ((rc = apply_add(p, add, ob)) != PQ_OK) return rc;
    return launch(ta, tb, p, bk, bn, (cudaStream_t)stream);
}

int conv_impl(const int8_t *x_nhwc, const int8_t *w_krsc, const int32_t *bias_q, const pq_conv_desc *desc_host,
              int flags, float *out_f32_nchw, int8_t *out_s8_nhwc, const pq_add_desc *add, pq_stream_t stream)
{
    if (!x_nhwc || !w_krsc || !bias_q || !desc_host || (!out_f32_nchw && !out_s8_nhwc)) return PQ_EINVAL;
    const pq_conv_desc &d = *desc_host;
    if (d.N <= 0 || d.H <= 0 || d.W <= 0 || d.C <= 0 || d.K <= 0 || d.R <= 0 || d.S <= 0) return PQ_EINVAL;
    if (d.stride_h <= 0 || d.stride_w <= 0 || d.pad_h < 0 || d.pad_w < 0 || d.dil_h <= 0 || d.dil_w <= 0) return PQ_EINVAL;
    const int r_eff = (d.R - 1) * d.dil_h + 1, s_eff = (d.S - 1) * d.dil_w + 1;   // footprint of the dilated filter
    if (d.H + 2 * d.pad_h < r_eff || d.W + 2 * d.pad_w < s_eff) return PQ_EINVAL;
    if (d.P != (d.H + 2 * d.pad_h - r_eff) / d.stride_h + 1 || d.Q != (d.W + 2 * d.pad_w - s_eff) / d.stride_w + 1)
        return PQ_EINVAL;
    if (r_eff > 255 || s_eff > 255) return PQ_EUNSUPPORTED;
    if ((d.C & 15) || (((uintptr_t)x_nhwc | (uintptr_t)w_krsc) & 15)) return PQ_EALIGN;
    if (d.ob < -100 || d.ob > 100 || d.rs > 24 || d.rs < -24 || d.stride_h > 8 || d.stride_w > 8) return PQ_EUNSUPPORTED;
    if ((uintptr_t)bias_q & 15) return PQ_EALIGN;
    const long long M = (long long)d.N * d.P * d.Q;
    if (M > 0x7fffffffLL) return PQ_EUNSUPPORTED;
    const bool plain = d.R == 1 && d.S == 1 && d.stride_h == 1 && d.stride_w == 1 && d.pad_h == 0 && d.pad_w == 0;
    Grouping grp = {0, 1, 0};
    const bool grouped = d.groups > 1;
    if (d.groups < 0) return PQ_EINVAL;
    if (grouped) {                                                   // weights [K][R][S][Wb], see the header
        if (add) return PQ_EUNSUPPORTED;
        if (d.C % d.groups || d.K % d.groups) return PQ_EINVAL;
        const int cg = d.C / d.groups, kg = d.K / d.groups, b = d.group_block;
        if ((b != 32 && b != 64 && b != 128 && b != 256) || (b % kg && kg % b) || d.K % b) return PQ_EUNSUPPORTED;
        grp.wb = cg * (b > kg ? b / kg : 1);
        grp.tpg = kg > b ? kg / b : 1;
        grp.block = b;
        if (grp.wb % (plain ? 16 : 32)) return PQ_EUNSUPPORTED;     // box width of the path below
    }
    if (plain)                                                       // 1x1 stride-1: a plain GEMM over NHWC
        return gemm_impl(x_nhwc, w_krsc, bias_q, (int)M, d.K, d.C, d.rs, d.ob, d.P * d.Q, flags, out_f32_nchw,
                         out_s8_nhwc, add, stream, grouped ? &grp : nullptr);
    if (d.C & 31) return PQ_EUNSUPPORTED;                            // im2col path: channel blocks of >= 32
    int rc = load_driver_entry_points();
    if (rc != PQ_OK) return rc;
    // 3x3 / stride 1 / pad 1 with one K block per tap and one n tile (ResNet: C = 64 at 56x56, C = 128 at 28x28): patch
    // windows (GemmParams, a_im2col == 3).  The im2col gather re-reads every input byte nine times out of L2 and bounds
    // these layers at ~9.5 TB/s of L2 -> SM traffic; the window box is read (TH + 2) / TH times.
    if (!add && !grouped && !(flags & PQ_FLAG_NO_WINDOWS) && d.R == 3 && d.S == 3 && d.stride_h == 1 && d.stride_w == 1 &&
        d.pad_h == 1 && d.pad_w == 1 && d.dil_h == 1 && d.dil_w == 1 &&
        ((d.C == 64 && d.K <= 64) || (d.C == 128 && d.K > 64 && d.K <= 128)) && d.W + 2 <= 64) {
        const int tw_shift = d.W + 2 <= 16 ? 4 : (d.W + 2 <= 32 ? 5 : 6);
        const int TW = 1 << tw_shift, TH = pq::kBM / TW;
        const int slot = ((TH + 2) * TW * d.C + 1023) / 1024 * 1024;
        const int a_region = d.C == 64 ? 18 * pq::kBM * 64 : 3 * pq::kBM * 128;       // the A ring of the configurations below
        const int max_slots = d.C == 64 ? 18 : 3;                                      // (their mbarrier pairs)
        int slots = a_region / slot;
        if (slots > max_slots) slots = max_slots;
        const long long patches = (long long)d.N * ((d.P + TH - 1) / TH);
        if (slots >= 2 && patches * pq::kBM <= 0x7fffffffLL) {
            CUtensorMap ta, tb;
            const cuuint64_t adims[4] = {(cuuint64_t)d.C, (cuuint64_t)d.W, (cuuint64_t)d.H, (cuuint64_t)d.N};
            const cuuint64_t astr[3] = {(cuuint64_t)d.C, (cuuint64_t)d.W * d.C, (cuuint64_t)d.H * d.W * d.C};
            const cuuint32_t abox[4] = {(cuuint32_t)d.C, (cuuint32_t)TW, (cuuint32_t)(TH + 2), 1};
            if ((rc = encode_nd(&ta, x_nhwc, 4, adims, astr, abox, d.C)) != PQ_OK) return rc;
            const uint64_t ktot = (uint64_t)9 * d.C;
            if ((rc = encode_2d(&tb, w_krsc, ktot, d.K, ktot, d.C, d.C == 64 ? 64 : 128)) != PQ_OK) return rc;
            pq::GemmParams p = {};
            p.a_im2col = 3; p.N = d.K; p.M = (int)(patches * pq::kBM);
            p.R = 3; p.S = 3; p.C = d.C; p.cblocks = 1; p.num_kb = 9; p.tps = 1;
            p.P = d.P; p.Q = d.Q; p.stride_h = 1; p.stride_w = 1; p.pad_h = 1; p.pad_w = 1; p.dil_h = 1; p.dil_w = 1;
            p.tw_shift = tw_shift; p.TW = TW; p.TH = TH; p.tiles_q = 1; p.tiles_p = (d.P + TH - 1) / TH;
            p.win_slot_bytes = slot; p.win_slots = slots;
            set_epilogue(p, bias_q, d.rs, d.ob, d.P * d.Q, flags, out_f32_nchw, out_s8_nhwc);
            return d.C == 64 ? launch_cfg<64, 64, 18, 9>(ta, tb, p, (cudaStream_t)stream)
                             : launch_cfg<128, 128, 3, 9>(ta, tb, p, (cudaStream_t)stream);
        }
    }
    const int cw = grouped ? grp.wb : d.C;       // input channels one output channel reads, per tap
    const int bk = (cw % 128 == 0) ? 128 : ((cw % 64 == 0) ? 64 : 32);
    int bn = grouped ? grp.block : pick_bn(M, d.K);
    if (add && bn < 64) bn = 64;                 // the fused-add pass works on 64-column slabs
    CUtensorMap ta, tb;
    if ((rc = encode_im2col(&ta, x_nhwc, d, bk)) != PQ_OK) return rc;
    const uint64_t ktot = (uint64_t)d.R * d.S * cw;
    pq::GemmParams p = {};
    p.M = (int)M; p.N = d.K; p.a_im2col = 1;
    p.R = d.R; p.S = d.S; p.C = d.C; p.cblocks = cw / bk; p.num_kb = d.R * d.S * p.cblocks;
    p.g_wb = grp.wb; p.g_tpg = grp.tpg;
    // short K blocks (<= 64 bytes of K: ~70 cycles of tensor work per block at BN = 64) are bound by the producers'
    // per-stage mbarrier round trip, not by TMA or the tensor pipe: move three K blocks per stage
    p.tps = (bk <= 64 && p.num_kb % 3 == 0) ? 3 : 1;
    if (p.tps == 1) {
        if ((rc = encode_2d(&tb, w_krsc, ktot, d.K, ktot, bk, bn)) != PQ_OK) return rc;
    } else {                                     // weights as [K block][N][bk]: box = tps blocks x bn filters x bk bytes
        const cuuint64_t bdims[3] = {(cuuint64_t)bk, (cuuint64_t)d.K, (cuuint64_t)p.num_kb};
        const cuuint64_t bstr[2] = {(cuuint64_t)ktot, (cuuint64_t)bk};
        const cuuint32_t bbox[3] = {(cuuint32_t)bk, (cuuint32_t)bn, (cuuint32_t)p.tps};
        if ((rc = encode_nd(&tb, w_krsc, 3, bdims, bstr, bbox, bk)) != PQ_OK) return rc;
    }
    p.P = d.P; p.Q = d.Q; p.stride_h = d.stride_h; p.stride_w = d.stride_w; p.pad_h = d.pad_h; p.pad_w = d.pad_w;
    p.dil_h = d.dil_h; p.dil_w = d.dil_w;
    set_epilogue(p, bias_q, d.rs, d.ob, d.P * d.Q, flags, out_f32_nchw, out_s8_nhwc);
    if ((rc = apply_add(p, add, d.ob)) != PQ_OK) return rc;
    return launch(ta, tb, p, bk, bn, (cudaStream_t)stream);
}
}  // namespace

extern "C" int pq_gemm_s8(const int8_t *a, const int8_t *w, const int32_t *bias_q, int M, int N, int K, int rs,
                          int ob, int hw, int flags, float *out_f32, int8_t *out_s8, pq_stream_t stream)
{
    return gemm_impl(a, w, bias_q, M, N, K, rs, ob, hw, flags, out_f32, out_s8, nullptr, stream);
}

extern "C" int pq_conv2d_s8(const int8_t *x_nhwc, const int8_t *w_krsc, const int32_t *bias_q,
                            const pq_conv_desc *desc_host, int flags, float *out_f32_nchw, int8_t *out_s8_nhwc,
                            pq_stream_t stream)
{
    return conv_impl(x_nhwc, w_krsc, bias_q, desc_host, flags, out_f32_nchw, out_s8_nhwc, nullptr, stream);
}

extern "C" int pq_conv2d_s8_add(const int8_t *x_nhwc, const int8_t *w_krsc, const int32_t *bias_q,
                                const pq_conv_desc *desc_host, const pq_add_desc *add_host, int flags,
                                pq_stream_t stream)
{
    if (!add_host || (flags & PQ_FLAG_RELU)) return PQ_EINVAL;   // the ReLU of a fused add is add_host->out_relu
    return conv_impl(x_nhwc, w_krsc, bias_q, desc_host, flags, nullptr, add_host->out8, add_host, stream);
}

// Convolution with <= 8 input channels over a zero-padded NHWC image with 8-byte pixels (see GemmParams):
// xp is [N][Hp][Wp][8] int8 as written by pq_quantize_nchw_to_padded_nhwc8_s8 (image pixel (h, w) at
// (h + pad_h, w + pad_w)), w_krs8 is [K][R][64] int8: 8 pixel slots x 8 channel slots per filter row, zero
// where s >= S or c >= C.  Requires stride_w * 8 % 16 == 0 (even stride_w), S <= 8, Hp % stride_h == 0.
extern "C" int pq_conv2d_smallc_s8(const int8_t *xp, const int8_t *w_krs8, const int32_t *bias_q,
                                   const pq_conv_desc *desc_host, int Hp, int Wp, int flags, float *out_f32_nchw,
                                   int8_t *out_s8_nhwc, pq_stream_t stream)
{
    if (!xp || !w_krs8 || !bias_q || !desc_host || (!out_f32_nchw && !out_s8_nhwc)) return PQ_EINVAL;
    const pq_conv_desc &d = *desc_host;
    if (d.N <= 0 || d.H <= 0 || d.W <= 0 || d.K <= 0 || d.R <= 0 || d.S <= 0) return PQ_EINVAL;
    if (d.stride_h <= 0 || d.stride_w <= 0 || d.pad_h < 0 || d.pad_w < 0) return PQ_EINVAL;
    if (d.dil_h != 1 || d.dil_w != 1) return PQ_EUNSUPPORTED;
    if (d.P != (d.H + 2 * d.pad_h - d.R) / d.stride_h + 1 || d.Q != (d.W + 2 * d.pad_w - d.S) / d.stride_w + 1)
        return PQ_EINVAL;
    constexpr int kPix = 8, kBK = 64;
    if (d.C != kPix || d.S > kBK / kPix || (d.stride_w & 1) || d.R > 64) return PQ_EUNSUPPORTED;
    if (Hp % d.stride_h || Hp < (d.P - 1) * d.stride_h + d.R || Hp < d.H + d.pad_h) return PQ_EUNSUPPORTED;
    if ((Wp * kPix) % 16 || Wp < (d.Q - 1) * d.stride_w + kBK / kPix || Wp < d.W + d.pad_w) return PQ_EUNSUPPORTED;
    if (d.ob < -100 || d.ob > 100 || d.rs > 24 || d.rs < -24) return PQ_EUNSUPPORTED;
    if ((((uintptr_t)xp | (uintptr_t)w_krs8 | (uintptr_t)bias_q) & 15)) return PQ_EALIGN;
    int rc = load_driver_entry_points();
    if (rc != PQ_OK) return rc;
    pq::GemmParams p = {};
    p.a_im2col = 2;
    p.tw_shift = d.Q >= 16 ? 4 : (d.Q >= 8 ? 3 : 2);
    p.TW = 1 << p.tw_shift; p.TH = pq::kBM / p.TW;
    p.tiles_q = (d.Q + p.TW - 1) / p.TW; p.tiles_p = (d.P + p.TH - 1) / p.TH;
    const long long patches = (long long)d.N * p.tiles_p * p.tiles_q;
    if (patches * pq::kBM > 0x7fffffffLL) return PQ_EUNSUPPORTED;
    p.M = (int)(patches * pq::kBM); p.N = d.K; p.num_kb = d.R;
    p.R = d.R; p.S = d.S; p.C = kPix; p.P = d.P; p.Q = d.Q;
    p.stride_h = d.stride_h; p.stride_w = d.stride_w; p.pad_h = d.pad_h; p.pad_w = d.pad_w;
    set_epilogue(p, bias_q, d.rs, d.ob, d.P * d.Q, flags, out_f32_nchw, out_s8_nhwc);
    // Preferred: the row kernel (stride_w == 2: GEMM rows 16 bytes apart == an un-swizzled core matrix)
    if (d.stride_w == 2 && d.R <= 8) {
        const int n_tiles = (d.K + 63) / 64;
        const int pitch = Wp * kPix;
        const int tiles_q = (d.Q + pq::kBM - 1) / pq::kBM;
        const int a_stage = (d.R * pitch + 2112 + 1023) / 1024 * 1024;       // + over-read of the last window rows
        const long long fixed = 1024 + (long long)n_tiles * d.R * 4096 + pq::kEpiWarps * pq::EpiCfg<64, true>::kSlabBytes + 256;
        const long long stages_fit = (227 * 1024 - fixed) / a_stage;
        const long long tiles_m = (long long)d.N * d.P * tiles_q;
        if (stages_fit >= 2 && tiles_m * pq::kBM <= 0x7fffffffLL &&
            (long long)(d.R - 1) * pitch + (long long)(tiles_q * pq::kBM - 1) * 16 + 64 <= a_stage) {
            pq::RowsParams rp;
            rp.xp = xp; rp.pitch = pitch; rp.Hp = Hp; rp.a_stage = a_stage;
            rp.stages = (int)(stages_fit < 8 ? stages_fit : 8);
            pq::GemmParams q = p;
            q.tw_shift = 7; q.TW = pq::kBM; q.TH = 1; q.tiles_q = tiles_q; q.tiles_p = d.P;
            q.M = (int)(tiles_m * pq::kBM);
            CUtensorMap tb, to = {};
            const uint64_t ktot = (uint64_t)d.R * kBK;
            if ((rc = encode_2d(&tb, w_krs8, ktot, d.K, ktot, kBK, 64)) != PQ_OK) return rc;
            q.stage_s8 = 0;
            if (q.out_s8 && !q.out_f32 && (q.N & 15) == 0 && (((uintptr_t)q.out_s8) & 15) == 0) {
                const cuuint64_t odims[4] = {(cuuint64_t)q.N, (cuuint64_t)q.Q, (cuuint64_t)q.P, (cuuint64_t)d.N};
                const cuuint64_t ostr[3] = {(cuuint64_t)q.N, (cuuint64_t)q.N * q.Q, (cuuint64_t)q.N * q.Q * q.P};
                // one epilogue warp stores 32 output columns x kSlab channels
                constexpr int slab = pq::EpiCfg<64, true>::kSlab;
                const cuuint32_t obox[4] = {(cuuint32_t)slab, 32, 1, 1};
                if ((rc = encode_nd(&to, q.out_s8, 4, odims, ostr, obox, slab)) != PQ_OK) return rc;
                q.stage_s8 = 1;
            }
            const size_t smem = (size_t)fixed + (size_t)rp.stages * a_stage;
            static size_t attr = 0;
            if (smem > attr) {
                PQ_CUDA_TRY(cudaFuncSetAttribute(pq::conv_rows_s8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                attr = smem;
            }
            const long long tiles = tiles_m * n_tiles;
            const int grid = (int)(tiles < num_sms() ? tiles : num_sms());
            return launch_pdl(pq::conv_rows_s8_kernel, dim3((unsigned)grid), pq::kGemmThreads, smem, (cudaStream_t)stream, tb, to, q, rp);
        }
    }
    // A: (byte in window, output column, row group, row phase, image); the column step overlaps the windows
    CUtensorMap ta, tb;
    const cuuint64_t row_pitch = (cuuint64_t)Wp * kPix;
    const cuuint64_t dims[5] = {(cuuint64_t)kBK, (cuuint64_t)d.Q, (cuuint64_t)(Hp / d.stride_h), (cuuint64_t)d.stride_h,
                                (cuuint64_t)d.N};
    const cuuint64_t strides[4] = {(cuuint64_t)d.stride_w * kPix, row_pitch * d.stride_h, row_pitch, row_pitch * Hp};
    const cuuint32_t box[5] = {(cuuint32_t)kBK, (cuuint32_t)p.TW, (cuuint32_t)p.TH, 1, 1};
    if ((rc = encode_nd(&ta, xp, 5, dims, strides, box, kBK)) != PQ_OK) return rc;
    const int bn = pick_bn((long long)p.M, d.K);
    const uint64_t ktot = (uint64_t)d.R * kBK;
    if ((rc = encode_2d(&tb, w_krs8, ktot, d.K, ktot, kBK, bn)) != PQ_OK) return rc;
    return launch(ta, tb, p, kBK, bn, (cudaStream_t)stream);
}
