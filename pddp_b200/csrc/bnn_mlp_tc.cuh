// Particle MLP on the 5th-generation tensor cores (tcgen05 + TMEM), fp32 in / fp32 out.
//
//   X'_p = X_p + dX_std * fc_out(relu(M1_p * fc_1(relu(M0_p * fc_0(norm([aug(X_p), u])))))) + dX_mean
//   (ref: pddp/models/bnn/modules.py:200-264, 774-789; dropout masks are [P,H], one row per particle)
// and, for the linearisation, its Jacobian w.r.t. (X_p, u) by forward-mode tangents that share the
// primal's activation pattern (SURVEY.md appendix B).
//
// Design (measurements and the road here: profiles/r1_summary.md; DESIGN.md section 4):
//   * a tile holds 128 items of ONE particle p (rows gathered with stride P), so the dropout masks
//     are per-column constants of the tile: M0_p is folded into a per-particle image of W0|b0
//     (relu(m*x) = m*relu(x), m >= 0) and M1_p into a per-particle copy of the output weights --
//     no mask is read in the inner loops;
//   * layer 0 runs on the tensor core too: A0 = [norm(aug(X),u), 1] (K padded to 8/16) times the
//     per-particle image, split FP16 like layer 1, 32 hidden units at a time into a small TMEM accumulator.  Row
//     H0 of the image is the unit vector of the bias column, so hidden unit H0 is the constant 1
//     that carries b1 through the second GEMM (b1 is column H0 of the W1 image);
//   * layer 1 (the 200x200 contraction) runs in split FP16, a0*b0 + a0*b1 + a1*b0 with fp32
//     accumulation: fp32-class accuracy from three FP16 passes and 4 operand bytes per element;
//   * tangents are pass-major: a super-tile is the primal pass followed by one pass per direction
//     over the same 128 items, so a thread meets the primal and the tangent pre-activation of the
//     same (item, hidden unit) and the ReLU gate is a per-thread bit mask, never a shuffle;
//   * two independent tile "tracks" per CTA consume the same streamed W1 K-block (16 wide,
//     SWIZZLE_64B rows of [b0 | b1]): half the L2->smem traffic per row.  Track 1 runs half a tile behind track 0,
//     and each track has its own layer-1 issuer thread, so one track's epilogue is covered by the
//     other's MMAs (they can drift NB W1 stages apart);
//   * warp roles (20 warps): per track 4 epilogue warps (16x256b TMEM fragments, output layer on
//     the CUDA cores with quad-shuffle column sums), 4 mid-stage warps (tcgen05.ld of the layer-0
//     chunk, ReLU / gate, hi-lo split, st.shared into the UMMA K-major layout) and one layer-1
//     MMA-issuer thread; one polling layer-0 issuer thread for both tracks; one bulk-copy loader.
//
//   * per-particle COMPACTION: a hidden unit whose dropout mask is below 2^-24 (CDropout at temperature 0.1: ~16 % of
//     the units of a particle; BDropout: every dropped unit) contributes less than fp32 rounding to anything
//     downstream.  Tiles are particle-uniform, so such units are simply left out of that particle's images: the
//     layer-1 GEMM of particle p is M128 x N(p) x K(p) with K(p) = kept layer-0 units + the bias unit (rounded up
//     to 16) and N(p) = kept layer-1 units (rounded up to 16) -- typically 11 K-blocks x 176 columns instead of
//     13 x 208, 0.72x the tensor work.  The W1 image is therefore per particle too, and the W1 stream the two
//     tracks share is organised in SEGMENTS (runs of super-tiles of one particle inside the CTA's range).
//
// TMEM (512 columns): track t owns columns [256t, 256t+208) for the layer-1 accumulator and
// [256t+208, 256t+240) for the layer-0 chunk.
#pragma once
#include "bnn_mlp_simt.cuh"
#include <cuda_fp16.h>
#include <type_traits>

namespace pddp {
namespace tc {

#ifdef PDDP_EXP_TRACE
// Timeline experiment: CTA 0 records clock64() stamps per role (regions of 8192 entries) for the LAST launch.
// Without PDDP_EXP_TRACE, TCLK() is a constant 0 and TR() is empty, so the stamps and per-tile sums in the role
// loops compile to nothing.
__device__ long long g_trace[8 * 8192];
#define TR_ON (blockIdx.x == 0)
#define TR(region, idx, val) do { if (TR_ON && (idx) < 8192) g_trace[(region) * 8192 + (idx)] = (val); } while (0)
#define TCLK() clock64()
#else
#define TR(region, idx, val) do { } while (0)
#define TCLK() 0ll
#endif

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase completes or the
// hint expires.  Without a hint the default window is ~50 cycles: the waiting roles re-polled 60 M
// times per launch, and the kernel runs into the board's power cap.
constexpr uint32_t MBAR_SUSPEND_NS = 20000;
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra.uni WAIT_DONE;\n\t"
        "bra.uni WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity), "r"(MBAR_SUSPEND_NS) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

constexpr int TILE_M = 128, TILE_N = 208, KB = 16, MAX_NKB = 13, MAX_NCH = 7, N0 = 32;
// Layer 1 in split FP16: a = a0 + a1, b = b0 + b1 with a0 = fp16(a), a1 = fp16(a - a0) (22
// significand bits together) and a*b ~ a0*b0 + a0*b1 + a1*b0 accumulated in fp32 by the tensor
// core -- three FP16 passes of K = 16 per K-block.  That is fp32-class accuracy (the dropped a1*b1
// is 2^-24 of the product) for 3/4 of the tensor time and 5/8..1/2 of the shared-memory and L2
// bytes of TF32-based splitting (a 4-byte [a0 | a1] pair per element instead of 8 bytes), which
// matters because the kernel is bound by the shared-memory data pipe (profiles/r1_summary.md).
// FP16 range: the W1 image is scaled by a power of two so that max |w| * scale is ~2^14 (the lo
// parts stay normal); the scale is undone inside the per-particle output weights.  Hidden
// activations must stay below 65504 (they are O(1) for any network that rolls out finitely).
constexpr int B_STAGE = TILE_N * 64;   // W1 K-block: 208 rows x [b0 (16 fp16) | b1 (16 fp16)], 13 312 B
constexpr int A1_SLOT = TILE_M * 64;   // 128 rows x [a0 (16 fp16) | a1 (16 fp16)], 8 192 B
constexpr int THREADS = 20 * 32;
constexpr int TM_ACC1 = 0, TM_ACC0 = 208, TM_TRACK = 256;

// byte offset of element (row, kk) in a K-major tile whose rows are ROWB bytes (32 / 64 / 128 =
// SWIZZLE_32B / 64B / 128B): 16-byte chunk index XORed with the matching bits of the row index.
template <int ROWB>
__host__ __device__ __forceinline__ uint32_t swz(int row, int kk) {
    constexpr int SH = ROWB == 32 ? 2 : ROWB == 64 ? 1 : 0;
    const int chunk = (kk >> 2) ^ ((row & 7) >> SH);
    return (uint32_t)((row >> 3) * (8 * ROWB) + (row & 7) * ROWB + (chunk << 4) + (kk & 3) * 4);
}
// same, for a byte position inside the row
template <int ROWB>
__host__ __device__ __forceinline__ uint32_t swz_byte(int row, int byte) {
    constexpr int SH = ROWB == 32 ? 2 : ROWB == 64 ? 1 : 0;
    return (uint32_t)((row >> 3) * (8 * ROWB) + (row & 7) * ROWB + ((((byte >> 4) ^ ((row & 7) >> SH))) << 4) + (byte & 15));
}
// K-major shared-memory descriptor for rows of ROWB bytes (cute::UMMA::SmemDescriptor bit layout):
// [0,14) addr>>4, [16,30) LBO>>4 = 1, [32,46) SBO>>4 = 8 rows, [46,48) version 1, [61,64) layout type.
template <int ROWB>
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    constexpr uint64_t LT = ROWB == 32 ? 6 : ROWB == 64 ? 4 : 2;
    uint64_t d = (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((8 * ROWB) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= LT << 61;
    return d;
}


// two floats -> packed fp16x2 (a in the low half = lower address)
__device__ __forceinline__ uint32_t pack_f16(float a, float b) {
    uint32_t d;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
    return d;
}
__device__ __forceinline__ float2 unpack_f16(uint32_t h) {
    return __half22float2(*reinterpret_cast<const __half2*>(&h));
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void sts128f(uint32_t addr, float x, float y, float z, float w) {
    sts128(addr, __float_as_uint(x), __float_as_uint(y), __float_as_uint(z), __float_as_uint(w));
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t x) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(x) : "memory");
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
    uint32_t x;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(x) : "r"(addr));
    return x;
}
__device__ __forceinline__ float4 lds128f(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
// packed fp32 pairs for FFMA2 (fma.rn.f32x2: two fp32 FMAs per issue slot; nvcc does not generate it on its own)
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float lo2(unsigned long long v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return a; }
__device__ __forceinline__ float hi2(unsigned long long v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return b; }
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc),
        "r"(accumulate) : "memory");
}
constexpr uint32_t idesc_f16(int M, int N) {      // A, B = F16 (format 0), D = F32
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void tc_ld32(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tc_ld16_nowait(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
// 16 lanes x 256 bit fragments: register 4i+{0,1} = row lane/4, columns 8i + 2*(lane%4) + {0,1};
// register 4i+{2,3} = row lane/4 + 8, same columns (measured with tools/probe/tmem_layout.cu).
__device__ __forceinline__ void tc_ld_16x256b_x4(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_16x256b_x2(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld8(float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])
                 :: "memory");
}
// tcgen05.wait::ld that also names the destination registers, so no use of them can be scheduled
// above the wait.
__device__ __forceinline__ void tc_wait_ld16(float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :: "memory");
}
__device__ __forceinline__ void tc_wait_ld32(float* v) {
    tc_wait_ld16(v);
    tc_wait_ld16(v + 16);
}
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// true in exactly one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <int K0P, int DP>
struct Cfg {
    static constexpr int NB = K0P == 8 ? 5 : 4;    // W1 K-block stages
    static constexpr int NS = K0P == 8 ? 6 : 4;    // layer-1 A-operand slots per track
    static constexpr int ROWB0 = K0P * 4;          // layer-0 operand row [x0 (K0P fp16) | x1 (K0P fp16)]: SWIZZLE_32B / 64B
    static constexpr int A0_BYTES = TILE_M * ROWB0;
    static constexpr int W0_CHUNK_PART = N0 * ROWB0, W0_CHUNK = 2 * W0_CHUNK_PART, W0_BYTES = MAX_NCH * W0_CHUNK;
    static constexpr int W2_BYTES = TILE_N * DP * 4;
    static constexpr int B_OFF = 0;
    static constexpr int A1_OFF = B_OFF + NB * B_STAGE;
    static constexpr int A0_OFF = A1_OFF + 2 * NS * A1_SLOT;
    static constexpr int W0_OFF = A0_OFF + 2 * A0_BYTES;
    static constexpr int W2_OFF = W0_OFF + 2 * W0_BYTES;
    static constexpr int BAR_OFF = W2_OFF + 2 * W2_BYTES;
    static constexpr int NBARS = 2 * NB + 4 * NS + 14;
    static constexpr int GATE_OFF = BAR_OFF + NBARS * 8 + 16;    // epilogue gate words (TAN): [track][trip][row]
    static constexpr int TOTAL = GATE_OFF + 2 * MAX_NCH * TILE_M * 4;
    static constexpr int ALIGN_PAD = 512;
};

// ---- one-time images (global memory, L2 resident) -------------------------------------------
// scale[0] = power of two with max(|W1|, |b1|) * scale in [2^13, 2^14]; scale[1] = 1 / scale[0]
__global__ void prep_scale_kernel(const float* W1, const float* b1, int H0, int H1, float* scale) {
    __shared__ float red[256];
    float m = 0.f;
    for (int i = threadIdx.x; i < H0 * H1; i += blockDim.x) m = fmaxf(m, fabsf(W1[i]));
    for (int i = threadIdx.x; i < H1; i += blockDim.x) m = fmaxf(m, fabsf(b1[i]));
    red[threadIdx.x] = m;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] = fmaxf(red[threadIdx.x], red[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int e = 0;
        const float mx = red[0];
        if (mx > 0.f && isfinite(mx)) { frexpf(mx, &e); e = 14 - e; }      // mx = f * 2^(e0), f in [0.5, 1)
        e = e > 24 ? 24 : (e < -24 ? -24 : e);
        scale[0] = ldexpf(1.f, e);
        scale[1] = ldexpf(1.f, -e);
    }
}
// Per-particle compaction lists.  A unit is KEPT when its mask is >= DROP_BELOW (NaN masks are kept too): below
// that its contribution is under half an ulp of any sum it enters.  idx0[p][q] / idx1[p][c] = q-th / c-th kept
// unit of layer 0 / layer 1 (ascending), meta[p] = {K-blocks, accumulator columns, kept layer-0 units, kept
// layer-1 units}: the K range is the kept layer-0 units followed by the bias unit, rounded up to 16.
constexpr float DROP_BELOW = 5.9604645e-8f;    // 2^-24
constexpr int META = 4;
static_assert(META == IMG_META, "bnn_mlp_iface.h sizes");
__global__ void prep_index_kernel(const float* mask0 /*[P][H0]*/, const float* mask1 /*[P][H1]*/, int P, int H0, int H1,
                                  int* idx0 /*[P][TILE_N]*/, int* idx1 /*[P][TILE_N]*/, int* meta /*[P][META]*/) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    int n0 = 0, n1 = 0;
    for (int n = 0; n < H0; ++n)
        if (!(mask0[(size_t)p * H0 + n] < DROP_BELOW)) idx0[(size_t)p * TILE_N + n0++] = n;
    for (int c = 0; c < H1; ++c)
        if (!(mask1[(size_t)p * H1 + c] < DROP_BELOW)) idx1[(size_t)p * TILE_N + n1++] = c;
    const int ncol = (n1 + 15) & ~15;
    meta[p * META + 0] = (n0 + 1 + KB - 1) / KB;
    meta[p * META + 1] = ncol < 16 ? 16 : ncol;
    meta[p * META + 2] = n0;
    meta[p * META + 3] = n1;
}
// W1 image of particle p: [K-block][N(p) rows x (b0[16] | b1[16]) fp16] SWIZZLE_64B, scaled; row c is kept layer-1
// unit idx1[p][c], K position q is kept layer-0 unit idx0[p][q], position n0 (the bias unit) carries b1.  Blocks sit
// B_STAGE bytes apart; only the first N(p) * 64 bytes of a block are read.
constexpr size_t W1_PSTRIDE = (size_t)13 * 208 * 64;       // MAX_NKB * B_STAGE
static_assert(W1_PSTRIDE == IMG_W1_PSTRIDE && TILE_N == IMG_TILE_N, "bnn_mlp_iface.h sizes");
__global__ void prep_w1_kernel(const float* W1 /*[H1][H0]*/, const float* b1, int P, int H0, int H1, const int* idx0,
                               const int* idx1, const int* meta, const float* scale, unsigned char* img) {
    const long long total = (long long)P * MAX_NKB * TILE_N * KB;
    const float sc = scale[0];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int p = (int)(i / (MAX_NKB * TILE_N * KB)), rem0 = (int)(i - (long long)p * (MAX_NKB * TILE_N * KB));
        const int kb = rem0 / (TILE_N * KB), rem = rem0 - kb * TILE_N * KB;
        const int n = rem / KB, kk = rem - n * KB, k = kb * KB + kk;
        const int nkb = meta[p * META], ncol = meta[p * META + 1], n0 = meta[p * META + 2], n1 = meta[p * META + 3];
        if (kb >= nkb || n >= ncol) continue;
        float w = 0.f;
        if (n < n1) {
            const int c = idx1[(size_t)p * TILE_N + n];
            w = k < n0 ? W1[(size_t)c * H0 + idx0[(size_t)p * TILE_N + k]] : (k == n0 ? b1[c] : 0.f);
        }
        w *= sc;
        const __half h0 = __float2half_rn(w);
        const __half h1 = __float2half_rn(w - __half2float(h0));
        // element kk of [b0 | b1] sits at 2-byte index kk (b0) or 16 + kk (b1) of the 64-byte row
        unsigned char* row = img + (size_t)p * W1_PSTRIDE + (size_t)kb * B_STAGE + (n >> 3) * 512 + (n & 7) * 64;
        const int sw = (n >> 1) & 3;
        *reinterpret_cast<__half*>(row + (((kk >> 3) ^ sw) << 4) + (kk & 7) * 2) = h0;
        *reinterpret_cast<__half*>(row + (((2 + (kk >> 3)) ^ sw) << 4) + (kk & 7) * 2) = h1;
    }
}
// Per-particle layer-0 image: [P][chunk][X | Y][32 rows], split FP16 like layer 1: with w = b0 + b1 the row
// of part X is [b0 | b0] and of part Y is [b1 | 0], so that against the operand row [a0 | a1]
// X gives a0*b0 + a1*b0 and Y gives a0*b1.  Row q < n0(p) is m0[p][n]*[W0[n][:], b0[n]] of kept unit n = idx0[p][q],
// row n0(p) is the unit vector of the bias column (the constant-1 hidden unit), the rest zero.
template <int K0P>
__global__ void prep_w0_kernel(const float* W0 /*[H0][K0]*/, const float* b0, const float* mask0 /*[P][H0]*/, int P,
                               int H0, int K0, const int* idx0, const int* meta, unsigned char* img) {
    typedef Cfg<K0P, 4> C;
    const int total = P * MAX_NCH * N0 * K0P;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int p = i / (MAX_NCH * N0 * K0P), rem = i - p * (MAX_NCH * N0 * K0P);
        const int j = rem / (N0 * K0P), rem2 = rem - j * (N0 * K0P);
        const int rr = rem2 / K0P, k = rem2 - rr * K0P, q = j * N0 + rr, n0 = meta[p * META + 2];
        float w = 0.f;
        if (q < n0) {
            const int n = idx0[(size_t)p * TILE_N + q];
            w = mask0[(size_t)p * H0 + n] * (k < K0 ? W0[(size_t)n * K0 + k] : (k == K0 ? b0[n] : 0.f));
        } else if (q == n0) w = k == K0 ? 1.f : 0.f;
        const __half h0 = __float2half_rn(w);
        const __half h1 = __float2half_rn(w - __half2float(h0));
        unsigned char* base = img + (size_t)p * C::W0_BYTES + (size_t)j * C::W0_CHUNK;
        *reinterpret_cast<__half*>(base + swz_byte<C::ROWB0>(rr, 2 * k)) = h0;
        *reinterpret_cast<__half*>(base + swz_byte<C::ROWB0>(rr, 2 * (K0P + k))) = h0;
        *reinterpret_cast<__half*>(base + C::W0_CHUNK_PART + swz_byte<C::ROWB0>(rr, 2 * k)) = h1;
        *reinterpret_cast<__half*>(base + C::W0_CHUNK_PART + swz_byte<C::ROWB0>(rr, 2 * (K0P + k))) = __float2half_rn(0.f);
    }
}
// Per-particle output weights m1[p][c] * W2[o][c] / scale (mean head only, o < D), stored per COLUMN PAIR as
// W2p[p][c / 2][o][c % 2] when D <= 4 (the epilogue's FFMA2 takes (column 2j, column 2j+1) of one output as a 64-bit
// operand), as W2p[p][c][o] otherwise
__global__ void prep_w2_kernel(const float* W2 /*[2D][H1]*/, const float* mask1 /*[P][H1]*/, int P, int H1, int D, int DP,
                               const int* idx1, const int* meta, const float* scale, float* out) {
    const bool pairs = D <= 4;
    const int total = P * TILE_N * DP;
    const float inv = scale[1];              // the layer-1 accumulator carries the W1 image's scale
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int p = i / (TILE_N * DP), rem = i - p * (TILE_N * DP);
        const int jp = rem / (2 * DP), rem2 = rem - jp * (2 * DP);
        const int o = pairs ? rem2 >> 1 : rem % DP, c = pairs ? 2 * jp + (rem2 & 1) : rem / DP;
        float v = 0.f;                           // accumulator column c of particle p is kept layer-1 unit idx1[p][c]
        if (c < meta[p * META + 3] && o < D) {
            const int u = idx1[(size_t)p * TILE_N + c];
            v = mask1[(size_t)p * H1 + u] * W2[(size_t)o * H1 + u] * inv;
        }
        out[i] = v;
    }
}


// ---- tile schedule ------------------------------------------------------------------------------------------
// The CTA owns super-tiles [T0, T1) (tau = particle * tiles_p + item block).  A SEGMENT is the run of super-tiles of
// one particle inside that range: within a segment track 0 takes the 1st, 3rd, ... and track 1 the 2nd, 4th, ...
// super-tile, and the W1 stream carries that particle's image: len = max over the tracks of the blocks they
// consume (track 1 starts `skew` blocks into the segment, so the epilogues of the two tracks interleave).
struct Seg {
    int ta, cnt, p, nkb, ncol, skew, n[2], len;
};
// K-blocks by which track 1 trails track 0 in the W1 stream of a particle with nkb K-blocks: about half a tile, and
// even, because a layer-0 chunk (32 hidden units) is two K-blocks and the tracks walk them from chunk boundaries
__device__ __forceinline__ int track_skew(int nkb) { return (nkb / 2) & ~1; }
__device__ __forceinline__ bool seg_at(int ta, int T1, int tiles_p, const int* meta, int rpp, Seg& s) {
    if (ta >= T1) return false;
    s.ta = ta;
    s.p = ta / tiles_p;
    const int end = min((s.p + 1) * tiles_p, T1);
    s.cnt = end - ta;
    s.nkb = __ldg(meta + s.p * META);
    s.ncol = __ldg(meta + s.p * META + 1);
    s.skew = track_skew(s.nkb);
    s.n[0] = ((s.cnt + 1) / 2) * rpp;
    s.n[1] = (s.cnt / 2) * rpp;
    const int len0 = s.n[0] * s.nkb, len1 = s.n[1] ? s.skew + s.n[1] * s.nkb : 0;
    s.len = len0 > len1 ? len0 : len1;
    return true;
}
// the super-tiles of ONE track, in order, across segments.  Three registers of state (the worker roles run at the
// register cap): the kernel-uniform T1 / tiles_p / t / meta are passed in, particle and item block are recomputed
// from tau where they are needed (once per tile).
struct TrackIter {
    int seg_end, tau, kn;                                     // kn = nkb | ncol << 8 of the current particle; tau < 0: done
    __device__ __forceinline__ bool valid() const { return tau >= 0; }
    __device__ __forceinline__ int nkb() const { return kn & 255; }
    __device__ __forceinline__ int ncol() const { return kn >> 8; }
    __device__ __forceinline__ int skew() const { return track_skew(nkb()); }
    __device__ __forceinline__ int p(int tiles_p) const { return tau / tiles_p; }
    __device__ __forceinline__ void locate(int seg_start, int T1, int tiles_p, int t, const int* meta) {
        tau = -1;
        while (seg_start < T1) {
            const int pp = seg_start / tiles_p;
            const int end = min((pp + 1) * tiles_p, T1);
            if (seg_start + t < end) {
                tau = seg_start + t; seg_end = end;
                kn = __ldg(meta + pp * META) | (__ldg(meta + pp * META + 1) << 8);
                return;
            }
            seg_start = end;
        }
    }
    __device__ __forceinline__ void next(int T1, int tiles_p, int t, const int* meta) {
        tau += 2;
        if (tau >= seg_end) locate(seg_end, T1, tiles_p, t, meta);
    }
};

// What the epilogue's column loop does to one layer-1 pre-activation v, element e of a gate word of NE bits:
// EPI_RELU (rollout) and EPI_PRIMAL (first pass of a linearisation super-tile) apply the ReLU, EPI_PRIMAL also shifts the
// sign of v into the word (element e ends at bit NE-1-e); EPI_TANGENT zeroes v where the primal's sign bit is set.
enum { EPI_RELU, EPI_PRIMAL, EPI_TANGENT };
template <int KIND, int NE>
__device__ __forceinline__ float epi_act(float v, uint32_t& word, int e) {
    if constexpr (KIND == EPI_PRIMAL) word = __funnelshift_l(__float_as_uint(v), word, 1);
    if constexpr (KIND == EPI_TANGENT) return (word & (1u << (NE - 1 - e))) ? 0.f : v;
    else return fmaxf(v, 0.f);
}

template <int GEO, bool TAN>
__global__ void __launch_bounds__(THREADS, 1)
bnn_mlp_tc_kernel(const BnnMlpArgs<float> a, const Images im, int S, int tiles_p) {
    typedef Geo<GEO> G;
    constexpr int D = G::D, DA = G::DA, NNA = G::NNA, NANG = G::NANG, K0 = DA + G::NU;
    constexpr int K0P = K0 + 1 <= 8 ? 8 : 16, DP = D <= 4 ? 4 : 8;
    typedef Cfg<K0P, DP> C;
    constexpr int NB = C::NB, NS = C::NS, ROWB0 = C::ROWB0;
    constexpr int TD = TAN ? D + G::NU : 0, RPP = 1 + TD;     // passes per super-tile: primal + one per tangent direction
    constexpr uint32_t IDESC0 = idesc_f16(TILE_M, N0);

    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + C::ALIGN_PAD - 1) & ~(uintptr_t)(C::ALIGN_PAD - 1));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::BAR_OFF);
    uint64_t* b_full = bars;                 // [NB]
    uint64_t* b_empty = b_full + NB;         // [NB]
    uint64_t* a1_full = b_empty + NB;        // [2][NS]
    uint64_t* a1_empty = a1_full + 2 * NS;   // [2][NS]
    uint64_t* acc0_full = a1_empty + 2 * NS; // [2]
    uint64_t* acc0_empty = acc0_full + 2;
    uint64_t* a0_full = acc0_empty + 2;
    uint64_t* acc1_full = a0_full + 2;
    uint64_t* acc1_empty = acc1_full + 2;
    uint64_t* w0_full = acc1_empty + 2;
    uint64_t* w2_full = w0_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + C::NBARS);

    const BnnNet<float>& n = a.net;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int P = n.P;

    // ---- tile schedule.  A super-tile is 128 items (rollout: (problem, alpha) pairs; linearise:
    // problems) of one particle; it is RPP consecutive MMA tiles ("passes") on one track: the primal
    // rows, then one pass per tangent direction -- so a thread sees the primal and the tangent
    // pre-activations of the same (item, hidden unit) and the ReLU gate never crosses lanes.
    // Each CTA owns a contiguous range of super-tiles; track t takes every other one.  Track 1 is
    // `skew` K-blocks behind track 0 in the W1 stream.
    const long long NT = (long long)P * tiles_p;            // < 2^31 (checked by the launcher)
    const int T0 = (int)(NT * blockIdx.x / gridDim.x), T1 = (int)(NT * (blockIdx.x + 1) / gridDim.x);

    if (tid == 0) {
        for (int s = 0; s < NB; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 2); }   // both tracks release a W1 stage
        for (int s = 0; s < 2 * NS; ++s) { mbar_init(&a1_full[s], 128); mbar_init(&a1_empty[s], 1); }
        for (int t = 0; t < 2; ++t) {
            mbar_init(&acc0_full[t], 1);
            mbar_init(&acc0_empty[t], 128);
            mbar_init(&a0_full[t], 128);
            mbar_init(&acc1_full[t], 1);
            mbar_init(&acc1_empty[t], 128);
            mbar_init(&w0_full[t], 1);
            mbar_init(&w2_full[t], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // Register re-balancing between the roles (640 threads -> 96 registers per thread at launch): the warpgroup of
    // the loader / issuer warps (16-19) needs ~40, the four worker warpgroups run at the cap and spilled (the
    // tangent instantiations: gate words + packed accumulators + TMEM fragments).  56 x 128 + 104 x 512 <= 96 x 640.
    // (The instruction sits at the top of each role's branch so that it dominates exactly that role's code.)
    if (warp >= 16) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (warp == 18) {
        // ================= loader: W1 K-blocks, shared by both tracks =================
        if (lane == 0) {
            uint32_t s = 0, ph = 1;
            Seg sg;
            for (bool live = seg_at(T0, T1, tiles_p, im.meta, RPP, sg); live; live = seg_at(sg.ta + sg.cnt, T1, tiles_p, im.meta, RPP, sg)) {
                const unsigned char* img = im.W1img + (size_t)sg.p * W1_PSTRIDE;
                const uint32_t bytes = (uint32_t)sg.ncol * 64u;
                int kb = 0;
                for (int nb = 0; nb < sg.len; ++nb) {
                    mbar_wait(&b_empty[s], ph);
                    mbar_expect_tx(&b_full[s], bytes);
                    bulk_g2s(smem + C::B_OFF + s * B_STAGE, img + (size_t)kb * B_STAGE, bytes, &b_full[s]);
                    if (++s == NB) { s = 0; ph ^= 1; }
                    if (++kb == sg.nkb) kb = 0;
                }
            }
        }
    } else if (warp == 19) {
        // ================= layer-0 issuer (one thread, both tracks, polling): chunk c+1 of a track is
        // issued the moment its mid-stage has drained chunk c, independent of where layer 1 stands ====
        if (lane == 0) {
            uint32_t l0cnt[2] = {0, 0}, w0loads[2] = {0, 0};
            int curp[2] = {-1, -1}, k[2] = {0, 0}, pos[2] = {0, 0}, d[2] = {0, 0};   // k = tiles issued (track-global), d = pass
            int tp[2];                             // particle of the track's current super-tile (a division: not in the poll loop)
            bool fresh[2] = {true, true};          // next chunk is the first of its tile
            TrackIter it[2];
            it[0].locate(T0, T1, tiles_p, 0, im.meta);
            it[1].locate(T0, T1, tiles_p, 1, im.meta);
            tp[0] = it[0].valid() ? it[0].p(tiles_p) : -1;
            tp[1] = it[1].valid() ? it[1].p(tiles_p) : -1;
            while (it[0].valid() || it[1].valid()) {
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    if (!it[t].valid()) continue;
                    const int nkb = it[t].nkb(), skew = it[t].skew();
                    if (fresh[t]) {
                        const int p = tp[t];
                        if (p != curp[t]) {
                            if (!mbar_test(&w0_full[t], w0loads[t] & 1)) continue;
                            ++w0loads[t];
                            curp[t] = p;
                        }
                        if (!mbar_test(&a0_full[t], (uint32_t)k[t] & 1)) continue;
                        fresh[t] = false;
                    }
                    if (!mbar_test(&acc0_empty[t], (l0cnt[t] & 1) ^ 1)) continue;
                    tc_fence_after();
                    int kb = t * skew + pos[t];
                    if (kb >= nkb) kb -= nkb;
                    const int nk = kb + 1 < nkb ? 2 : 1, j = kb >> 1;
                    const uint32_t d_tmem = tmem_base + (uint32_t)(t * TM_TRACK + TM_ACC0);
                    const uint32_t a0 = smem_u32(smem + C::A0_OFF + t * C::A0_BYTES);
                    const uint32_t b0 = smem_u32(smem + C::W0_OFF + t * C::W0_BYTES + j * C::W0_CHUNK);
                    const uint64_t ad = make_desc<ROWB0>(a0);
                    const uint64_t bx = make_desc<ROWB0>(b0), by = make_desc<ROWB0>(b0 + C::W0_CHUNK_PART);
                    // one K-step = 32 B of a row = 16 fp16: K0P = 8 -> [a0 | a1] in one step; K0P = 16 -> a0, then a1
                    tc_mma_f16(d_tmem, ad, bx, IDESC0, 0);                          // a0*b0 (+ a1*b0)
                    if (K0P == 16) tc_mma_f16(d_tmem, ad + 2, bx + 2, IDESC0, 1);   // a1*b0
                    tc_mma_f16(d_tmem, ad, by, IDESC0, 1);                          // a0*b1
                    tc_commit(&acc0_full[t]);
                    ++l0cnt[t];
                    pos[t] += nk;
                    if (pos[t] >= nkb) {
                        pos[t] = 0; ++k[t]; fresh[t] = true;
                        if (++d[t] == RPP) { d[t] = 0; it[t].next(T1, tiles_p, t, im.meta); tp[t] = it[t].valid() ? it[t].p(tiles_p) : -1; }
                    }
                }
            }
        }
    } else {
        // ================= layer-1 issuers: one thread per track (a track that waits for its epilogue
        // or its mid-stage does not hold the other one up; they drift at most NB W1 stages apart) ====
        // The whole warp runs the loop with warp-uniform state (so the compiler keeps it in uniform
        // registers and feeds UTCHMMA without per-operand R2UR / elect loops: the single-lane version
        // spent ~1000 cycles of dependent scalar code per step for 318 cycles of MMA); one elected lane
        // issues.  Descriptors advance by adding to their low word (address field, 16-byte units).
        {
            const int t = __shfl_sync(0xffffffffu, warp, 0) - 16;
            const bool leader = elect_one();
            const uint32_t d_tmem = tmem_base + (uint32_t)(t * TM_TRACK + TM_ACC1);
            const uint64_t desc_hi = make_desc<64>(0) & 0xFFFFFFFF00000000ull;
            const uint32_t a_lo0 = (uint32_t)make_desc<64>(smem_u32(smem + C::A1_OFF + t * NS * A1_SLOT));
            const uint32_t b_lo0 = (uint32_t)make_desc<64>(smem_u32(smem + C::B_OFF));
            uint64_t* const a1f = a1_full + t * NS;
            uint64_t* const a1e = a1_empty + t * NS;
            uint32_t s = 0, bph = 0, slot = 0, sph = 0;
            int kg = 0;                                      // tiles of this track so far (accumulator phase)
            long long tr_wb = 0, tr_wa = 0, tr_is = 0;
            Seg sg;
            for (bool live = seg_at(T0, T1, tiles_p, im.meta, RPP, sg); live; live = seg_at(sg.ta + sg.cnt, T1, tiles_p, im.meta, RPP, sg)) {
            const int ntiles = t == 0 ? sg.n[0] : sg.n[1], first_blk = t * sg.skew, nkb = sg.nkb;
            const uint32_t IDESC1 = idesc_f16(TILE_M, sg.ncol);
            int k = 0, pos = 0;
            for (int nb = 0; nb < sg.len; ++nb) {
                long long tq0 = TCLK();
                mbar_wait(&b_full[s], bph);
                tr_wb += TCLK() - tq0;
                if (nb < first_blk || k >= ntiles) {
                    if (leader) mbar_arrive(&b_empty[s]);   // this track does not use the block
                } else {
                    long long tq1 = TCLK();
                    if (pos == 0) { if (leader) TR(t, kg * 8 + 0, tq1); }
                    if (pos == 0) mbar_wait(&acc1_empty[t], ((uint32_t)kg & 1) ^ 1);
                    long long tq2 = TCLK();
                    if (pos == 0) { if (leader) TR(t, kg * 8 + 1, tq2); }
                    mbar_wait(&a1f[slot], sph);
                    long long tq3 = TCLK();
                    tr_wa += tq3 - tq2;
                    tc_fence_after();
                    if (leader) {
                        const uint64_t ad = desc_hi | (uint64_t)(a_lo0 + slot * (A1_SLOT >> 4));
                        const uint64_t bd = desc_hi | (uint64_t)(b_lo0 + s * (B_STAGE >> 4));
                        // one UMMA K-step = 32 B of a row = 16 fp16: [x0 | x1] halves are +2 apart in the >>4 address field
                        tc_mma_f16(d_tmem, ad, bd, IDESC1, pos != 0);     // a0 * b0
                        tc_mma_f16(d_tmem, ad, bd + 2, IDESC1, 1);        // a0 * b1
                        tc_mma_f16(d_tmem, ad + 2, bd, IDESC1, 1);        // a1 * b0
                        tc_commit(&a1e[slot]);
                        tc_commit(&b_empty[s]);
                        if (pos == nkb - 1) tc_commit(&acc1_full[t]);
                    }
                    __syncwarp();
                    tr_is += TCLK() - tq3;
                    if (pos == nkb - 1 && leader) {
                        TR(t, kg * 8 + 2, TCLK()); TR(t, kg * 8 + 3, tr_wb); TR(t, kg * 8 + 4, tr_wa); TR(t, kg * 8 + 5, tr_is);
                        tr_wb = tr_wa = tr_is = 0;
                    }
                    if (++slot == NS) { slot = 0; sph ^= 1; }
                    if (++pos == nkb) { pos = 0; ++k; ++kg; }
                }
                if (++s == NB) { s = 0; bph ^= 1; }
            }
            }
        }
    }
    } else {
        // ================= worker teams: warps 0-7 epilogue (track 0, 1), warps 8-15 mid-stage =================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
        const int team = warp >> 2, t = team & 1;
        const int r = tid & 127, w = r >> 5;                  // w = TMEM lane quarter of this warp
        const uint32_t track_taddr = tmem_base + (uint32_t)(t * TM_TRACK);
        TrackIter cur;
        cur.locate(T0, T1, tiles_p, t, im.meta);
        if (!cur.valid()) goto done;
        if (team >= 2) {
            // ---------------- mid-stage (thread = row r): inputs -> A0, layer-0 accumulator -> A1 ----------------
            const uint32_t A0 = smem_u32(smem + C::A0_OFF + t * C::A0_BYTES);
            const uint32_t lane_taddr = track_taddr + ((uint32_t)(w * 32) << 16);
            const uint32_t row_off = (uint32_t)((r >> 3) * 512 + (r & 7) * 64), row_sw = (uint32_t)((r >> 1) & 3);   // SWIZZLE_64B row
            float inc[K0], inn[K0];            // features [aug(x), u] of this row's item: current / next super-tile
            bool vc = false, vn = false;
            uint32_t gate[MAX_NCH];            // sign bits of the primal pre-activations, one word per chunk (TAN)
#pragma unroll
            for (int j = 0; j < MAX_NCH; ++j) gate[j] = 0;
            auto fetch = [&](const TrackIter& st) {   // item r of a super-tile: particle p, item i -> global row i*P + p
                const int p = st.p(tiles_p), l = st.tau - p * tiles_p;
                const int i = l * TILE_M + r;
                vn = i < S;
#pragma unroll
                for (int k = 0; k < K0; ++k) inn[k] = 0.f;
                if (vn) {
                    float x[D];
                    const float* xp = a.X + ((size_t)i * P + p) * D;
                    if (D % 4 == 0) {
#pragma unroll
                        for (int e = 0; e < D; e += 4) *reinterpret_cast<float4*>(x + e) = __ldg(reinterpret_cast<const float4*>(xp + e));
                    } else {
#pragma unroll
                        for (int e = 0; e < D; e += 2) *reinterpret_cast<float2*>(x + e) = __ldg(reinterpret_cast<const float2*>(xp + e));
                    }
#pragma unroll
                    for (int i2 = 0; i2 < NNA; ++i2) inn[i2] = x[G::nonang(i2)];
#pragma unroll
                    for (int i2 = 0; i2 < NANG; ++i2) { inn[NNA + 2 * i2] = sinf(x[G::ang(i2)]); inn[NNA + 2 * i2 + 1] = cosf(x[G::ang(i2)]); }
#pragma unroll
                    for (int j = 0; j < G::NU; ++j) inn[DA + j] = __ldg(a.u + (size_t)i * G::NU + j);
                }
            };
            auto write_a0 = [&](int d) {       // [norm(aug(x), u), 1] (d == 0) or its tangent along direction d-1
                float row[K0P];
#pragma unroll
                for (int k = 0; k < K0P; ++k) row[k] = 0.f;
                if (vc) {
                    float sc[K0];
#pragma unroll
                    for (int k = 0; k < K0; ++k) sc[k] = n.X_std_inv ? n.X_std_inv[k] : 1.f;
                    if (!TAN || d == 0) {
#pragma unroll
                        for (int k = 0; k < K0; ++k) row[k] = (inc[k] - (n.X_mean ? n.X_mean[k] : 0.f)) * sc[k];
                        row[K0] = 1.f;
                    } else {
                        const int dir = d - 1;
#pragma unroll
                        for (int i2 = 0; i2 < NNA; ++i2) if (dir == G::nonang(i2)) row[i2] = sc[i2];
#pragma unroll
                        for (int i2 = 0; i2 < NANG; ++i2) if (dir == G::ang(i2)) {
                            row[NNA + 2 * i2] = inc[NNA + 2 * i2 + 1] * sc[NNA + 2 * i2];          // d sin = cos
                            row[NNA + 2 * i2 + 1] = -inc[NNA + 2 * i2] * sc[NNA + 2 * i2 + 1];     // d cos = -sin
                        }
#pragma unroll
                        for (int j = 0; j < G::NU; ++j) if (dir == D + j) row[DA + j] = sc[DA + j];
                    }
                }
                uint32_t x0[K0P / 2], x1[K0P / 2];       // fp16 pairs: x0 = fp16(row), x1 = fp16(row - x0)
#pragma unroll
                for (int e = 0; e < K0P / 2; ++e) {
                    x0[e] = pack_f16(row[2 * e], row[2 * e + 1]);
                    const float2 back = unpack_f16(x0[e]);
                    x1[e] = pack_f16(row[2 * e] - back.x, row[2 * e + 1] - back.y);
                }
#pragma unroll
                for (int c = 0; c < K0P / 8; ++c) {      // 16-byte chunks: [x0 ...][x1 ...]
                    sts128(A0 + swz_byte<ROWB0>(r, 16 * c), x0[4 * c], x0[4 * c + 1], x0[4 * c + 2], x0[4 * c + 3]);
                    sts128(A0 + swz_byte<ROWB0>(r, 16 * (K0P / 8 + c)), x1[4 * c], x1[4 * c + 1], x1[4 * c + 2], x1[4 * c + 3]);
                }
                fence_async_smem();
                mbar_arrive(&a0_full[t]);
            };
            auto load_w0 = [&](int p, int nkb_p) {     // the chunks this particle uses: 32 hidden units = 2 K-blocks each
                const uint32_t w0_bytes = (uint32_t)((nkb_p + 1) / 2) * C::W0_CHUNK;
                mbar_expect_tx(&w0_full[t], w0_bytes);
                bulk_g2s(smem + C::W0_OFF + t * C::W0_BYTES, im.W0img + (size_t)p * C::W0_BYTES, w0_bytes, &w0_full[t]);
            };
            int curp = cur.p(tiles_p);
            if (r == 0) load_w0(curp, cur.nkb());
            fetch(cur);
#pragma unroll
            for (int k = 0; k < K0; ++k) inc[k] = inn[k];
            vc = vn;
            write_a0(0);
            uint32_t ci = 0, slot = 0, sph = 1;
            TrackIter nxt = cur;
            nxt.next(T1, tiles_p, t, im.meta);
            int d = 0;                         // pass of the current tile inside its super-tile
            int tr_k = 0;
            while (cur.valid()) {
                long long tr_w0 = 0, tr_w1 = 0, tr_t0 = TCLK();
                const bool last_pass = d == RPP - 1;
                const bool more = !last_pass || nxt.valid();        // another tile follows on this track
                const int nkb = cur.nkb(), kb0 = t * cur.skew();
                if (last_pass && nxt.valid()) fetch(nxt);
                for (int pos = 0; pos < nkb;) {
                    int kb = kb0 + pos;
                    if (kb >= nkb) kb -= nkb;
                    const int nk = kb + 1 < nkb ? 2 : 1, j = kb >> 1;
                    float v[32];
                    long long tq0 = TCLK();
                    mbar_wait(&acc0_full[t], ci & 1);
                    tr_w0 += TCLK() - tq0;
                    ++ci;
                    tc_fence_after();
                    tc_ld32(lane_taddr + TM_ACC0, v);
                    tc_wait_ld32(v);
                    tc_fence_before();
                    mbar_arrive(&acc0_empty[t]);
                    if (pos + nk >= nkb && more) {
                        // every layer-0 MMA of this tile has completed: A0 (and, between super-tiles, the W0 image) is free
                        if (last_pass) {
                            const int pn = nxt.p(tiles_p);
                            if (pn != curp) { if (r == 0) load_w0(pn, nxt.nkb()); curp = pn; }
#pragma unroll
                            for (int k2 = 0; k2 < K0; ++k2) inc[k2] = inn[k2];
                            vc = vn;
                            write_a0(0);
                        } else {
                            write_a0(d + 1);
                        }
                    }
                    if (!TAN) {
#pragma unroll
                        for (int e = 0; e < 32; ++e) v[e] = fmaxf(v[e], 0.f);
                    } else if (d == 0) {
                        uint32_t word = 0;
#pragma unroll
                        for (int e = 0; e < 32; ++e) {
                            word = __funnelshift_l(__float_as_uint(v[e]), word, 1);     // sign of v[e] ends up at bit 31 - e
                            v[e] = fmaxf(v[e], 0.f);
                        }
#pragma unroll
                        for (int jj = 0; jj < MAX_NCH; ++jj) if (jj == j) gate[jj] = word;
                    } else {
                        uint32_t word = 0;
#pragma unroll
                        for (int jj = 0; jj < MAX_NCH; ++jj) if (jj == j) word = gate[jj];
#pragma unroll
                        for (int e = 0; e < 32; ++e) v[e] = (word & (0x80000000u >> e)) ? 0.f : v[e];
                    }
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        if (h < nk) {
                            long long tq1 = TCLK();
                            mbar_wait(&a1_empty[t * NS + slot], sph);
                            tr_w1 += TCLK() - tq1;
                            const uint32_t A1 = smem_u32(smem + C::A1_OFF + (t * NS + slot) * A1_SLOT) + row_off;
                            uint32_t a0[8], a1[8];            // fp16 pairs: a0 = fp16(v), a1 = fp16(v - a0)
#pragma unroll
                            for (int e = 0; e < 8; ++e) {
                                const float v0 = v[16 * h + 2 * e], v1 = v[16 * h + 2 * e + 1];
                                a0[e] = pack_f16(v0, v1);
                                const float2 back = unpack_f16(a0[e]);
                                a1[e] = pack_f16(v0 - back.x, v1 - back.y);
                            }
#pragma unroll
                            for (int c = 0; c < 2; ++c) {     // 16-byte chunks 0,1 = a0[0..7], a0[8..15]; 2,3 = a1
                                sts128(A1 + ((c ^ row_sw) << 4), a0[4 * c], a0[4 * c + 1], a0[4 * c + 2], a0[4 * c + 3]);
                                sts128(A1 + (((2 + c) ^ row_sw) << 4), a1[4 * c], a1[4 * c + 1], a1[4 * c + 2], a1[4 * c + 3]);
                            }
                            fence_async_smem();
                            mbar_arrive(&a1_full[t * NS + slot]);
                            if (++slot == NS) { slot = 0; sph ^= 1; }
                        }
                    }
                    pos += nk;
                }
                if (r == 0) { TR(4 + t, tr_k * 4 + 0, tr_t0); TR(4 + t, tr_k * 4 + 1, TCLK()); TR(4 + t, tr_k * 4 + 2, tr_w0); TR(4 + t, tr_k * 4 + 3, tr_w1); }
                ++tr_k;
                if (++d == RPP) { d = 0; cur = nxt; nxt.next(T1, tiles_p, t, im.meta); }
            }
        } else {
            // ---------------- epilogue: layer-1 accumulator -> ReLU -> output layer -> X', dX'/d(X,u) ----------------
            // 16x256b TMEM fragments: this thread holds rows 32w + 16hf + 8hb + lane/4 (hf, hb in {0,1}) and, of
            // every group of 8 columns, columns 2*(lane%4) and +1 -- so one pair of LDS.128 of the output weights
            // feeds 4 rows (a thread-per-row layout needs a broadcast LDS.128 per column: 4x the shared-memory
            // wavefronts, and this kernel is bound by the shared-memory pipe).  Column sums are completed
            // across the 4 lanes of a quad with two shuffles per value.
            const uint32_t W2s = smem_u32(smem + C::W2_OFF + t * C::W2_BYTES);
            const int q4 = lane & 3, rq = lane >> 2;
            int curp = -1;
            uint32_t w2loads = 0;
            // sign bits of this thread's (up to 208) primal pre-activations (TAN), one word per 32-column trip
            const uint32_t gate_s = smem_u32(smem + C::GATE_OFF) + (uint32_t)(t * MAX_NCH * TILE_M + r) * 4u;
            int d = 0;
            for (int k = 0; cur.valid(); ++k) {   // k = tiles of this track so far (accumulator phase)
                const int p = cur.p(tiles_p), l = cur.tau - p * tiles_p, ncol = cur.ncol();
                if (p != curp) {
                    named_bar_sync(1 + t, 128);      // every warp of the team is done with the old weights
                    if (r == 0) {
                        mbar_expect_tx(&w2_full[t], C::W2_BYTES);
                        bulk_g2s(smem + C::W2_OFF + t * C::W2_BYTES, im.W2p + (size_t)p * TILE_N * DP, C::W2_BYTES, &w2_full[t]);
                    }
                    mbar_wait(&w2_full[t], w2loads & 1);
                    ++w2loads;
                    curp = p;
                }
                // D <= 4: packed accumulators (even column, odd column) for FFMA2; wider outputs would spill them
                constexpr bool PK = D <= 4;
                unsigned long long y2[PK ? 4 : 1][PK ? D : 1];
                float y[4][D];
#pragma unroll
                for (int jr = 0; jr < 4; ++jr)
#pragma unroll
                    for (int o = 0; o < D; ++o) {
                        y[jr][o] = 0.f;
                        if constexpr (PK) y2[jr][o] = 0ull;
                    }
                // the primal pass adds X to the network's output: request it now, the accumulator is not ready yet anyway
                float xin[4][(D + 3) / 4];
                if (!TAN || d == 0) {
#pragma unroll
                    for (int oo = 0; oo < (D + 3) / 4; ++oo)
#pragma unroll
                        for (int jr = 0; jr < 4; ++jr) {
                            const int i = l * TILE_M + w * 32 + (jr >> 1) * 16 + (jr & 1) * 8 + rq, o = q4 + 4 * oo;
                            xin[jr][oo] = (i < S && o < D) ? __ldg(a.X + ((size_t)i * P + p) * D + o) : 0.f;
                        }
                }
                if (r == 0) TR(2 + t, k * 4 + 0, TCLK());
                mbar_wait(&acc1_full[t], (uint32_t)k & 1);
                if (r == 0) TR(2 + t, k * 4 + 1, TCLK());
                tc_fence_after();
                // half = 16 columns (two 8-column groups) of both row halves; consumes fragment buffer fb and
                // shifts (EPI_PRIMAL) / tests (EPI_TANGENT) bits [ebase, ebase+16) of the current gate word
                auto half = [&](const int c0, float (&fb)[2][8], uint32_t& word, auto kind_tag, auto ebase_tag, auto ne_tag) {
                    constexpr int KIND = decltype(kind_tag)::value, EBASE = decltype(ebase_tag)::value, NE = decltype(ne_tag)::value;
                    if constexpr (PK) {
#pragma unroll
                        for (int gi = 0; gi < 2; ++gi) {
                            // output weights of this thread's column pair, interleaved by prep_w2_kernel as [o][cc]: one 64-bit
                            // operand of FFMA2 per output (packed fp32 FMA: both columns of the pair in one instruction -- the
                            // output layer is 832 FMAs per thread and tile, and the epilogue's duration is on the critical
                            // path of a track: layer-1 MMAs of the next tile wait for it to release the accumulator)
                            unsigned long long w2p[DP];
#pragma unroll
                            for (int o2 = 0; o2 < DP / 2; ++o2) {
                                const float4 q = lds128f(W2s + (uint32_t)((((c0 + 8 * gi) / 2 + q4) * (2 * DP) + 4 * o2) * 4));
                                w2p[2 * o2] = pack2(q.x, q.y);
                                w2p[2 * o2 + 1] = pack2(q.z, q.w);
                            }
#pragma unroll
                            for (int hf = 0; hf < 2; ++hf)
#pragma unroll
                                for (int hb = 0; hb < 2; ++hb) {
                                    float vv[2];
#pragma unroll
                                    for (int cc = 0; cc < 2; ++cc) {
                                        vv[cc] = epi_act<KIND, NE>(fb[hf][4 * gi + 2 * hb + cc], word, EBASE + (gi * 2 + hf) * 4 + 2 * hb + cc);
                                    }
                                    const unsigned long long vp = pack2(vv[0], vv[1]);
#pragma unroll
                                    for (int o = 0; o < D; ++o) y2[2 * hf + hb][o] = ffma2(vp, w2p[o], y2[2 * hf + hb][o]);
                                }
                        }
                    } else {
#pragma unroll
                        for (int gi = 0; gi < 2; ++gi) {
                            float w2[2][DP];                                        // output weights of this thread's 2 columns
#pragma unroll
                            for (int cc = 0; cc < 2; ++cc)
#pragma unroll
                                for (int o4 = 0; o4 < DP / 4; ++o4)
                                    *reinterpret_cast<float4*>(&w2[cc][4 * o4]) =
                                        lds128f(W2s + (uint32_t)(((c0 + 8 * gi + 2 * q4 + cc) * DP + 4 * o4) * 4));
#pragma unroll
                            for (int hf = 0; hf < 2; ++hf)
#pragma unroll
                                for (int hb = 0; hb < 2; ++hb)
#pragma unroll
                                    for (int cc = 0; cc < 2; ++cc) {
                                        const float vv = epi_act<KIND, NE>(fb[hf][4 * gi + 2 * hb + cc], word, EBASE + (gi * 2 + hf) * 4 + 2 * hb + cc);
#pragma unroll
                                        for (int o = 0; o < D; ++o) y[2 * hf + hb][o] += vv * w2[cc][o];
                                    }
                        }
                    }
                };
                auto issue = [&](const int c0, float (&fb)[2][8]) {
                    const uint32_t ta = track_taddr + ((uint32_t)(w * 32) << 16) + TM_ACC1 + c0;
                    tc_ld_16x256b_x2(ta, fb[0]);
                    tc_ld_16x256b_x2(ta + (16u << 16), fb[1]);
                };
                // gate word of 32-column trip j: written by the primal pass, read by the tangent passes.  In shared
                // memory, not registers: the epilogue runs at the register cap, and a register array indexed by the
                // trip costs a 7-way select per trip.
                auto gate_put = [&](int j, uint32_t word) { sts32(gate_s + (uint32_t)(j * TILE_M * 4), word); };
                auto gate_get = [&](int j) -> uint32_t { return lds32(gate_s + (uint32_t)(j * TILE_M * 4)); };
                // ncol / 16 sixteen-column batches, two per trip of a ROLLED loop (a fully unrolled epilogue is 1 400 SASS
                // instructions: with five roles resident, instruction-cache misses were 26 % of its stall samples),
                // software pipelined over two fragment buffers: the TMEM loads of the next batch are issued right
                // after the wait for the current one (tcgen05.wait::ld waits for everything outstanding).
                // The pass kind is chosen once per tile: each kind has its own copy of the loop, carrying only its own
                // per-element work (a runtime kind inside the loop costs every element the work of all kinds).
                // (The fragment buffers live outside the lambda: declared inside it, they change how nvcc schedules the
                // rollout instantiation, whose code this split leaves as it was.)
                float fa[2][8], fb2[2][8];
                const int cfull = ncol & ~31;               // columns covered by whole 32-column trips
                auto columns = [&](auto kind_tag) {
                    constexpr int KIND = decltype(kind_tag)::value;
                    issue(0, fa);
                    int j = 0;
#pragma unroll 1
                    for (int c0 = 0; c0 < cfull; c0 += 32, ++j) {
                        uint32_t word = KIND == EPI_TANGENT ? gate_get(j) : 0u;
                        tc_wait_ld8(fa[0]); tc_wait_ld8(fa[1]);
                        issue(c0 + 16, fb2);
                        half(c0, fa, word, kind_tag, std::integral_constant<int, 0>(), std::integral_constant<int, 32>());
                        tc_wait_ld8(fb2[0]); tc_wait_ld8(fb2[1]);
                        if (c0 + 32 < ncol) issue(c0 + 32, fa);
                        half(c0 + 16, fb2, word, kind_tag, std::integral_constant<int, 16>(), std::integral_constant<int, 32>());
                        if (KIND == EPI_PRIMAL) gate_put(j, word);
                    }
                    if (cfull < ncol) {                      // one more 16-column batch
                        uint32_t word = KIND == EPI_TANGENT ? gate_get(j) : 0u;
                        tc_wait_ld8(fa[0]); tc_wait_ld8(fa[1]);
                        half(cfull, fa, word, kind_tag, std::integral_constant<int, 0>(), std::integral_constant<int, 16>());
                        if (KIND == EPI_PRIMAL) gate_put(j, word);
                    }
                };
                if constexpr (!TAN) columns(std::integral_constant<int, EPI_RELU>());
                else if (d == 0) columns(std::integral_constant<int, EPI_PRIMAL>());
                else columns(std::integral_constant<int, EPI_TANGENT>());
                tc_fence_before();
                mbar_arrive(&acc1_empty[t]);
                if (r == 0) TR(2 + t, k * 4 + 2, TCLK());
                // complete the column sums across the quad, then lane q4 writes outputs o = q4 (and q4 + 4)
#pragma unroll
                for (int jr = 0; jr < 4; ++jr)
#pragma unroll
                    for (int o = 0; o < D; ++o) {
                        if constexpr (PK) y[jr][o] = lo2(y2[jr][o]) + hi2(y2[jr][o]);
                        y[jr][o] += __shfl_xor_sync(0xffffffffu, y[jr][o], 1);
                        y[jr][o] += __shfl_xor_sync(0xffffffffu, y[jr][o], 2);
                    }
#pragma unroll
                for (int oo = 0; oo < (D + 3) / 4; ++oo) {
                    const int o = q4 + 4 * oo;
                    if (o < D) {
                        const float sd = n.dX_std ? n.dX_std[o] : 1.f, mn = n.dX_mean ? n.dX_mean[o] : 0.f, bo = n.b2[o];
#pragma unroll
                        for (int jr = 0; jr < 4; ++jr) {
                            const int i = l * TILE_M + w * 32 + (jr >> 1) * 16 + (jr & 1) * 8 + rq;
                            if (i < S) {
                                float yo = 0.f;
#pragma unroll
                                for (int o2 = 0; o2 < D; ++o2) if (o2 == o) yo = y[jr][o2];
                                const size_t g = (size_t)i * P + p;
                                if (!TAN || d == 0) a.Xn[g * D + o] = xin[jr][oo] + ((yo + bo) * sd + mn);
                                else a.Jp[(g * D + o) * TD + (d - 1)] = ((d - 1) == o ? 1.f : 0.f) + yo * sd;
                            }
                        }
                    }
                }
                if (r == 0) TR(2 + t, k * 4 + 3, TCLK());
                if (++d == RPP) { d = 0; cur.next(T1, tiles_p, t, im.meta); }
            }
        }
    }
done:
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base));
    }
}

}  // namespace tc
}  // namespace pddp
