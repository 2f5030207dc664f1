// The particle MLP of the BNN path: dispatch between the tcgen05 kernel (bnn_mlp_tc.cuh) and the CUDA-core kernel
// (bnn_mlp_simt.cuh), and the one-time weight images of the former.  Its own translation unit: the kernels are most of
// the library's compile time.   ref: pddp/models/bnn/modules.py:200-264
#include "bnn_mlp_simt.cuh"
#include "bnn_mlp_tc.cuh"
#include "profile.h"
#include <stdio.h>
#include <stdlib.h>

namespace pddp {

#define CK(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) return e__; } while (0)

static int g_num_sms = 0;
int num_sms() {
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_num_sms <= 0) g_num_sms = 148;
    }
    return g_num_sms;
}

// The tcgen05 kernel covers fp32 with hidden widths in (64, 207] x (64, 208] (H0 + 1 <= 208: the
// bias column); everything else (fp64, small nets) runs the SIMT kernel.  PDDP_FORCE_SIMT=1
// disables it (A/B comparisons, tools/tc_stats.py).
template <class T> bool use_tensor_cores(int H0, int H1) { return false; }
template bool use_tensor_cores<double>(int, int);
template <> bool use_tensor_cores<float>(int H0, int H1) {
    static int forced = -1;
    if (forced < 0) { const char* e = getenv("PDDP_FORCE_SIMT"); forced = (e && e[0] == '1') ? 1 : 0; }
    return !forced && H0 > 64 && H1 > 64 && H0 + 1 <= tc::MAX_NKB * tc::KB && H1 <= tc::TILE_N;
}


cudaError_t bnn_mlp_prep_images(int geo, const pddp_bnn* n, const tc::Images& im, cudaStream_t st) {
    const GeoDims g = geo_dims(geo);
    const int D = g.D, K0 = g.DA + g.NU;
    int* meta = const_cast<int*>(im.meta);
    tc::prep_index_kernel<<<(n->P + 63) / 64, 64, 0, st>>>((const float*)n->mask0, (const float*)n->mask1, n->P, n->H0, n->H1,
                                                           im.idx0, im.idx1, meta);
    tc::prep_scale_kernel<<<1, 256, 0, st>>>((const float*)n->W1, (const float*)n->b1, n->H0, n->H1,
                                             const_cast<float*>(im.scale));
    tc::prep_w1_kernel<<<592, 256, 0, st>>>((const float*)n->W1, (const float*)n->b1, n->P, n->H0, n->H1, im.idx0, im.idx1,
                                            meta, im.scale, const_cast<unsigned char*>(im.W1img));
    if (K0 + 1 <= 8)
        tc::prep_w0_kernel<8><<<64, 256, 0, st>>>((const float*)n->W0, (const float*)n->b0, (const float*)n->mask0,
                                                   n->P, n->H0, K0, im.idx0, meta, const_cast<unsigned char*>(im.W0img));
    else
        tc::prep_w0_kernel<16><<<64, 256, 0, st>>>((const float*)n->W0, (const float*)n->b0, (const float*)n->mask0,
                                                    n->P, n->H0, K0, im.idx0, meta, const_cast<unsigned char*>(im.W0img));
    tc::prep_w2_kernel<<<64, 256, 0, st>>>((const float*)n->W2, (const float*)n->mask1, n->P, n->H1, D, D <= 4 ? 4 : 8,
                                           im.idx1, meta, im.scale, const_cast<float*>(im.W2p));
    return cudaGetLastError();
}

// MLP dispatch: SIMT kernel (the tcgen05 kernel hooks in here for fp32 / H = 200)
template <class T, int GEO, bool TAN, int NJ, bool PSTD = false>
static cudaError_t launch_mlp_simt(const BnnMlpArgs<T>& a, cudaStream_t st) {
    constexpr int RPT = sizeof(T) == 4 ? 8 : 4;
    typedef MlpSmem<T, GEO, NJ, RPT, TAN, PSTD> SM;
    auto kern = bnn_mlp_simt_kernel<T, GEO, NJ, RPT, TAN, PSTD>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM::bytes);
    if (e != cudaSuccess) return e;
    const long long ntiles = (a.total + SM::NPART - 1) / SM::NPART;
    const int grid = (int)(ntiles < (long long)num_sms() ? ntiles : (long long)num_sms());
    kern<<<grid, 256, SM::bytes, st>>>(a);
    return cudaGetLastError();
}
template <int GEO, bool TAN>
static cudaError_t launch_mlp_tc(const BnnMlpArgs<float>& a, const tc::Images& im, cudaStream_t st) {
    typedef Geo<GEO> G;
    constexpr int K0P = G::DA + G::NU + 1 <= 8 ? 8 : 16, DP = G::D <= 4 ? 4 : 8;
    auto kern = tc::bnn_mlp_tc_kernel<GEO, TAN>;
    const int smem = tc::Cfg<K0P, DP>::TOTAL + tc::Cfg<K0P, DP>::ALIGN_PAD;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    const int S = (int)(a.total / a.net.P);                  // items per particle: (problem, alpha) pairs / problems
    const int tiles_p = (S + tc::TILE_M - 1) / tc::TILE_M;      // super-tiles per particle (TAN: 1 + T passes each)
    const long long ntiles = (long long)tiles_p * a.net.P;
    if (ntiles >= (1ll << 31)) return cudaErrorInvalidValue;
    const int grid = (int)(ntiles < (long long)num_sms() ? ntiles : (long long)num_sms());
    kern<<<grid, tc::THREADS, smem, st>>>(a, im, S, tiles_p);
    return cudaGetLastError();
}
template <class T, int GEO, bool TAN>
static cudaError_t launch_mlp(const BnnMlpArgs<T>& a, const tc::Images& im, cudaStream_t st) {
    const int H = a.net.H0 > a.net.H1 ? a.net.H0 : a.net.H1;
    if (a.net.eps_out) {                     // use_predicted_std: both output heads, CUDA-core kernel
        if (H <= 32) return launch_mlp_simt<T, GEO, TAN, 2, true>(a, st);
        if (H <= 208) return launch_mlp_simt<T, GEO, TAN, 13, true>(a, st);
        if (H <= 256) return launch_mlp_simt<T, GEO, TAN, 16, true>(a, st);
        return cudaErrorInvalidValue;
    }
    if (use_tensor_cores<T>(a.net.H0, a.net.H1)) {
        if constexpr (sizeof(T) == 4) return launch_mlp_tc<GEO, TAN>(a, im, st);
    }
    if (H <= 32) return launch_mlp_simt<T, GEO, TAN, 2>(a, st);
    if (H <= 208) return launch_mlp_simt<T, GEO, TAN, 13>(a, st);
    if (H <= 256) return launch_mlp_simt<T, GEO, TAN, 16>(a, st);
    return cudaErrorInvalidValue;
}


template <class T>
cudaError_t bnn_mlp_launch(int geo, bool tan, const BnnMlpArgs<T>& a, const tc::Images& im, cudaStream_t st) {
    switch (geo * 2 + (tan ? 1 : 0)) {
        case GEO_PENDULUM * 2: return launch_mlp<T, GEO_PENDULUM, false>(a, im, st);
        case GEO_PENDULUM * 2 + 1: return launch_mlp<T, GEO_PENDULUM, true>(a, im, st);
        case GEO_CARTPOLE * 2: return launch_mlp<T, GEO_CARTPOLE, false>(a, im, st);
        case GEO_CARTPOLE * 2 + 1: return launch_mlp<T, GEO_CARTPOLE, true>(a, im, st);
        case GEO_DOUBLE_CARTPOLE * 2: return launch_mlp<T, GEO_DOUBLE_CARTPOLE, false>(a, im, st);
        case GEO_DOUBLE_CARTPOLE * 2 + 1: return launch_mlp<T, GEO_DOUBLE_CARTPOLE, true>(a, im, st);
        case GEO_RENDEZVOUS * 2: return launch_mlp<T, GEO_RENDEZVOUS, false>(a, im, st);
        case GEO_RENDEZVOUS * 2 + 1: return launch_mlp<T, GEO_RENDEZVOUS, true>(a, im, st);
    }
    return cudaErrorInvalidValue;
}
template cudaError_t bnn_mlp_launch<float>(int, bool, const BnnMlpArgs<float>&, const tc::Images&, cudaStream_t);
template cudaError_t bnn_mlp_launch<double>(int, bool, const BnnMlpArgs<double>&, const tc::Images&, cudaStream_t);

}  // namespace pddp

#ifdef PDDP_EXP_TRACE
// (timeline experiment) copies CTA 0's trace of the last tcgen05 MLP launch to the host
extern "C" int pddp_debug_trace(long long* dst, size_t n) {
    cudaDeviceSynchronize();
    return (int)cudaMemcpyFromSymbol(dst, pddp::tc::g_trace, n * sizeof(long long));
}
#endif
