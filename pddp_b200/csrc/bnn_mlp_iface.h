// Interface between bnn.cu (time loops, moment matching) and bnn_mlp.cu (the particle-MLP kernels: tcgen05 and
// CUDA-core), so that the two compile as separate translation units.
#pragma once
#include "../../include/pddp_b200.h"
#include "bnn_common.cuh"

namespace pddp {

template <class T>
struct BnnMlpArgs {
    BnnNet<T> net;
    const T* X;        // [S, P, D] particles in
    const T* u;        // [S, nu] action per particle group
    T* Xn;             // [S, P, D] particles out
    T* Jp;             // [S, P, D, D+nu] per-particle Jacobian (TAN only)
    long long total;   // S * P
};

// sizes of a BNN geometry for host code that dispatches on the runtime geometry id
struct GeoDims { int D, NU, DA; };
inline GeoDims geo_dims(int geo) {
    switch (geo) {
        case GEO_PENDULUM: return {Geo<GEO_PENDULUM>::D, Geo<GEO_PENDULUM>::NU, Geo<GEO_PENDULUM>::DA};
        case GEO_CARTPOLE: return {Geo<GEO_CARTPOLE>::D, Geo<GEO_CARTPOLE>::NU, Geo<GEO_CARTPOLE>::DA};
        case GEO_DOUBLE_CARTPOLE: return {Geo<GEO_DOUBLE_CARTPOLE>::D, Geo<GEO_DOUBLE_CARTPOLE>::NU, Geo<GEO_DOUBLE_CARTPOLE>::DA};
        default: return {Geo<GEO_RENDEZVOUS>::D, Geo<GEO_RENDEZVOUS>::NU, Geo<GEO_RENDEZVOUS>::DA};
    }
}

namespace tc {
// sizes of the tcgen05 kernel's global images (bnn_mlp_tc.cuh has the layouts)
constexpr int IMG_TILE_N = 208, IMG_META = 4;
constexpr size_t IMG_W1_PSTRIDE = (size_t)13 * 208 * 64;    // per-particle W1 image: MAX_NKB blocks of TILE_N x 64 B
constexpr size_t IMG_W0_PSTRIDE = (size_t)7 * 2 * 32 * 64;  // per-particle layer-0 image (K0P = 16 rows)
struct Images {
    const unsigned char* W1img;   // [P] per-particle images, W1_PSTRIDE apart
    const unsigned char* W0img;
    const float* W2p;
    const float* scale;        // [2]: power-of-two scale of the W1 image and its inverse
    const int* meta;           // [P][META]: K-blocks, accumulator columns, kept units of layer 0 / layer 1
    int* idx0;                 // [P][TILE_N] compaction lists (prep kernels only)
    int* idx1;
};
}  // namespace tc

int num_sms();
template <class T> bool use_tensor_cores(int H0, int H1);
// builds the tcgen05 images (compaction lists, W1 / W0 / output-weight images) from the network of this call
cudaError_t bnn_mlp_prep_images(int geo, const pddp_bnn* n, const tc::Images& im, cudaStream_t st);
// one launch of the particle MLP over a.total rows: tcgen05 kernel when it applies, CUDA-core kernel otherwise
template <class T> cudaError_t bnn_mlp_launch(int geo, bool tan, const BnnMlpArgs<T>& a, const tc::Images& im, cudaStream_t st);

}  // namespace pddp
