// MC-dropout MLP over particle rows on the CUDA cores (any dtype, any hidden width <= 256).
//
// This is the precision-reference implementation of the particle propagation
//   X'_p = X_p + dX_std * fc_out(relu(M1_p * fc_1(relu(M0_p * fc_0(norm([aug(X_p), u])))))) + dX_mean
// (ref: pddp/models/bnn/modules.py:200-264, 774-789; masks are [P,H], one row per particle,
// multiplied into the pre-activation BEFORE the ReLU) and, when TAN, of its Jacobian w.r.t.
// (X_p, u) by forward-mode tangents: each particle contributes 1 primal + (D+nu) tangent rows that
// share the primal's activation pattern (SURVEY.md appendix B).  fp64 always runs here; fp32 runs
// here unless the tcgen05 kernel (bnn_mlp_tc.cu) supports the shape.
//
// One CTA = 16x16 threads owns a tile of RT = 16*RPT rows and all H columns; the H0xH1 layer is a
// shared-memory-tiled FFMA GEMM (thread = RPT rows x NJ strided columns).
#pragma once
#include "bnn_mlp_iface.h"

namespace pddp {


constexpr int MLP_KC = 16;
constexpr int MLP_KP = 16;   // padded layer-0 input width (K0 = DA + nu <= 12)

// PSTD: use_predicted_std=True -- the log-std head of the output layer (rows D..2D-1 of fc_out) is evaluated
// too and exp(log_std) * eps_out[i] is added to every particle (ref: modules.py:242-262).
template <class T, int GEO, int NJ, int RPT, bool TAN, bool PSTD = false>
struct MlpSmem {
    typedef Geo<GEO> G;
    static constexpr int D = G::D, DO = PSTD ? 2 * D : D, K0 = G::DA + G::NU, TD = TAN ? D + G::NU : 0, RPP = 1 + TD;
    static constexpr int RT = 16 * RPT, NPART = RT / RPP, HP = NJ * 16, LDA = HP + 1;
    static_assert(DO <= MLP_KP, "the output rows reuse the layer-0 input staging");
    static constexpr size_t elems = (size_t)RT * LDA + (size_t)MLP_KC * HP + (TAN ? (size_t)NPART * HP : 0) +
                                    (size_t)RT * MLP_KP + (size_t)HP * DO + (size_t)NPART * D;
    static constexpr size_t bytes = elems * sizeof(T);
};

template <class T, int GEO, int NJ, int RPT, bool TAN, bool PSTD = false>
__global__ void __launch_bounds__(256) bnn_mlp_simt_kernel(const BnnMlpArgs<T> a) {
    typedef Geo<GEO> G;
    typedef MlpSmem<T, GEO, NJ, RPT, TAN, PSTD> SM;
    constexpr int DO = SM::DO;
    constexpr int D = SM::D, K0 = SM::K0, TD = SM::TD, RPP = SM::RPP, RT = SM::RT, NPART = SM::NPART;
    constexpr int HP = SM::HP, LDA = SM::LDA, DA = G::DA, NNA = G::NNA, NANG = G::NANG;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* A = reinterpret_cast<T*>(smem_raw);          // [RT][LDA] activations (layer in / out)
    T* Wc = A + (size_t)RT * LDA;                   // [KC][HP] chunk of W1T
    T* act = Wc + (size_t)MLP_KC * HP;              // [NPART][HP] primal (pre*mask), TAN only
    T* A0 = act + (TAN ? (size_t)NPART * HP : 0);   // [RT][MLP_KP] layer-0 inputs, later Y[RT][D]
    T* W2s = A0 + (size_t)RT * MLP_KP;              // [H1][DO]
    T* xs = W2s + (size_t)HP * DO;                  // [NPART][D]
    const BnnNet<T>& n = a.net;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int H0 = n.H0, H1 = n.H1, P = n.P;
    const long long ntiles = (a.total + NPART - 1) / NPART;

    for (int i = tid; i < H1 * DO; i += 256) W2s[i] = n.W2T[i];     // W2T is [H1][DO] (bnn.cu prep_weights)

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long g0 = tile * NPART;
        // ---- phase 0: inputs -------------------------------------------------------------
        for (int i = tid; i < RT * MLP_KP; i += 256) A0[i] = T(0);
        __syncthreads();
        if (tid < NPART && g0 + tid < a.total) {
            const long long g = g0 + tid;
            const T* u = a.u + (g / P) * G::NU;
            T x[D], in[K0], sc[K0];
#pragma unroll
            for (int d = 0; d < D; ++d) { x[d] = a.X[g * D + d]; xs[tid * D + d] = x[d]; }
#pragma unroll
            for (int k = 0; k < K0; ++k) sc[k] = n.X_std_inv ? n.X_std_inv[k] : T(1);
#pragma unroll
            for (int i = 0; i < NNA; ++i) in[i] = x[G::nonang(i)];
#pragma unroll
            for (int i = 0; i < NANG; ++i) { in[NNA + 2 * i] = jsin(x[G::ang(i)]); in[NNA + 2 * i + 1] = jcos(x[G::ang(i)]); }
#pragma unroll
            for (int j = 0; j < G::NU; ++j) in[DA + j] = u[j];
            T* r0 = A0 + (size_t)tid * RPP * MLP_KP;
#pragma unroll
            for (int k = 0; k < K0; ++k) r0[k] = (in[k] - (n.X_mean ? n.X_mean[k] : T(0))) * sc[k];
            if (TAN) {
#pragma unroll
                for (int i = 0; i < NNA; ++i) r0[(1 + G::nonang(i)) * MLP_KP + i] = sc[i];
#pragma unroll
                for (int i = 0; i < NANG; ++i) {
                    r0[(1 + G::ang(i)) * MLP_KP + NNA + 2 * i] = in[NNA + 2 * i + 1] * sc[NNA + 2 * i];        // d sin = cos
                    r0[(1 + G::ang(i)) * MLP_KP + NNA + 2 * i + 1] = -in[NNA + 2 * i] * sc[NNA + 2 * i + 1];   // d cos = -sin
                }
#pragma unroll
                for (int j = 0; j < G::NU; ++j) r0[(1 + D + j) * MLP_KP + DA + j] = sc[DA + j];
            }
        }
        __syncthreads();
        // ---- phase 1: layer 0 (K0 -> H0), primal rows first -------------------------------
        for (int idx = tid; idx < NPART * H0; idx += 256) {
            const int q = idx / H0, c = idx - q * H0;
            const long long g = g0 + q;
            T v = T(0);
            if (g < a.total) {
                T pre = n.b0[c];
                const T* r = A0 + (size_t)q * RPP * MLP_KP;
#pragma unroll
                for (int k = 0; k < K0; ++k) pre += r[k] * n.W0T[k * H0 + c];
                v = pre * n.mask0[(g % P) * H0 + c];
            }
            if (TAN) act[q * HP + c] = v;
            A[(size_t)(q * RPP) * LDA + c] = v > T(0) ? v : T(0);
        }
        if (TAN) {
            __syncthreads();
            for (int idx = tid; idx < NPART * TD * H0; idx += 256) {
                const int qd = idx / H0, c = idx - qd * H0;
                const int q = qd / TD, d = qd - q * TD;
                const long long g = g0 + q;
                T v = T(0);
                if (g < a.total && act[q * HP + c] > T(0)) {
                    const T* r = A0 + (size_t)(q * RPP + 1 + d) * MLP_KP;
                    T pre = T(0);
#pragma unroll
                    for (int k = 0; k < K0; ++k) pre += r[k] * n.W0T[k * H0 + c];
                    v = pre * n.mask0[(g % P) * H0 + c];
                }
                A[(size_t)(q * RPP + 1 + d) * LDA + c] = v;
            }
        }
        for (int idx = tid; idx < (RT - NPART * RPP) * LDA; idx += 256) A[(size_t)NPART * RPP * LDA + idx] = T(0);
        __syncthreads();
        // ---- phase 2: layer 1 (H0 -> H1) as a tiled GEMM ----------------------------------
        T acc[RPT][NJ];
#pragma unroll
        for (int i = 0; i < RPT; ++i)
#pragma unroll
            for (int j = 0; j < NJ; ++j) acc[i][j] = T(0);
        for (int k0 = 0; k0 < H0; k0 += MLP_KC) {
            for (int idx = tid; idx < MLP_KC * HP; idx += 256) {
                const int kc = idx / HP, c = idx - kc * HP;
                Wc[idx] = (k0 + kc < H0 && c < H1) ? n.W1T[(size_t)(k0 + kc) * H1 + c] : T(0);
            }
            __syncthreads();
            const int kmax = min(MLP_KC, H0 - k0);
            for (int kc = 0; kc < kmax; ++kc) {
                T av[RPT], wv[NJ];
#pragma unroll
                for (int i = 0; i < RPT; ++i) av[i] = A[(size_t)(ty * RPT + i) * LDA + k0 + kc];
#pragma unroll
                for (int j = 0; j < NJ; ++j) wv[j] = Wc[kc * HP + tx + 16 * j];
#pragma unroll
                for (int i = 0; i < RPT; ++i)
#pragma unroll
                    for (int j = 0; j < NJ; ++j) acc[i][j] += av[i] * wv[j];
            }
            __syncthreads();
        }
        // epilogue: bias + mask + relu; tangent rows follow their primal's activation pattern
        if (TAN) {
#pragma unroll
            for (int i = 0; i < RPT; ++i) {
                const int row = ty * RPT + i, q = row / RPP, d = row - q * RPP;
                if (q < NPART && d == 0 && g0 + q < a.total) {
                    const int p = (int)((g0 + q) % P);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const int c = tx + 16 * j;
                        if (c < H1) act[q * HP + c] = (acc[i][j] + n.b1[c]) * n.mask1[p * H1 + c];
                    }
                }
            }
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            const int row = ty * RPT + i, q = row / RPP, d = row - q * RPP;
            const bool live = q < NPART && g0 + q < a.total;
            const int p = live ? (int)((g0 + q) % P) : 0;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int c = tx + 16 * j;
                if (c >= H1) continue;
                T v = T(0);
                if (live) {
                    if (!TAN) {
                        v = (acc[i][j] + n.b1[c]) * n.mask1[p * H1 + c];
                        v = v > T(0) ? v : T(0);
                    } else if (d == 0) {
                        v = act[q * HP + c];
                        v = v > T(0) ? v : T(0);
                    } else {
                        v = act[q * HP + c] > T(0) ? acc[i][j] * n.mask1[p * H1 + c] : T(0);
                    }
                }
                A[(size_t)row * LDA + c] = v;
            }
        }
        __syncthreads();
        // ---- phase 3: output layer (H1 -> D), only the mean head is used --------------------
        T* Y = A0;
        for (int idx = tid; idx < RT * DO; idx += 256) {
            const int row = idx / DO, o = idx - row * DO;
            T s = T(0);
            const T* ar = A + (size_t)row * LDA;
            for (int k = 0; k < H1; ++k) s += ar[k] * W2s[k * DO + o];
            Y[idx] = s;
        }
        __syncthreads();
        // ---- phase 4: X' = X + dx, J = [I | 0] + d dx -------------------------------------
        if (tid < NPART && g0 + tid < a.total) {
            const long long g = g0 + tid;
            const int r0 = tid * RPP;
#pragma unroll
            for (int o = 0; o < D; ++o) {
                const T sd = n.dX_std ? n.dX_std[o] : T(1), mn = n.dX_mean ? n.dX_mean[o] : T(0);
                T dx = (Y[r0 * DO + o] + n.b2[o]) * sd + mn;
                T noise = T(0);                                  // exp(log_std) * eps_out[i][p]   ref: modules.py:254-262
                if (PSTD) {
                    noise = sd * jexp(Y[r0 * DO + D + o] + n.b2[D + o]) * n.eps_out[(g % P) * D + o];
                    dx += noise;
                    if (n.independent_noise) noise = T(0);       // exp(log_std) detached: no tangent through it
                }
                a.Xn[g * D + o] = xs[tid * D + o] + dx;
                if (TAN) {
#pragma unroll
                    for (int d = 0; d < TD; ++d) {
                        T j = (d == o ? T(1) : T(0)) + Y[(r0 + 1 + d) * DO + o] * sd;
                        if (PSTD) j += noise * Y[(r0 + 1 + d) * DO + D + o];
                        a.Jp[(g * D + o) * TD + d] = j;
                    }
                }
            }
        }
        __syncthreads();
    }
}

}  // namespace pddp
