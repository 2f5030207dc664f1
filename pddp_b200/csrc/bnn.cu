// BNN (MC-dropout particle) dynamics: linearisation and line-search rollout.
//
// ref: pddp/models/bnn/modules.py:287-386 (BNNDynamicsModel.forward) + 200-264 (particle MLP),
//      pddp/utils/particles.py:136-149, pddp/utils/encoding.py (moment matching back to z),
//      pddp/controllers/ilqr.py:393-486 (forward), 677-723 (_control_law), 764-791 (cost).
//
// Time is sequential; every step is two launches over ALL problems:
//   (1) the particle MLP (bnn_mlp_*): rows = problems x particles x (1 + tangents)   [tensor roofline]
//   (2) a moment-matching kernel: mean / covariance / Cholesky of the new particles and -- in the
//       linearise pass -- their forward-mode tangents w.r.t. every encoded input, chained through
//       X_p = m + eps_p U with eps_p = (X_p - m) U^-1 held constant (SURVEY.md appendix B).
// Particles are carried from step to step in the workspace; eps_in[0] and the dropout masks are
// data supplied by the caller, so there is no RNG on this path.
#include "../../include/pddp_b200.h"
#include "bnn_common.cuh"
#include "bnn_mlp_iface.h"
#include "kernels.h"
#include "profile.h"
#include "rdv_cost.cuh"
#include <stdio.h>
#include <stdlib.h>

namespace pddp {

#define CK(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) return e__; } while (0)

// ------------------------------------------------------------------------------------------
// weight prep: torch [out,in] -> [in,out] copies in the workspace (coalesced over outputs)
// ------------------------------------------------------------------------------------------
template <class T>
__global__ void bnn_transpose_kernel(const T* W, int out, int in, int out_used, T* WT) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < in * out_used; i += gridDim.x * blockDim.x) {
        const int k = i / out_used, o = i - k * out_used;
        WT[i] = W[(size_t)o * in + k];
    }
}

// ------------------------------------------------------------------------------------------
// input particles of step t: X_p = m + eps_p U(z_t), one thread per (group s, particle p); eps == nullptr
// puts every particle on the mean (sample_input_distribution=False).  The encoded state of group s is
// row (s / zdiv, t) of z, its status word is status[s / sdiv].   ref: modules.py:320-358
// ------------------------------------------------------------------------------------------
template <class T, int GEO, int ENC>
__global__ void bnn_init_particles_kernel(const T* z, Layout lz, int t, int zdiv, int sdiv, long long S, int P,
                                          const T* eps, const int32_t* active, int active_skip_other,
                                          const int32_t* bw_status, T* X, int32_t* status) {
    constexpr int D = Geo<GEO>::D, NZ = enc_size(D, ENC);
    const long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (id >= S * P) return;
    const long long s = id / P;
    const int p = (int)(id - s * P);
    const int b = (int)(s / zdiv), sb = (int)(s / sdiv);
    if (active && (active_skip_other ? active[sb] != 1 : active[sb] == 0)) return;
    if (bw_status && bw_status[sb] != 0) return;
    T zz[NZ];
#pragma unroll
    for (int e = 0; e < NZ; ++e) zz[e] = z[lz.at(b, t, e)];
    T U[D][D];
    if (!load_factor<D, ENC, T>(zz, U) && status) atomicOr(&status[sb], 2);
#pragma unroll
    for (int c = 0; c < D; ++c) {
        T v = zz[c];
        if (eps) {
#pragma unroll
            for (int r = 0; r <= c; ++r) v += eps[p * D + r] * U[r][c];
        }
        X[id * D + c] = v;
    }
}

// ------------------------------------------------------------------------------------------
// linearise: moment matching + Jacobian of one step, a team of 1 or 2 warps per problem
// ------------------------------------------------------------------------------------------
// per-warp slots of the cross-warp reduction scratch: the sums are D means or D (D + 1) / 2 covariance entries
__host__ __device__ constexpr int moment_lin_red(int D) { return D * (D + 1) / 2 > 32 ? D * (D + 1) / 2 : 32; }
// shared-memory elements of ONE problem in bnn_moment_lin_kernel (arrays padded to 16 bytes)
template <int D, int NU, int WPP>
__host__ __device__ constexpr int moment_lin_smem_elems(int P) {
    return 2 * ((P * D + 3) & ~3) + ((P * (D + NU) * D + 3) & ~3) + (WPP > 1 ? WPP * moment_lin_red(D) : 0);
}

template <class T>
struct MomentLinArgs {
    int B, N, t, P;
    const T* X; const T* Xn; const T* Jp;       // [B,P,D], [B,P,D], [B,P,D,D+nu]
    const int32_t* active;
    T* Z; T* F_z; T* F_u; int32_t* status;
    Layout lZ, lFz, lFu;
};

// N consecutive elements with the widest vector access the alignment allows: 16 bytes when a row (N elements) is a
// multiple of 16 bytes, else 8 bytes (every array here starts 16-byte aligned and N is even), else scalar.
template <int N, class T>
__device__ __forceinline__ void load_row(const T* p, T* out) {
    constexpr int ROWB = N * (int)sizeof(T);
    if constexpr (ROWB % 16 == 0) {
#pragma unroll
        for (int i = 0; i < ROWB / 16; ++i) reinterpret_cast<float4*>(out)[i] = reinterpret_cast<const float4*>(p)[i];
    } else if constexpr (ROWB % 8 == 0) {
#pragma unroll
        for (int i = 0; i < ROWB / 8; ++i) reinterpret_cast<float2*>(out)[i] = reinterpret_cast<const float2*>(p)[i];
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) out[i] = p[i];
    }
}

// One problem = a TEAM of WPP warps (4 warps per CTA).  Phase 1, lanes = particles: eps = (X - m) U^-1, X' and the
// per-particle Jacobian [dX'/dX | dX'/du] staged in shared memory TRANSPOSED (row c = derivative w.r.t. input c, so
// one direction reads one contiguous row; nu control rows follow the D state rows), mean and covariance by warp shuffles (+ a shared-memory step across the
// team's warps).  Phase 2, lanes = (input direction j, 1 of SPLIT particle subsets): the tangent of every particle
// along j, its mean and its second moment with the centred particles, then the encode differential.
// For the sparse encodings (everything but FULL_COVARIANCE_MATRIX) a direction moves ONE component of the input
// particle: dX_p = s_p e_c with s_p = 1 (mean directions), eps_p[r] dU_rr/dz_j (factor directions) -- or it is the
// control direction -- so dX'_p is one scaled row of the staged Jacobian instead of a dense D x D product
// (the dense form added exact zeros: same values).  The rendezvous geometry (D = 8, nu = 4) has up to 76 directions
// (full covariance); it runs 4 warps per problem, and the directions loop when they outnumber the team's lanes.
template <class T, int GEO, int ENC, int WPP>
__global__ void __launch_bounds__(128, (sizeof(T) == 4 && WPP == 1 && Geo<GEO>::D <= 4) ? 8 : (sizeof(T) == 4 && Geo<GEO>::D <= 6 ? 4 : 1)) bnn_moment_lin_kernel(const MomentLinArgs<T> a) {
    typedef Geo<GEO> G;
    constexpr int D = G::D, NU = G::NU, NZ = enc_size(D, ENC), NT = D * (D + 1) / 2, TL = WPP * 32, PPB = 4 / WPP;
    constexpr int RED = moment_lin_red(D), NJAC = D * (D + NU);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = warp / WPP, wq = warp % WPP, tl = wq * 32 + lane;
    const int b = blockIdx.x * PPB + slot;
    if (b >= a.B) return;                                 // (the whole team leaves together)
    if (a.active && a.active[b] != 1) return;
    const int P = a.P, t = a.t;
    const int PD4 = (P * D + 3) & ~3, PG4 = (P * NJAC + 3) & ~3;
    T* sm = reinterpret_cast<T*>(smem_raw) + (size_t)slot * moment_lin_smem_elems<D, NU, WPP>(P);
    T *s_eps = sm, *s_xc = sm + PD4, *s_G = sm + 2 * PD4, *s_red = s_G + PG4;   // eps, X'-M', [dX'/dX | dX'/du]^T, scratch
    auto team_sync = [&]() {
        if constexpr (WPP == 1) __syncwarp();
        else asm volatile("bar.sync %0, %1;" ::"r"(1 + slot), "r"(TL) : "memory");
    };
    // sums of N <= RED per-lane values over the team
    auto team_sum = [&](auto& v) {
        constexpr int N = (int)(sizeof(v) / sizeof(v[0]));
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = warp_sum(v[i]);
        if constexpr (WPP > 1) {
            if (lane == 0) {
#pragma unroll
                for (int i = 0; i < N; ++i) s_red[wq * RED + i] = v[i];
            }
            team_sync();
#pragma unroll
            for (int i = 0; i < N; ++i) {
                T acc = s_red[i];
#pragma unroll
                for (int w2 = 1; w2 < WPP; ++w2) acc += s_red[w2 * RED + i];
                v[i] = acc;
            }
            team_sync();
        }
    };

    T z[NZ];
#pragma unroll
    for (int e = 0; e < NZ; ++e) z[e] = a.Z[a.lZ.at(b, t, e)];
    T U[D][D];
    bool ok = load_factor<D, ENC, T>(z, U);

    // particles: eps = (X - m) U^-1 ; stage X', J ; partial sums for the mean
    T msum[D];
#pragma unroll
    for (int d = 0; d < D; ++d) msum[d] = T(0);
    for (int p = tl; p < P; p += TL) {
        const size_t g = (size_t)b * P + p;
        alignas(16) T x[D], xn[D], jac[NJAC];
        T delta[D], eps[D];
        load_row<D, T>(a.X + g * D, x);
        load_row<D, T>(a.Xn + g * D, xn);
        load_row<NJAC, T>(a.Jp + g * NJAC, jac);
#pragma unroll
        for (int d = 0; d < D; ++d) delta[d] = x[d] - z[d];
        solve_right_upper<D, T>(U, delta, eps);
#pragma unroll
        for (int d = 0; d < D; ++d) {
            s_eps[p * D + d] = eps[d];
            s_xc[p * D + d] = xn[d];
            msum[d] += xn[d];
#pragma unroll
            for (int c = 0; c < D + NU; ++c) s_G[(p * (D + NU) + c) * D + d] = jac[d * (D + NU) + c];
        }
    }
    T M[D];
#pragma unroll
    for (int d = 0; d < D; ++d) M[d] = msum[d];
    team_sum(M);
#pragma unroll
    for (int d = 0; d < D; ++d) M[d] /= T(P);
    T csum[NT];
#pragma unroll
    for (int i = 0; i < NT; ++i) csum[i] = T(0);
    for (int p = tl; p < P; p += TL) {
        T xc[D];
#pragma unroll
        for (int d = 0; d < D; ++d) { xc[d] = s_xc[p * D + d] - M[d]; s_xc[p * D + d] = xc[d]; }
#pragma unroll
        for (int r = 0; r < D; ++r)
#pragma unroll
            for (int c = r; c < D; ++c) csum[tri<D>(r, c)] += xc[r] * xc[c];
    }
    team_sum(csum);
    T Cov[D][D];
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
        for (int c = r; c < D; ++c) {
            T v = csum[tri<D>(r, c)] / T(P - 1);    // ref: utils/particles.py:136-149
            Cov[r][c] = v;
            Cov[c][r] = v;
        }
    team_sync();
    T zn[NZ], Un[D][D];
    ok = encode_moments<D, ENC, T>(M, Cov, zn, Un) && ok;
#pragma unroll
    for (int e = 0; e < NZ; ++e)
        if ((e % TL) == tl) a.Z[a.lZ.at(b, t + 1, e)] = zn[e];
    if (tl == 0 && !ok && a.status) a.status[b] |= 2;

    // SPLIT lanes per input direction j in [z (NZ), u (NU)], each taking every SPLIT-th particle
    constexpr int NJ = NZ + NU;
    constexpr int SPLIT = NJ * 8 <= TL ? 8 : NJ * 4 <= TL ? 4 : (NJ * 2 <= TL ? 2 : 1), JPW = 32 / SPLIT, JPT = WPP * JPW;
    const int sub = lane % SPLIT;
    for (int j0 = 0; j0 < NJ; j0 += JPT) {
        const int jraw = j0 + wq * JPW + lane / SPLIT;
        const bool jvalid = jraw < NJ;
        if (SPLIT == 1 && !jvalid) continue;              // no shuffles below in that case
        const int j = jvalid ? jraw : NJ - 1;
        T dM[D], S2[D][D];
#pragma unroll
        for (int r = 0; r < D; ++r) {
            dM[r] = T(0);
#pragma unroll
            for (int c = 0; c < D; ++c) S2[r][c] = T(0);
        }
        if constexpr (ENC == ENC_FULL) {
            T dm[D], dUd[D][D], du = T(0);
#pragma unroll
            for (int d = 0; d < D; ++d) dm[d] = (j == d) ? T(1) : T(0);
#pragma unroll
            for (int r = 0; r < D; ++r)
#pragma unroll
                for (int c = 0; c < D; ++c) dUd[r][c] = T(0);
            const int ju = j >= NZ ? j - NZ : 0;      // control component of a control direction
            if (j >= NZ) du = T(1);
            else if (j >= D) {
                // symmetrised direction (E_ab + E_ba)/2 through the Cholesky differential
                T S[D][D];
                const int ja = (j - D) / D, jb = (j - D) - ja * D;
#pragma unroll
                for (int r = 0; r < D; ++r)
#pragma unroll
                    for (int c = 0; c < D; ++c)
                        S[r][c] = ((r == ja && c == jb) ? T(0.5) : T(0)) + ((r == jb && c == ja) ? T(0.5) : T(0));
                chol_upper_diff<D, T>(U, S, dUd);
            }
            for (int p = sub; p < P; p += SPLIT) {
                alignas(16) T eps[D], xc[D], g[D + 1][D];     // rows of dX'/dX, then the row of control ju
                T dx[D];
                load_row<D, T>(s_eps + p * D, eps);
                load_row<D, T>(s_xc + p * D, xc);
                if constexpr (NU == 1) {
                    load_row<(D + 1) * D, T>(s_G + p * (D + 1) * D, &g[0][0]);
                } else {
                    load_row<D * D, T>(s_G + p * (D + NU) * D, &g[0][0]);
                    load_row<D, T>(s_G + (p * (D + NU) + D + ju) * D, g[D]);
                }
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    T v = dm[c];
#pragma unroll
                    for (int r = 0; r <= c; ++r) v += eps[r] * dUd[r][c];
                    dx[c] = v;
                }
#pragma unroll
                for (int r = 0; r < D; ++r) {
                    T v = g[D][r] * du;
#pragma unroll
                    for (int c = 0; c < D; ++c) v += g[c][r] * dx[c];
                    dM[r] += v;
#pragma unroll
                    for (int c = 0; c < D; ++c) S2[r][c] += v * xc[c];
                }
            }
        } else {
            // row of the staged Jacobian this direction reads, the eps component that scales it (-1: none) and
            // the constant factor dU_rr/dz_j
            int row = j < D ? j : (j >= NZ ? D + j - NZ : D), er = -1;
            T wgt = T(1);
            if (j >= D && j < NZ) {
                if (ENC == ENC_UT) {
#pragma unroll
                    for (int r = 0; r < D; ++r)
#pragma unroll
                        for (int c = r; c < D; ++c) if (j - D == tri<D>(r, c)) { er = r; row = c; }
                } else {                                  // VAR: U = diag(sqrt(v)), dU_aa/dv_a = 1 / (2 U_aa); STD: U = diag(s)
                    er = row = j - D;
                    if (ENC == ENC_VAR) {
#pragma unroll
                        for (int r = 0; r < D; ++r) if (r == er) wgt = T(0.5) / U[r][r];
                    }
                }
            }
            for (int p = sub; p < P; p += SPLIT) {
                alignas(16) T xc[D], g[D];
                load_row<D, T>(s_G + (p * (D + NU) + row) * D, g);
                T sc = T(1);
                if (ENC != ENC_IGNORE && er >= 0) sc = s_eps[p * D + er] * wgt;
                if (ENC != ENC_IGNORE) load_row<D, T>(s_xc + p * D, xc);
#pragma unroll
                for (int r = 0; r < D; ++r) {
                    const T v = er >= 0 ? g[r] * sc : g[r];
                    dM[r] += v;
                    if (ENC != ENC_IGNORE) {
#pragma unroll
                        for (int c = 0; c < D; ++c) S2[r][c] += v * xc[c];
                    }
                }
            }
        }
        if (SPLIT > 1) {
#pragma unroll
            for (int off = 1; off < SPLIT; off <<= 1) {
#pragma unroll
                for (int r = 0; r < D; ++r) {
                    dM[r] += __shfl_xor_sync(0xffffffffu, dM[r], off);
                    if (ENC != ENC_IGNORE) {
#pragma unroll
                        for (int c = 0; c < D; ++c) S2[r][c] += __shfl_xor_sync(0xffffffffu, S2[r][c], off);
                    }
                }
            }
        }
        if (!jvalid || sub != 0) continue;
        T col[NZ];
#pragma unroll
        for (int r = 0; r < D; ++r) col[r] = dM[r] / T(P);
        if (ENC != ENC_IGNORE) {
            T dC[D][D];
#pragma unroll
            for (int r = 0; r < D; ++r)
#pragma unroll
                for (int c = 0; c < D; ++c) dC[r][c] = (S2[r][c] + S2[c][r]) / T(P - 1);
            if (ENC == ENC_FULL) {
#pragma unroll
                for (int r = 0; r < D; ++r)
#pragma unroll
                    for (int c = 0; c < D; ++c) col[D + r * D + c] = dC[r][c];
            } else if (ENC == ENC_VAR || ENC == ENC_STD) {      // var' = diag(C'), std' = sqrt(diag(C'))
#pragma unroll
                for (int r = 0; r < D; ++r) col[D + r] = ENC == ENC_VAR ? dC[r][r] : dC[r][r] / (T(2) * zn[D + r]);
            } else {
                T dUn[D][D];
                chol_upper_diff<D, T>(Un, dC, dUn);
#pragma unroll
                for (int r = 0; r < D; ++r)
#pragma unroll
                    for (int c = r; c < D; ++c) col[D + tri<D>(r, c)] = dUn[r][c];
            }
        }
        if (j < NZ) {
#pragma unroll
            for (int r = 0; r < NZ; ++r) a.F_z[a.lFz.at(b, t, r * NZ + j)] = col[r];
        } else {
#pragma unroll
            for (int r = 0; r < NZ; ++r) a.F_u[a.lFu.at(b, t, r * NU + (j - NZ))] = col[r];
        }
    }
}

// clamp the nominal controls of EVERY step into uall[t][b][nu] (the MLP of step t reads row t) and park them in the
// problem layout for the cost pass -- one launch instead of one per time step (they do not depend on the state)
template <class T>
__global__ void bnn_lin_control_kernel(int B, int N, int nu, const T* U, Layout lU, const T* u_min, const T* u_max,
                                       T* uall, T* U_clamped) {
    const long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (id >= (long long)B * N) return;
    const int t = (int)(id / B), b = (int)(id - (long long)t * B);
    for (int j = 0; j < nu; ++j) {
        T u = U[lU.at(b, t, j)];
        if (u_min && u_max) u = clampv(u, u_min[j], u_max[j]);
        uall[id * nu + j] = u;
        U_clamped[lU.at(b, t, j)] = u;
    }
}

// ------------------------------------------------------------------------------------------
// rollout: 8 or 4 lanes per (problem, alpha) pair, then one finishing thread per pair
// ------------------------------------------------------------------------------------------
template <class T>
struct RollStepArgs {
    int B, N, A, t, P;            // t = -1: initialise (z_0, u_0, J = l(z_0,u_0)); else transition t -> t+1
    CostParams<T> cost;
    const T* Xn;                  // [B*A, P, D] particles after the MLP of step t
    const T* Z; const T* U; const T* k; const T* K; const T* alphas; const T* u_min; const T* u_max;
    const int32_t* active; const int32_t* bw_status;
    T* Zall; T* Uall; T* ucur; T* J;          // [B*A, N+1, nz], [B*A, N, nu], [B*A, nu], [B*A]
    int32_t* status;
    Layout lZ, lU, lk, lK;
};

// CTA = 256 threads = 256 / LPP (problem, alpha) pairs.  The particles of the CTA's pairs are ONE contiguous block of
// the [pair][particle][D] array: a single cp.async.bulk stages it in shared memory while the threads that will finish
// the pairs already fetch their rows of the nominal trajectory and the gains (Z[t+1], K[t+1], k, U: ilqr.py:701-719).
// Phase A: LPP (8 or 4) lanes per pair reduce mean and covariance from shared memory (xor-shuffles); phase B: the
// first 256 / LPP threads, one per pair, do the encode (Cholesky), control law and moment-matched cost.  With nu > 1
// (rendezvous: K is 4 x nz, up to 288 values) the gains and the reference row are streamed inside the control law
// instead of being prefetched into registers, and the cost is the rendezvous QR cost on the un-augmented state.
// (History: one thread per pair issued 2 x P strided 4-byte loads per sector and ran at 9 % issue utilisation; 8 lanes
// per pair reading global memory directly spent the launch in 2 x P / LPP dependent round trips to L2: 28 us.)
// STAGE = false: the particles of 32 pairs do not fit shared memory (very large P): phase A reads them from global memory.
template <class T, int GEO, int ENC, int LPP, bool STAGE = true>
__global__ void __launch_bounds__(256) bnn_roll_step_kernel(const RollStepArgs<T> a) {
    typedef Geo<GEO> G;
    constexpr int D = G::D, NU = G::NU, NZ = enc_size(D, ENC), NT = D * (D + 1) / 2, PPC = 256 / LPP;
    constexpr int NZP = NU == 1 ? NZ : 1;                    // prefetched reference row and gains (nu == 1 only)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ T s_mom[PPC][D + NT];
    __shared__ __align__(8) uint64_t s_bar;
    T* s_X = reinterpret_cast<T*>(smem_raw);                 // [PPC][P][D]
    const int tid = threadIdx.x;
    const long long S = (long long)a.B * a.A;
    const int P = a.P, t1 = a.t + 1;
    const long long s0 = (long long)blockIdx.x * PPC;
    if (STAGE && a.t >= 0) {
        if (tid == 0) bulk_mbar_init(&s_bar, 1);
        __syncthreads();
        if (tid == 0) {
            const long long np = S - s0 < PPC ? S - s0 : PPC;
            const uint32_t bytes = (uint32_t)((np * P * D * sizeof(T) + 15) & ~15ull);   // (the workspace arrays are padded)
            bulk_load(s_X, a.Xn + (size_t)s0 * P * D, bytes, &s_bar);
        }
    }
    // the finishing thread of a pair: rows it needs, requested before anything waits
    const long long sB = s0 + tid;
    const bool fin = tid < PPC && sB < S;
    int b = 0, al = 0;
    bool run = false;
    T zref[NZP], Krow[NZP], kk[NU], uu[NU], alpha = T(0), Jprev = T(0);
#pragma unroll
    for (int i = 0; i < NU; ++i) kk[i] = uu[i] = T(0);
    if (fin) {
        b = (int)(sB / a.A); al = (int)(sB - (long long)b * a.A);
        run = !((a.active && a.active[b] == 0) || (a.bw_status && a.bw_status[b] != 0));
        if (run && t1 < a.N) {
            if constexpr (NU == 1) {
#pragma unroll
                for (int e = 0; e < NZ; ++e) { zref[e] = a.Z[a.lZ.at(b, t1, e)]; Krow[e] = a.K[a.lK.at(b, t1, e)]; }
            }
#pragma unroll
            for (int i = 0; i < NU; ++i) { kk[i] = a.k[a.lk.at(b, t1, i)]; uu[i] = a.U[a.lU.at(b, t1, i)]; }
            alpha = a.alphas[al];
        }
        if (run && a.t >= 0) Jprev = a.J[sB];
    }
    if (a.t >= 0) {
        if (STAGE) bulk_mbar_wait(&s_bar, 0);
        const int pr = tid / LPP, sub = tid % LPP;
        const bool live = s0 + pr < S;
        const T* X = STAGE ? s_X + (size_t)pr * P * D : a.Xn + (size_t)(live ? s0 + pr : 0) * P * D;
        T M[D];
#pragma unroll
        for (int d = 0; d < D; ++d) M[d] = T(0);
        if (live)
            for (int p = sub; p < P; p += LPP) {
                alignas(16) T x[D];
                load_row<D, T>(X + p * D, x);
#pragma unroll
                for (int d = 0; d < D; ++d) M[d] += x[d];
            }
#pragma unroll
        for (int d = 0; d < D; ++d) {
#pragma unroll
            for (int off = 1; off < LPP; off <<= 1) M[d] += __shfl_xor_sync(0xffffffffu, M[d], off);
            M[d] /= T(P);
        }
        T cs[NT];
#pragma unroll
        for (int i = 0; i < NT; ++i) cs[i] = T(0);
        if (live)
            for (int p = sub; p < P; p += LPP) {
                alignas(16) T x[D];
                T xc[D];
                load_row<D, T>(X + p * D, x);
#pragma unroll
                for (int d = 0; d < D; ++d) xc[d] = x[d] - M[d];
#pragma unroll
                for (int r = 0; r < D; ++r)
#pragma unroll
                    for (int c = r; c < D; ++c) cs[tri<D>(r, c)] += xc[r] * xc[c];
            }
#pragma unroll
        for (int i = 0; i < NT; ++i) {
#pragma unroll
            for (int off = 1; off < LPP; off <<= 1) cs[i] += __shfl_xor_sync(0xffffffffu, cs[i], off);
        }
        if (sub == 0) {
#pragma unroll
            for (int d = 0; d < D; ++d) s_mom[pr][d] = M[d];
#pragma unroll
            for (int i = 0; i < NT; ++i) s_mom[pr][D + i] = cs[i] / T(P - 1);     // ref: utils/particles.py:136-149
        }
    }
    __syncthreads();
    if (!fin || !run) return;
    const long long s = sB;
    T zn[NZ];
    bool ok = true;
    if (a.t < 0) {
#pragma unroll
        for (int e = 0; e < NZ; ++e) zn[e] = a.Z[a.lZ.at(b, 0, e)];
    } else {
        T M[D], Cov[D][D], Un[D][D];
#pragma unroll
        for (int d = 0; d < D; ++d) M[d] = s_mom[tid][d];
#pragma unroll
        for (int r = 0; r < D; ++r)
#pragma unroll
            for (int c = r; c < D; ++c) {
                Cov[r][c] = s_mom[tid][D + tri<D>(r, c)];
                Cov[c][r] = Cov[r][c];
            }
        ok = encode_moments<D, ENC, T>(M, Cov, zn, Un);
    }
    T* zrow = a.Zall + ((size_t)s * (a.N + 1) + t1) * NZ;
#pragma unroll
    for (int e = 0; e < NZ; ++e) zrow[e] = zn[e];
    if (!ok && a.status) atomicOr(&a.status[b], 2);
    T J = Jprev;
    if (t1 < a.N) {                                       // control law (ref: ilqr.py:701-719)
        T du[NU];
#pragma unroll
        for (int i = 0; i < NU; ++i) du[i] = alpha * kk[i];
        if constexpr (NU == 1) {
#pragma unroll
            for (int e = 0; e < NZ; ++e) du[0] += (zn[e] - zref[e]) * Krow[e];
        } else {
            const T* pK = a.K + a.lK.at(b, t1, 0);
            const int64_t seK = a.lK.se;
#pragma unroll 4
            for (int e = 0; e < NZ; ++e) {
                const T dz = zn[e] - a.Z[a.lZ.at(b, t1, e)];
#pragma unroll
                for (int i = 0; i < NU; ++i) du[i] += dz * pK[(i * NZ + e) * seK];
            }
        }
        T u[NU];
#pragma unroll
        for (int i = 0; i < NU; ++i) {
            u[i] = uu[i] + du[i];
            if (a.u_min && a.u_max) u[i] = clampv(u[i], a.u_min[i], a.u_max[i]);
            a.ucur[s * NU + i] = u[i];
            a.Uall[((size_t)s * a.N + t1) * NU + i] = u[i];
        }
        if constexpr (GEO == GEO_RENDEZVOUS) {
            J += rdv_cost_state<ENC, T>(a.cost, zn, false) + rdv_cost_action(a.cost, u);
        } else {
            T la, lu, luu;
            cost_action(a.cost, u[0], la, lu, luu);
            J += cost_state<GEO, ENC, T, T>(a.cost, zn, false) + la;
        }
    } else {
        if constexpr (GEO == GEO_RENDEZVOUS) J += rdv_cost_state<ENC, T>(a.cost, zn, true);
        else J += cost_state<GEO, ENC, T, T>(a.cost, zn, true);
    }
    a.J[s] = J;
}

// argmin over alphas (torch semantics) + copy of the winner, one warp per problem
template <class T>
__global__ void bnn_roll_select_kernel(int B, int N, int A, int nz, int nu, const T* J, const T* Zall, const T* Uall,
                                       const int32_t* active, const int32_t* bw_status, T* J_all,
                                       int32_t* amin, T* J_new, T* Z_new, T* U_new, Layout lZ, Layout lU) {
    const int lane = threadIdx.x & 31;
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B) return;
    if ((active && active[b] == 0) || (bw_status && bw_status[b] != 0)) return;
    int best = 0;
    T bj = J[(size_t)b * A];
    bool bn = bj != bj;
    for (int i = 1; i < A; ++i) {
        T v = J[(size_t)b * A + i];
        bool vn = v != v;
        if (!bn && (vn || v < bj)) { best = i; bj = v; bn = vn; }
    }
    for (int i = lane; i < A; i += 32) J_all[(size_t)b * A + i] = J[(size_t)b * A + i];
    if (lane == 0) { amin[b] = best; J_new[b] = bj; }
    const size_t s = (size_t)b * A + best;
    for (int i = lane; i < (N + 1) * nz; i += 32) Z_new[lZ.at(b, i / nz, i % nz)] = Zall[s * (N + 1) * nz + i];
    for (int i = lane; i < N * nu; i += 32) U_new[lU.at(b, i / nu, i % nu)] = Uall[s * N * nu + i];
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
template <class T>
struct Workspace {
    T *W0T, *W1T, *W2T, *m0T, *m1T, *Xa, *Xb, *Jp, *ucur, *J, *Zall, *Uall;
    tc::Images im;   // tcgen05 path: W1 image, per-particle layer-0 images and output weights
    size_t bytes;
};

template <class T>
static Workspace<T> carve(void* base, const pddp_shape* s, const pddp_bnn* n, int A) {
    const GeoDims gd = geo_dims(s->geo);
    const int D = gd.D, NU = gd.NU;
    const size_t K0 = gd.DA + NU, S = (size_t)s->B * (A > 1 ? A : 1), P = n->P;
    Workspace<T> w;
    size_t off = 0;
    auto take = [&](size_t elems) { T* p = reinterpret_cast<T*>(reinterpret_cast<char*>(base) + off); off += ((elems * sizeof(T) + 255) / 256) * 256; return p; };
    w.W0T = take(K0 * n->H0);
    w.W1T = take((size_t)n->H0 * n->H1);
    w.W2T = take((size_t)n->H1 * 2 * D);
    w.m0T = take((size_t)n->H0 * P);
    w.m1T = take((size_t)n->H1 * P);
    w.Xa = take(S * P * D);
    w.Xb = take(S * P * D);
    w.Jp = take((size_t)s->B * P * D * (D + NU));
    w.ucur = take(S * NU);
    w.J = take(S);
    w.Zall = take(S * (s->N + 1) * s->nz);
    w.Uall = take(S * s->N * NU);
    w.im.W1img = reinterpret_cast<unsigned char*>(take(P * tc::IMG_W1_PSTRIDE / sizeof(T)));        // per-particle (compacted) images
    w.im.W0img = reinterpret_cast<unsigned char*>(take(P * tc::IMG_W0_PSTRIDE / sizeof(T)));
    w.im.W2p = reinterpret_cast<float*>(take(P * (size_t)tc::IMG_TILE_N * 8 * sizeof(float) / sizeof(T)));
    w.im.scale = reinterpret_cast<float*>(take(256 / sizeof(T)));
    w.im.meta = reinterpret_cast<int*>(take(P * (size_t)tc::IMG_META * sizeof(int) / sizeof(T) + 1));
    w.im.idx0 = reinterpret_cast<int*>(take(P * (size_t)tc::IMG_TILE_N * sizeof(int) / sizeof(T)));
    w.im.idx1 = reinterpret_cast<int*>(take(P * (size_t)tc::IMG_TILE_N * sizeof(int) / sizeof(T)));
    w.bytes = off;
    return w;
}

template <class T>
static BnnNet<T> make_net(const pddp_bnn* n, const Workspace<T>& w) {
    BnnNet<T> r;
    r.P = n->P; r.H0 = n->H0; r.H1 = n->H1;
    r.W0T = w.W0T; r.b0 = (const T*)n->b0; r.W1T = w.W1T; r.b1 = (const T*)n->b1; r.W2T = w.W2T; r.b2 = (const T*)n->b2;
    r.mask0 = (const T*)n->mask0; r.mask1 = (const T*)n->mask1; r.eps0 = (const T*)n->eps0;
    r.mask0T = w.m0T; r.mask1T = w.m1T;
    r.X_mean = (const T*)n->X_mean; r.X_std_inv = (const T*)n->X_std_inv;
    r.dX_mean = (const T*)n->dX_mean; r.dX_std = (const T*)n->dX_std;
    r.eps_out = (const T*)n->eps_out;                 // step 0; the time loops advance it by P*D per step
    r.independent_noise = n->independent_noise;
    return r;
}

template <class T>
static cudaError_t prep_weights(const pddp_shape* s, const pddp_bnn* n, const Workspace<T>& w, cudaStream_t st) {
    const GeoDims gd = geo_dims(s->geo);
    const int D = gd.D;
    bnn_transpose_kernel<T><<<8, 256, 0, st>>>((const T*)n->W0, n->H0, gd.DA + gd.NU, n->H0, w.W0T);
    bnn_transpose_kernel<T><<<64, 256, 0, st>>>((const T*)n->W1, n->H1, n->H0, n->H1, w.W1T);
    bnn_transpose_kernel<T><<<8, 256, 0, st>>>((const T*)n->W2, 2 * D, n->H1, n->eps_out ? 2 * D : D, w.W2T);
    bnn_transpose_kernel<T><<<16, 256, 0, st>>>((const T*)n->mask0, n->P, n->H0, n->P, w.m0T);
    bnn_transpose_kernel<T><<<16, 256, 0, st>>>((const T*)n->mask1, n->P, n->H1, n->P, w.m1T);
    if (use_tensor_cores<T>(n->H0, n->H1)) CK(bnn_mlp_prep_images(s->geo, n, w.im, st));
    return cudaGetLastError();
}

struct BnnCall {
    const pddp_shape* s; const pddp_bnn* n; const pddp_cost* cost;
    const void *z0, *U, *u_min, *u_max; const int32_t* active;
    void *Z, *F_z, *F_u, *L, *L_z, *L_u, *L_zz, *L_uz, *L_uu, *J_opt; int32_t* status;
    void* ws; cudaStream_t st;
};

template <class T>
static void fill_cost_params(const pddp_cost* c, int DA, CostParams<T>& out) {
    memset(&out, 0, sizeof(out));
    for (int i = 0; i < DA * DA; ++i) { out.Q[i] = (T)c->Q[i]; out.Qt[i] = (T)c->Q_term[i]; }
    for (int i = 0; i < DA; ++i) out.xg[i] = (T)c->x_goal[i];
    for (int i = 0; i < MAX_NU * MAX_NU; ++i) out.R[i] = (T)c->R[i];
    for (int i = 0; i < MAX_NU; ++i) out.ug[i] = (T)c->u_goal[i];
}


template <class T>
__global__ void bnn_set_z0_kernel(int B, int nz, const T* z0, T* Z, Layout lZ, const int32_t* active) {
    const int id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= B * nz) return;
    const int b = id / nz, e = id - b * nz;
    if (active && active[b] != 1) return;
    Z[lZ.at(b, 0, e)] = z0[id];
}

template <class T, int GEO, int ENC>
static cudaError_t linearize_bnn_impl(const BnnCall& c) {
    typedef Geo<GEO> G;
    constexpr int D = G::D;
    const pddp_shape* s = c.s;
    const int B = s->B, N = s->N, nz = s->nz, nu = s->nu, ly = s->layout, P = c.n->P;
    Workspace<T> w = carve<T>(c.ws, s, c.n, 1);
    CK(prep_weights<T>(s, c.n, w, c.st));
    BnnNet<T> net = make_net<T>(c.n, w);
    const Layout lZ = make_layout(ly, B, N + 1, nz), lU = make_layout(ly, B, N, nu);
    T* Z = (T*)c.Z;
    bnn_set_z0_kernel<T><<<(B * nz + 255) / 256, 256, 0, c.st>>>(B, nz, (const T*)c.z0, Z, lZ, c.active);
    const long long total = (long long)B * P;
    // input particles (ref: modules.py:320-358): INFER carries them from step to step, RESAMPLE / MEAN rebuild
    // them from z_t at every step
    const int mode = c.n->input_mode;
    auto eps_of = [&](int t) -> const T* {
        return mode == PDDP_BNN_INPUT_MEAN ? nullptr
             : mode == PDDP_BNN_INPUT_RESAMPLE ? (const T*)c.n->eps_in + (size_t)t * P * D : net.eps0;
    };
    const unsigned igrid = (unsigned)((total + 127) / 128);
    bnn_init_particles_kernel<T, GEO, ENC><<<igrid, 128, 0, c.st>>>(Z, lZ, 0, 1, 1, B, P, eps_of(0), nullptr, 0,
                                                                    nullptr, w.Xa, c.status);
    CK(cudaGetLastError());

    MomentLinArgs<T> m;
    m.B = B; m.N = N; m.P = P; m.Jp = w.Jp; m.active = c.active; m.Z = Z; m.F_z = (T*)c.F_z; m.F_u = (T*)c.F_u;
    m.status = c.status; m.lZ = lZ; m.lFz = make_layout(ly, B, N, nz * nz); m.lFu = make_layout(ly, B, N, nz * nu);
    // warps per problem: two when there are more input directions than lanes (double cartpole, full covariance: 43);
    // four for the rendezvous encodings with more than 32 (UT: 48, full covariance: 76)
    constexpr int NJ = enc_size(D, ENC) + G::NU, WPP = NJ > 32 ? (GEO == GEO_RENDEZVOUS ? 4 : 2) : 1, ppb = 4 / WPP;
    const size_t msmem = (size_t)ppb * moment_lin_smem_elems<D, G::NU, WPP>(P) * sizeof(T);
    auto mk = bnn_moment_lin_kernel<T, GEO, ENC, WPP>;
    CK(cudaFuncSetAttribute(mk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem));

    BnnMlpArgs<T> a;
    a.net = net; a.Jp = w.Jp; a.total = total;
    T *cur = w.Xa, *nxt = w.Xb;
    // (w.Uall is [N, B, nu] in this pass: the all-alpha control buffer of the rollout pass, free here)
    bnn_lin_control_kernel<T><<<(unsigned)(((long long)B * N + 255) / 256), 256, 0, c.st>>>(
        B, N, nu, (const T*)c.U, lU, (const T*)c.u_min, (const T*)c.u_max, w.Uall, (T*)c.L_u);
    for (int t = 0; t < N; ++t) {
        a.u = w.Uall + (size_t)t * B * nu;
        if (mode != PDDP_BNN_INPUT_INFER && t > 0)
            bnn_init_particles_kernel<T, GEO, ENC><<<igrid, 128, 0, c.st>>>(Z, lZ, t, 1, 1, B, P, eps_of(t), c.active, 1,
                                                                            nullptr, cur, c.status);
        a.X = cur; a.Xn = nxt;
        if (net.eps_out) a.net.eps_out = net.eps_out + (size_t)t * P * D;
        prof_begin(PROF_MLP_LIN, c.st);
        CK(bnn_mlp_launch<T>(GEO, true, a, w.im, c.st));
        prof_end(PROF_MLP_LIN, c.st);
        m.t = t; m.X = cur; m.Xn = nxt;
        prof_begin(PROF_MOMENT_LIN, c.st);
        mk<<<(B + ppb - 1) / ppb, 128, msmem, c.st>>>(m);
        prof_end(PROF_MOMENT_LIN, c.st);
        T* tmp = cur; cur = nxt; nxt = tmp;
    }
    CK(cudaGetLastError());
    // cost value / gradient / Hessian over the whole nominal trajectory (clamped u parked in L_u)
    CostDerivArgs<T> cd;
    cd.B = B; cd.N = N;
    fill_cost_params<T>(c.cost, G::DA, cd.cost);
    cd.Z = Z; cd.U = (const T*)c.L_u; cd.active = c.active;
    cd.L = (T*)c.L; cd.L_z = (T*)c.L_z; cd.L_u = (T*)c.L_u; cd.L_zz = (T*)c.L_zz; cd.L_uz = (T*)c.L_uz;
    cd.L_uu = (T*)c.L_uu; cd.J_opt = (T*)c.J_opt;
    cd.lZ = lZ; cd.lU = lU; cd.lL = make_layout(ly, B, N + 1, 1); cd.lLz = make_layout(ly, B, N + 1, nz);
    cd.lLu = make_layout(ly, B, N, nu); cd.lLzz = make_layout(ly, B, N + 1, nz * nz);
    cd.lLuz = make_layout(ly, B, N, nu * nz); cd.lLuu = make_layout(ly, B, N, nu * nu);
    note_launches((use_tensor_cores<T>(c.n->H0, c.n->H1) ? 10 : 5) + 3 + 2LL * N + 2
                  + (s->enc == PDDP_ENC_FULL_COVARIANCE_MATRIX && GEO != GEO_RENDEZVOUS ? 1 : 0)
                  + (mode != PDDP_BNN_INPUT_INFER ? N - 1 : 0));
    prof_begin(PROF_COST, c.st);
    // rendezvous: the closed-form QR cost on the un-augmented state (the known-dynamics path's cost kernel)
    cudaError_t ce = GEO == GEO_RENDEZVOUS ? cost_derivatives_lq<T>(s->enc, cd, c.st)
                                           : cost_derivatives<T>(s->geo, s->enc, cd, c.st);
    prof_end(PROF_COST, c.st);
    return ce;
}

struct BnnRollCall {
    const pddp_shape* s; const pddp_bnn* n; const pddp_cost* cost;
    const void *Z, *U, *k, *K, *alphas; int A; const void *u_min, *u_max;
    const int32_t *active, *bw_status;
    void* J_all; int32_t* amin; void *J_new, *Z_new, *U_new; int32_t* status;
    void* ws; cudaStream_t st;
};

template <class T, int GEO, int ENC>
static cudaError_t rollout_bnn_impl(const BnnRollCall& c) {
    typedef Geo<GEO> G;
    const pddp_shape* s = c.s;
    const int B = s->B, N = s->N, nz = s->nz, nu = s->nu, ly = s->layout, P = c.n->P, A = c.A;
    Workspace<T> w = carve<T>(c.ws, s, c.n, A);
    CK(prep_weights<T>(s, c.n, w, c.st));
    BnnNet<T> net = make_net<T>(c.n, w);
    const long long S = (long long)B * A, total = S * P;
    RollStepArgs<T> r;
    r.B = B; r.N = N; r.A = A; r.P = P;
    fill_cost_params<T>(c.cost, G::DA, r.cost);
    r.Z = (const T*)c.Z; r.U = (const T*)c.U; r.k = (const T*)c.k; r.K = (const T*)c.K; r.alphas = (const T*)c.alphas;
    r.u_min = (const T*)c.u_min; r.u_max = (const T*)c.u_max; r.active = c.active; r.bw_status = c.bw_status;
    r.Zall = w.Zall; r.Uall = w.Uall; r.ucur = w.ucur; r.J = w.J; r.status = c.status;
    r.lZ = make_layout(ly, B, N + 1, nz); r.lU = make_layout(ly, B, N, nu);
    r.lk = make_layout(ly, B, N, nu); r.lK = make_layout(ly, B, N, nu * nz);
    constexpr int D = G::D;
    const int mode = c.n->input_mode;
    auto eps_of = [&](int t) -> const T* {
        return mode == PDDP_BNN_INPUT_MEAN ? nullptr
             : mode == PDDP_BNN_INPUT_RESAMPLE ? (const T*)c.n->eps_in + (size_t)t * P * D : net.eps0;
    };
    const unsigned igrid = (unsigned)((total + 127) / 128);
    const Layout lZall = make_layout(PDDP_PROBLEM_MAJOR, (int)S, N + 1, nz);
    bnn_init_particles_kernel<T, GEO, ENC><<<igrid, 128, 0, c.st>>>(r.Z, r.lZ, 0, A, A, S, P, eps_of(0), nullptr, 0,
                                                                    nullptr, w.Xa, c.status);
    // 8 lanes per (problem, alpha) pair while that grid fits the SMs in one wave, else 4 (cfg 2: 1 280 CTAs were 1.7 waves)
    const size_t pair_bytes = (size_t)P * D * sizeof(T);
    const bool lpp4 = (S + 31) / 32 > (long long)num_sms() * 4 && 64 * pair_bytes <= 100 * 1024;
    const unsigned rgrid = (unsigned)(lpp4 ? (S + 63) / 64 : (S + 31) / 32);
    const bool stage = 32 * pair_bytes + 16 <= 200 * 1024;       // else: particles straight from global memory
    const size_t rsmem = stage ? (lpp4 ? 64 : 32) * pair_bytes + 16 : 0;
    auto roll_step = !stage ? bnn_roll_step_kernel<T, GEO, ENC, 8, false>
                   : lpp4 ? bnn_roll_step_kernel<T, GEO, ENC, 4> : bnn_roll_step_kernel<T, GEO, ENC, 8>;
    CK(cudaFuncSetAttribute(roll_step, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsmem));
    r.t = -1; r.Xn = w.Xa;
    roll_step<<<rgrid, 256, rsmem, c.st>>>(r);
    CK(cudaGetLastError());
    BnnMlpArgs<T> a;
    a.net = net; a.u = w.ucur; a.Jp = nullptr; a.total = total;
    T *cur = w.Xa, *nxt = w.Xb;
    for (int t = 0; t < N; ++t) {
        a.X = cur; a.Xn = nxt;
        if (net.eps_out) a.net.eps_out = net.eps_out + (size_t)t * P * D;
        prof_begin(PROF_MLP_ROLL, c.st);
        CK(bnn_mlp_launch<T>(GEO, false, a, w.im, c.st));
        prof_end(PROF_MLP_ROLL, c.st);
        r.t = t; r.Xn = nxt;
        prof_begin(PROF_ROLL_STEP, c.st);
        roll_step<<<rgrid, 256, rsmem, c.st>>>(r);
        prof_end(PROF_ROLL_STEP, c.st);
        if (mode != PDDP_BNN_INPUT_INFER && t + 1 < N)      // candidate particles of step t+1 from the z' just encoded
            bnn_init_particles_kernel<T, GEO, ENC><<<igrid, 128, 0, c.st>>>(w.Zall, lZall, t + 1, 1, A, S, P, eps_of(t + 1),
                                                                            c.active, 0, c.bw_status, nxt, c.status);
        T* tmp = cur; cur = nxt; nxt = tmp;
    }
    bnn_roll_select_kernel<T><<<(unsigned)(((long long)B * 32 + 127) / 128), 128, 0, c.st>>>(
        B, N, A, nz, nu, w.J, w.Zall, w.Uall, c.active, c.bw_status, (T*)c.J_all, c.amin, (T*)c.J_new, (T*)c.Z_new,
        (T*)c.U_new, r.lZ, r.lU);
    note_launches((use_tensor_cores<T>(c.n->H0, c.n->H1) ? 10 : 5) + 2 + 2LL * N + 1 + (mode != PDDP_BNN_INPUT_INFER ? N - 1 : 0));
    return cudaGetLastError();
}

#define BNN_DISPATCH(IMPL, call)                                                                          \
    switch (call.s->geo * 8 + call.s->enc) {                                                              \
        case GEO_PENDULUM * 8 + ENC_FULL: return IMPL<T, GEO_PENDULUM, ENC_FULL>(call);                   \
        case GEO_PENDULUM * 8 + ENC_UT: return IMPL<T, GEO_PENDULUM, ENC_UT>(call);                       \
        case GEO_PENDULUM * 8 + ENC_IGNORE: return IMPL<T, GEO_PENDULUM, ENC_IGNORE>(call);               \
        case GEO_PENDULUM * 8 + ENC_VAR: return IMPL<T, GEO_PENDULUM, ENC_VAR>(call);                     \
        case GEO_PENDULUM * 8 + ENC_STD: return IMPL<T, GEO_PENDULUM, ENC_STD>(call);                     \
        case GEO_CARTPOLE * 8 + ENC_VAR: return IMPL<T, GEO_CARTPOLE, ENC_VAR>(call);                     \
        case GEO_CARTPOLE * 8 + ENC_STD: return IMPL<T, GEO_CARTPOLE, ENC_STD>(call);                     \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_VAR: return IMPL<T, GEO_DOUBLE_CARTPOLE, ENC_VAR>(call);       \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_STD: return IMPL<T, GEO_DOUBLE_CARTPOLE, ENC_STD>(call);       \
        case GEO_CARTPOLE * 8 + ENC_FULL: return IMPL<T, GEO_CARTPOLE, ENC_FULL>(call);                   \
        case GEO_CARTPOLE * 8 + ENC_UT: return IMPL<T, GEO_CARTPOLE, ENC_UT>(call);                       \
        case GEO_CARTPOLE * 8 + ENC_IGNORE: return IMPL<T, GEO_CARTPOLE, ENC_IGNORE>(call);               \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_FULL: return IMPL<T, GEO_DOUBLE_CARTPOLE, ENC_FULL>(call);     \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_UT: return IMPL<T, GEO_DOUBLE_CARTPOLE, ENC_UT>(call);         \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_IGNORE: return IMPL<T, GEO_DOUBLE_CARTPOLE, ENC_IGNORE>(call); \
        case GEO_RENDEZVOUS * 8 + ENC_FULL: return IMPL<T, GEO_RENDEZVOUS, ENC_FULL>(call);               \
        case GEO_RENDEZVOUS * 8 + ENC_UT: return IMPL<T, GEO_RENDEZVOUS, ENC_UT>(call);                   \
        case GEO_RENDEZVOUS * 8 + ENC_VAR: return IMPL<T, GEO_RENDEZVOUS, ENC_VAR>(call);                 \
        case GEO_RENDEZVOUS * 8 + ENC_STD: return IMPL<T, GEO_RENDEZVOUS, ENC_STD>(call);                 \
        case GEO_RENDEZVOUS * 8 + ENC_IGNORE: return IMPL<T, GEO_RENDEZVOUS, ENC_IGNORE>(call);           \
        default: return cudaErrorInvalidValue;                                                            \
    }

template <class T> static cudaError_t linearize_bnn_t(const BnnCall& c) { BNN_DISPATCH(linearize_bnn_impl, c) }
template <class T> static cudaError_t rollout_bnn_t(const BnnRollCall& c) { BNN_DISPATCH(rollout_bnn_impl, c) }

}  // namespace pddp

using namespace pddp;

int pddp_capi_fail(int code, const char* msg);          // capi.cu
int pddp_capi_cuda(cudaError_t e, const char* what);    // capi.cu
int pddp_capi_check_shape(const pddp_shape* s);         // capi.cu

static int check_bnn(const pddp_shape* s, const pddp_bnn* n) {
    if (int e = pddp_capi_check_shape(s)) return e;
    if (s->layout != PDDP_PROBLEM_MAJOR) return pddp_capi_fail(PDDP_E_UNSUPPORTED, "BNN path uses PDDP_PROBLEM_MAJOR");
    if (s->geo > GEO_RENDEZVOUS) return pddp_capi_fail(PDDP_E_UNSUPPORTED, "BNN kernels exist for the pendulum, cartpole, double-cartpole and rendezvous geometries");
    if (!n) return pddp_capi_fail(PDDP_E_BADARG, "bnn is NULL");
    if (n->P < 2 || n->P > 1024) return pddp_capi_fail(PDDP_E_BADARG, "2 <= particles <= 1024");
    if (n->H0 < 1 || n->H1 < 1 || n->H0 > 256 || n->H1 > 256) return pddp_capi_fail(PDDP_E_UNSUPPORTED, "hidden widths must be in [1,256]");
    if (!n->W0 || !n->b0 || !n->W1 || !n->b1 || !n->W2 || !n->b2 || !n->mask0 || !n->mask1 || !n->eps0)
        return pddp_capi_fail(PDDP_E_BADARG, "bnn: NULL weight / mask / eps0 pointer");
    if (n->input_mode < PDDP_BNN_INPUT_INFER || n->input_mode > PDDP_BNN_INPUT_MEAN)
        return pddp_capi_fail(PDDP_E_BADARG, "bnn: input_mode must be PDDP_BNN_INPUT_INFER / RESAMPLE / MEAN");
    if (n->input_mode == PDDP_BNN_INPUT_RESAMPLE && !n->eps_in)
        return pddp_capi_fail(PDDP_E_BADARG, "bnn: PDDP_BNN_INPUT_RESAMPLE needs eps_in[N,P,D]");
    return 0;
}

extern "C" int64_t pddp_bnn_workspace_bytes(const pddp_shape* s, const pddp_bnn* n, int32_t A) {
    if (int e = check_bnn(s, n)) return e;
    if (A < 1 || A > 64) return pddp_capi_fail(PDDP_E_BADARG, "1 <= A <= 64");
    if (s->dtype == PDDP_F32) return (int64_t)carve<float>(nullptr, s, n, A).bytes;
    return (int64_t)carve<double>(nullptr, s, n, A).bytes;
}

extern "C" int pddp_linearize_bnn(const pddp_shape* s, const pddp_bnn* n, const pddp_cost* cost, const void* z0,
                                  const void* U, const void* u_min, const void* u_max, const int32_t* active,
                                  void* Z, void* F_z, void* F_u, void* L, void* L_z, void* L_u, void* L_zz,
                                  void* L_uz, void* L_uu, void* J_opt, int32_t* status, void* workspace,
                                  int64_t workspace_bytes, void* stream) {
    if (int e = check_bnn(s, n)) return e;
    if (!cost || !z0 || !U || !Z || !F_z || !F_u || !L || !L_z || !L_u || !L_zz || !L_uz || !L_uu || !J_opt || !workspace)
        return pddp_capi_fail(PDDP_E_BADARG, "pddp_linearize_bnn: NULL argument");
    if ((u_min == nullptr) != (u_max == nullptr)) return pddp_capi_fail(PDDP_E_BADARG, "u_min and u_max must be given together");
    if (workspace_bytes < pddp_bnn_workspace_bytes(s, n, 1)) return pddp_capi_fail(PDDP_E_BADARG, "workspace too small");
    BnnCall c{s, n, cost, z0, U, u_min, u_max, active, Z, F_z, F_u, L, L_z, L_u, L_zz, L_uz, L_uu, J_opt, status,
              workspace, (cudaStream_t)stream};
    cudaError_t e = s->dtype == PDDP_F32 ? linearize_bnn_t<float>(c) : linearize_bnn_t<double>(c);
    return pddp_capi_cuda(e, "pddp_linearize_bnn");
}

extern "C" int pddp_rollout_bnn(const pddp_shape* s, const pddp_bnn* n, const pddp_cost* cost, const void* Z,
                                const void* U, const void* k, const void* K, const void* alphas, int32_t A,
                                const void* u_min, const void* u_max, const int32_t* active,
                                const int32_t* bw_status, void* J_all, int32_t* amin, void* J_new, void* Z_new,
                                void* U_new, int32_t* status, void* workspace, int64_t workspace_bytes,
                                void* stream) {
    if (int e = check_bnn(s, n)) return e;
    if (!cost || !Z || !U || !k || !K || !alphas || !J_all || !amin || !J_new || !Z_new || !U_new || !workspace)
        return pddp_capi_fail(PDDP_E_BADARG, "pddp_rollout_bnn: NULL argument");
    if (A < 1 || A > 64) return pddp_capi_fail(PDDP_E_BADARG, "1 <= A <= 64");
    if ((u_min == nullptr) != (u_max == nullptr)) return pddp_capi_fail(PDDP_E_BADARG, "u_min and u_max must be given together");
    if (workspace_bytes < pddp_bnn_workspace_bytes(s, n, A)) return pddp_capi_fail(PDDP_E_BADARG, "workspace too small");
    BnnRollCall c{s, n, cost, Z, U, k, K, alphas, A, u_min, u_max, active, bw_status, J_all, amin, J_new, Z_new, U_new,
                  status, workspace, (cudaStream_t)stream};
    cudaError_t e = s->dtype == PDDP_F32 ? rollout_bnn_t<float>(c) : rollout_bnn_t<double>(c);
    return pddp_capi_cuda(e, "pddp_rollout_bnn");
}

