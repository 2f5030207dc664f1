// Known-dynamics path of the multi-vehicle rendezvous problem (D = 8, action_size = 4, no angles):
// linearisation and line-search rollout.
//
// ref: pddp/examples/rendezvous/model.py:79-115 (two point masses with friction; the WHOLE covariance
//      is passed through unchanged, `encode(mean, C=covar)`), pddp/examples/rendezvous/cost.py:29-43 +
//      pddp/costs/quadratic.py:60-99 (plain QRCost on the un-augmented state),
//      pddp/controllers/ilqr.py:393-486 (forward), 677-723 (_control_law), 764-791 (_trajectory_cost).
//
// The problem is linear-quadratic, so nothing is differentiated numerically or by jets: the mean rows of
// F_z / F_u are the constant A / B of the model, the cost Hessian is Q + Q^T on the mean block and, for the
// trace term sum(C o Q^T), constant in whatever parametrises C (zero for FULL / VARIANCE, (Q+Q^T)_ab
// between U_ka and U_kb for UT-Cholesky, 2 Q_aa for STANDARD_DEVIATION).  The only non-trivial derivative
// is the UT-Cholesky pass-through U' = chol(U^T U + 1e-12 I), linearised with the Cholesky differential.
// Mapping: one thread per problem (linearise, winner store) or per (problem, alpha) pair (line search);
// the encoded state (nz <= 72) lives in a per-thread array.
#include "bnn_common.cuh"
#include "kernels.h"
#include "rdv_cost.cuh"

namespace pddp {

namespace {

constexpr int RD = RDV_D, RNU = RDV_NU;

template <class T>
struct RdvModel { T dt, fr, gu, dvv, dvu; };   // acc = vel * fr + u * gu ; d vel'/d vel = dvv, d vel'/d u = dvu

template <class T>
__device__ __forceinline__ RdvModel<T> rdv_model(const KnownParams<T>& kp) {
    // ref: rendezvous/model.py:104-115: acc = v (1 - alpha dt / m) + u dt / m ; v' = v + acc dt
    const T dt = kp.p[0], m = kp.p[1], al = kp.p[2];
    RdvModel<T> r;
    r.dt = dt;
    r.fr = T(1) - al * dt / m;
    r.gu = dt / m;
    r.dvv = T(1) + r.fr * dt;
    r.dvu = r.gu * dt;
    return r;
}

template <class T>
__device__ __forceinline__ void rdv_mean_step(const RdvModel<T>& md, const T* x, const T* u, T* xn) {
    const T dt = md.dt;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        xn[i] = x[i] + x[4 + i] * dt;
        xn[4 + i] = x[4 + i] + (x[4 + i] * md.fr + u[i] * md.gu) * dt;   // same association as the reference
    }
}

// uncertainty part of z' (the covariance itself is unchanged; only its parametrisation is re-encoded)
template <int ENC, class T>
__device__ __forceinline__ bool rdv_uncertainty_step(const T* z, T* zn, T (&U)[RD][RD], T (&Un)[RD][RD]) {
    constexpr int D = RD;
    if (ENC == ENC_FULL) {
#pragma unroll 1
        for (int e = 0; e < D * D; ++e) zn[D + e] = z[D + e];
    } else if (ENC == ENC_VAR) {
#pragma unroll
        for (int a = 0; a < D; ++a) zn[D + a] = z[D + a];
    } else if (ENC == ENC_STD) {
#pragma unroll
        for (int a = 0; a < D; ++a) zn[D + a] = jsqrt(z[D + a] * z[D + a]);
    } else if (ENC == ENC_UT) {
        T C[D][D];
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = 0; b < D; ++b) U[a][b] = b >= a ? z[D + tri<D>(a, b)] : T(0);
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = a; b < D; ++b) {
                T s = T(0);
#pragma unroll
                for (int k = 0; k <= a; ++k) s += U[k][a] * U[k][b];
                C[a][b] = s;
                C[b][a] = s;
            }
        const bool ok = chol_upper_jitter<D, T>(C, Un);          // ref: utils/encoding.py:536-564
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = a; b < D; ++b) zn[D + tri<D>(a, b)] = Un[a][b];
        return ok;
    }
    return true;
}

// ------------------------------------------------------------------------------------------
// cost value / gradient / Hessian of one (problem, time) site in closed form; Args = LinKnownArgs or
// CostDerivArgs (same member names), goal = problem b's goal.  Replaces batch_eval_cost (utils/evaluation.py:134-239).
// ------------------------------------------------------------------------------------------
template <class T, int ENC, class Args>
__device__ __forceinline__ T lq_cost_site(const Args& a, const Goal<T, RD, RNU>& goal, int b, int t, const T* z, const T* u,
                                          bool terminal) {
    constexpr int D = RD, NU = RNU, NZ = enc_size(D, ENC);
    const T* Q = terminal ? a.cost.Qt : a.cost.Q;
    T l = rdv_cost_state<ENC, T>(a.cost, goal.x, z, terminal);
    for (int e = 0; e < NZ * NZ; ++e) a.L_zz[a.lLzz.at(b, t, e)] = T(0);
    for (int i = 0; i < D; ++i) {
        T g = T(0);
        for (int j = 0; j < D; ++j) {
            g += (Q[i * D + j] + Q[j * D + i]) * (z[j] - goal.x[j]);
            a.L_zz[a.lLzz.at(b, t, i * NZ + j)] = Q[i * D + j] + Q[j * D + i];
        }
        a.L_z[a.lLz.at(b, t, i)] = g;
    }
    if (ENC == ENC_FULL) {
        for (int i = 0; i < D; ++i)
            for (int j = 0; j < D; ++j) a.L_z[a.lLz.at(b, t, D + i * D + j)] = Q[j * D + i];
    } else if (ENC == ENC_UT) {
        for (int k = 0; k < D; ++k)
            for (int c = k; c < D; ++c) {
                T g = T(0);
                for (int j = k; j < D; ++j) g += z[D + tri<D>(k, j)] * (Q[j * D + c] + Q[c * D + j]);
                const int r = D + tri<D>(k, c);
                a.L_z[a.lLz.at(b, t, r)] = g;
                for (int c2 = k; c2 < D; ++c2)
                    a.L_zz[a.lLzz.at(b, t, r * NZ + D + tri<D>(k, c2))] = Q[c * D + c2] + Q[c2 * D + c];
            }
    } else if (ENC == ENC_VAR) {
        for (int c = 0; c < D; ++c) a.L_z[a.lLz.at(b, t, D + c)] = Q[c * D + c];
    } else if (ENC == ENC_STD) {
        for (int c = 0; c < D; ++c) {
            a.L_z[a.lLz.at(b, t, D + c)] = T(2) * z[D + c] * Q[c * D + c];
            a.L_zz[a.lLzz.at(b, t, (D + c) * NZ + D + c)] = T(2) * Q[c * D + c];
        }
    }
    if (!terminal) {
        l += rdv_cost_action(a.cost, goal.u, u);
#pragma unroll
        for (int i = 0; i < NU; ++i) {
            T g = T(0);
#pragma unroll
            for (int j = 0; j < NU; ++j) {
                g += (a.cost.R[i * NU + j] + a.cost.R[j * NU + i]) * (u[j] - goal.u[j]);
                a.L_uu[a.lLuu.at(b, t, i * NU + j)] = a.cost.R[i * NU + j] + a.cost.R[j * NU + i];
            }
            a.L_u[a.lLu.at(b, t, i)] = g;
        }
        for (int e = 0; e < NU * NZ; ++e) a.L_uz[a.lLuz.at(b, t, e)] = T(0);
    }
    a.L[a.lL.at(b, t, 0)] = l;
    return l;
}

// stand-alone cost linearisation of given trajectories: thread = (problem, time)
template <class T, int ENC>
__global__ void __launch_bounds__(64) lq_cost_kernel(const CostDerivArgs<T> a) {
    constexpr int NZ = enc_size(RD, ENC);
    const int64_t id = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (id >= (int64_t)a.B * (a.N + 1)) return;
    const int b = (int)(id / (a.N + 1)), t = (int)(id - (int64_t)b * (a.N + 1));
    if (a.active && a.active[b] != 1) return;
    T z[NZ], u[RNU];
    for (int e = 0; e < NZ; ++e) z[e] = a.Z[a.lZ.at(b, t, e)];
    if (t < a.N)
        for (int i = 0; i < RNU; ++i) u[i] = a.U[a.lU.at(b, t, i)];
    lq_cost_site<T, ENC>(a, site_goal<RD, RNU>(a.cost, b, t, t == a.N), b, t, z, u, t == a.N);
}
template <class T>
__global__ void lq_cost_sum_kernel(const CostDerivArgs<T> a) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    if (a.active && a.active[b] != 1) return;
    T J = T(0);
    for (int t = 0; t <= a.N; ++t) J += a.L[a.lL.at(b, t, 0)];
    a.J_opt[b] = J;
}

// ------------------------------------------------------------------------------------------
// linearise: thread = problem
// ------------------------------------------------------------------------------------------
// STEP: per-step goals (CostParams::xg_bt / ug_bt); a separate instantiation, launched only when they are given.
// PB: problem b's row of p_b (per-problem parameters) instead of dyn, likewise.
template <class T, int ENC, bool STEP, bool PB>
__global__ void __launch_bounds__(64) lq_linearize_kernel(const LinKnownArgs<T> a) {
    constexpr int D = RD, NU = RNU, NZ = enc_size(D, ENC);
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    if (a.active && a.active[b] != 1) return;
    const RdvModel<T> md = rdv_model(PB ? problem_params<GEO_RENDEZVOUS>(a.p_b, b) : a.dyn);
    const bool bounded = a.u_min != nullptr && a.u_max != nullptr;
    auto goal = problem_goal<RD, RNU>(a.cost, b);
    T z[NZ], zn[NZ];
    for (int e = 0; e < NZ; ++e) z[e] = a.z0[(int64_t)b * NZ + e];
    T J = T(0);
    bool finite = true;
    for (int t = 0; t <= a.N; ++t) {
        const bool terminal = t == a.N;
        for (int e = 0; e < NZ; ++e) a.Z[a.lZ.at(b, t, e)] = z[e];
        // ---- cost: value, gradient, Hessian (closed form) ----
        T u[NU];
        if (STEP) step_goal_x(a.cost, b, t, goal);
        if (!terminal) {
            if (STEP) step_goal_u(a.cost, b, t, goal);
#pragma unroll
            for (int i = 0; i < NU; ++i) {
                u[i] = a.U[a.lU.at(b, t, i)];
                if (bounded) u[i] = clampv(u[i], a.u_min[i], a.u_max[i]);   // ref: ilqr.py:459-462
            }
        }
        J += lq_cost_site<T, ENC>(a, goal, b, t, z, u, terminal);
        if (terminal) break;

        // ---- dynamics + Jacobians ----
        rdv_mean_step(md, z, u, zn);
        T U[D][D], Un[D][D];
        if (!rdv_uncertainty_step<ENC, T>(z, zn, U, Un)) finite = false;
        for (int e = 0; e < NZ * NZ; ++e) a.F_z[a.lFz.at(b, t, e)] = T(0);
        for (int e = 0; e < NZ * NU; ++e) a.F_u[a.lFu.at(b, t, e)] = T(0);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            a.F_z[a.lFz.at(b, t, i * NZ + i)] = T(1);
            a.F_z[a.lFz.at(b, t, i * NZ + 4 + i)] = md.dt;
            a.F_z[a.lFz.at(b, t, (4 + i) * NZ + 4 + i)] = md.dvv;
            a.F_u[a.lFu.at(b, t, (4 + i) * NU + i)] = md.dvu;
        }
        if (ENC == ENC_FULL || ENC == ENC_VAR) {
            for (int e = D; e < NZ; ++e) a.F_z[a.lFz.at(b, t, e * NZ + e)] = T(1);
        } else if (ENC == ENC_STD) {
            for (int e = D; e < NZ; ++e) a.F_z[a.lFz.at(b, t, e * NZ + e)] = z[e] / zn[e];
        } else if (ENC == ENC_UT) {
            // column (k, c) of the block: dC = E_kc^T U + U^T E_kc, dU' = chol_upper_diff(U', dC)
            for (int k = 0; k < D; ++k)
                for (int c = k; c < D; ++c) {
                    T dC[D][D], dU[D][D];
#pragma unroll
                    for (int i = 0; i < D; ++i)
#pragma unroll
                        for (int j = 0; j < D; ++j) dC[i][j] = (i == c ? U[k][j] : T(0)) + (j == c ? U[k][i] : T(0));
                    chol_upper_diff<D, T>(Un, dC, dU);
                    const int col = D + tri<D>(k, c);
#pragma unroll
                    for (int i = 0; i < D; ++i)
#pragma unroll
                        for (int j = i; j < D; ++j) a.F_z[a.lFz.at(b, t, (D + tri<D>(i, j)) * NZ + col)] = dU[i][j];
                }
        }
        for (int e = 0; e < NZ; ++e) z[e] = zn[e];
    }
    a.J_opt[b] = J;
    if (a.status && (!finite || !isfinite(J))) a.status[b] |= 2;
}

// ------------------------------------------------------------------------------------------
// rollout of one (problem, alpha)   ref: ilqr.py:677-723 + 764-791
// ------------------------------------------------------------------------------------------
template <class T, int ENC, bool STORE, bool STEP = false, bool PB = false>
__device__ __forceinline__ T lq_roll_one(const RollKnownArgs<T>& a, int b, T alpha) {
    constexpr int D = RD, NU = RNU, NZ = enc_size(D, ENC);
    const RdvModel<T> md = rdv_model(PB ? problem_params<GEO_RENDEZVOUS>(a.p_b, b) : a.dyn);
    const bool bounded = a.u_min != nullptr && a.u_max != nullptr;
    auto goal = problem_goal<RD, RNU>(a.cost, b);           // (dead in the STORE pass, which evaluates no cost)
    T z[NZ], zn[NZ];
    for (int e = 0; e < NZ; ++e) z[e] = a.Z[a.lZ.at(b, 0, e)];
    T J = T(0);
    // running pointers into the step records (48 loads per step: no Layout::at() index arithmetic in the loop)
    const T* pZ = a.Z + a.lZ.at(b, 0, 0);
    const T* pK = a.K + a.lK.at(b, 0, 0);
    const T* pk = a.k + a.lk.at(b, 0, 0);
    const T* pU = a.U + a.lU.at(b, 0, 0);
    T* pZn = STORE ? a.Z_new + a.lZ.at(b, 0, 0) : nullptr;
    T* pUn = STORE ? a.U_new + a.lU.at(b, 0, 0) : nullptr;
    const int64_t seZ = a.lZ.se, seK = a.lK.se, sek = a.lk.se, seU = a.lU.se;
    // per-step goals (NULL unless given), advanced like the step records
    const T* pXg = STEP && !STORE && a.cost.xg_bt ? a.cost.xg_bt + a.cost.lXg.at(b, 0, 0) : nullptr;
    const T* pUg = STEP && !STORE && a.cost.ug_bt ? a.cost.ug_bt + a.cost.lUg.at(b, 0, 0) : nullptr;
    for (int t = 0; t < a.N; ++t) {
        T u[NU];
#pragma unroll
        for (int i = 0; i < NU; ++i) u[i] = alpha * pk[i * sek];
        for (int e = 0; e < NZ; ++e) {
            const T dz = z[e] - pZ[e * seZ];
#pragma unroll
            for (int i = 0; i < NU; ++i) u[i] += dz * pK[(i * NZ + e) * seK];
        }
#pragma unroll
        for (int i = 0; i < NU; ++i) {
            u[i] += pU[i * seU];
            if (bounded) u[i] = clampv(u[i], a.u_min[i], a.u_max[i]);
        }
        pZ += a.lZ.st; pK += a.lK.st; pk += a.lk.st; pU += a.lU.st;
        if (STORE) {
            for (int e = 0; e < NZ; ++e) pZn[e * seZ] = z[e];
#pragma unroll
            for (int i = 0; i < NU; ++i) pUn[i * seU] = u[i];
            pZn += a.lZ.st; pUn += a.lU.st;
        } else {
            if (pXg) {
#pragma unroll
                for (int j = 0; j < D; ++j) goal.x[j] = pXg[j * a.cost.lXg.se];
                pXg += a.cost.lXg.st;
            }
            if (pUg) {
#pragma unroll
                for (int i = 0; i < NU; ++i) goal.u[i] = pUg[i * a.cost.lUg.se];
                pUg += a.cost.lUg.st;
            }
            J += rdv_cost_state<ENC, T>(a.cost, goal.x, z, false) + rdv_cost_action(a.cost, goal.u, u);
        }
        rdv_mean_step(md, z, u, zn);
        T U[D][D], Un[D][D];
        rdv_uncertainty_step<ENC, T>(z, zn, U, Un);
        for (int e = 0; e < NZ; ++e) z[e] = zn[e];
    }
    if (STORE) {
        for (int e = 0; e < NZ; ++e) pZn[e * seZ] = z[e];
    } else {
        if (pXg) {
#pragma unroll
            for (int j = 0; j < D; ++j) goal.x[j] = pXg[j * a.cost.lXg.se];         // row N
        }
        J += rdv_cost_state<ENC, T>(a.cost, goal.x, z, true);
    }
    return J;
}

template <class T, int ENC, bool STEP, bool PB>
__global__ void __launch_bounds__(64) lq_rollout_kernel(const RollKnownArgs<T> a) {
    const int64_t id = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (id >= (int64_t)a.B * a.A) return;
    const int b = (int)(id / a.A), al = (int)(id - (int64_t)b * a.A);
    if ((a.active && a.active[b] == 0) || (a.bw_status && a.bw_status[b] != 0)) return;
    a.J_all[id] = lq_roll_one<T, ENC, false, STEP, PB>(a, b, a.alphas[al]);
}

// argmin with torch semantics (first minimum; a NaN wins outright) + the winner's trajectory
template <class T, int ENC, bool PB>
__global__ void __launch_bounds__(64) lq_select_store_kernel(const RollKnownArgs<T> a) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    if ((a.active && a.active[b] == 0) || (a.bw_status && a.bw_status[b] != 0)) return;
    int best = 0;
    T bj = a.J_all[(int64_t)b * a.A];
    bool bn = bj != bj;
    for (int i = 1; i < a.A; ++i) {
        const T v = a.J_all[(int64_t)b * a.A + i];
        const bool vn = v != v;
        if (!bn && (vn || v < bj)) { best = i; bj = v; bn = vn; }
    }
    a.amin[b] = best;
    a.J_new[b] = bj;
    lq_roll_one<T, ENC, true, false, PB>(a, b, a.alphas[best]);
}

}  // namespace

template <class T>
cudaError_t linearize_lq(int enc, const LinKnownArgs<T>& a, cudaStream_t s) {
    const int th = 64, grid = (a.B + th - 1) / th;
    const bool step = a.cost.xg_bt || a.cost.ug_bt;
#define LQ_LIN(E) if (a.p_b) { if (step) lq_linearize_kernel<T, E, true, true><<<grid, th, 0, s>>>(a); \
                               else lq_linearize_kernel<T, E, false, true><<<grid, th, 0, s>>>(a); } \
                  else if (step) lq_linearize_kernel<T, E, true, false><<<grid, th, 0, s>>>(a); \
                  else lq_linearize_kernel<T, E, false, false><<<grid, th, 0, s>>>(a); break;
    switch (enc) {
        case ENC_FULL: LQ_LIN(ENC_FULL)
        case ENC_UT: LQ_LIN(ENC_UT)
        case ENC_VAR: LQ_LIN(ENC_VAR)
        case ENC_STD: LQ_LIN(ENC_STD)
        case ENC_IGNORE: LQ_LIN(ENC_IGNORE)
        default: return cudaErrorInvalidValue;
    }
#undef LQ_LIN
    return cudaGetLastError();
}

template <class T, bool PB>
__global__ void __launch_bounds__(128) lq_env_step_kernel(int B, KnownParams<T> dyn, const T* p_b, const T* x, const T* u,
                                                          T* xn) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const RdvModel<T> md = rdv_model(PB ? problem_params<GEO_RENDEZVOUS>(p_b, b) : dyn);
    T xi[RD], ui[RNU], xo[RD];
#pragma unroll
    for (int i = 0; i < RD; ++i) xi[i] = x[(int64_t)b * RD + i];
#pragma unroll
    for (int i = 0; i < RNU; ++i) ui[i] = u[(int64_t)b * RNU + i];
    rdv_mean_step(md, xi, ui, xo);
#pragma unroll
    for (int i = 0; i < RD; ++i) xn[(int64_t)b * RD + i] = xo[i];
}
template <class T>
cudaError_t env_step_lq(int B, const KnownParams<T>& dyn, const T* p_b, const T* x, const T* u, T* xn, cudaStream_t s) {
    if (p_b) lq_env_step_kernel<T, true><<<(B + 127) / 128, 128, 0, s>>>(B, dyn, p_b, x, u, xn);
    else lq_env_step_kernel<T, false><<<(B + 127) / 128, 128, 0, s>>>(B, dyn, p_b, x, u, xn);
    return cudaGetLastError();
}
template cudaError_t env_step_lq<float>(int, const KnownParams<float>&, const float*, const float*, const float*, float*,
                                        cudaStream_t);
template cudaError_t env_step_lq<double>(int, const KnownParams<double>&, const double*, const double*, const double*,
                                         double*, cudaStream_t);

template <class T>
cudaError_t cost_derivatives_lq(int enc, const CostDerivArgs<T>& a, cudaStream_t s) {
    const int th = 64;
    const unsigned grid = (unsigned)(((int64_t)a.B * (a.N + 1) + th - 1) / th);
    switch (enc) {
        case ENC_FULL: lq_cost_kernel<T, ENC_FULL><<<grid, th, 0, s>>>(a); break;
        case ENC_UT: lq_cost_kernel<T, ENC_UT><<<grid, th, 0, s>>>(a); break;
        case ENC_VAR: lq_cost_kernel<T, ENC_VAR><<<grid, th, 0, s>>>(a); break;
        case ENC_STD: lq_cost_kernel<T, ENC_STD><<<grid, th, 0, s>>>(a); break;
        case ENC_IGNORE: lq_cost_kernel<T, ENC_IGNORE><<<grid, th, 0, s>>>(a); break;
        default: return cudaErrorInvalidValue;
    }
    if (a.J_opt) lq_cost_sum_kernel<T><<<(a.B + 127) / 128, 128, 0, s>>>(a);
    return cudaGetLastError();
}

template <class T>
cudaError_t rollout_lq(int enc, const RollKnownArgs<T>& a, cudaStream_t s) {
    const int th = 64;
    const unsigned g1 = (unsigned)(((int64_t)a.B * a.A + th - 1) / th), g2 = (a.B + th - 1) / th;
    const bool step = a.cost.xg_bt || a.cost.ug_bt;
#define LQ_ROLL(E) if (a.p_b) { if (step) lq_rollout_kernel<T, E, true, true><<<g1, th, 0, s>>>(a); \
                                else lq_rollout_kernel<T, E, false, true><<<g1, th, 0, s>>>(a); \
                                lq_select_store_kernel<T, E, true><<<g2, th, 0, s>>>(a); } \
                   else { if (step) lq_rollout_kernel<T, E, true, false><<<g1, th, 0, s>>>(a); \
                          else lq_rollout_kernel<T, E, false, false><<<g1, th, 0, s>>>(a); \
                          lq_select_store_kernel<T, E, false><<<g2, th, 0, s>>>(a); } break;
    switch (enc) {
        case ENC_FULL: LQ_ROLL(ENC_FULL)
        case ENC_UT: LQ_ROLL(ENC_UT)
        case ENC_VAR: LQ_ROLL(ENC_VAR)
        case ENC_STD: LQ_ROLL(ENC_STD)
        case ENC_IGNORE: LQ_ROLL(ENC_IGNORE)
        default: return cudaErrorInvalidValue;
    }
#undef LQ_ROLL
    return cudaGetLastError();
}

template cudaError_t linearize_lq<float>(int, const LinKnownArgs<float>&, cudaStream_t);
template cudaError_t linearize_lq<double>(int, const LinKnownArgs<double>&, cudaStream_t);
template cudaError_t cost_derivatives_lq<float>(int, const CostDerivArgs<float>&, cudaStream_t);
template cudaError_t cost_derivatives_lq<double>(int, const CostDerivArgs<double>&, cudaStream_t);
template cudaError_t rollout_lq<float>(int, const RollKnownArgs<float>&, cudaStream_t);
template cudaError_t rollout_lq<double>(int, const RollKnownArgs<double>&, cudaStream_t);

}  // namespace pddp
