// Known-dynamics path: fused linearisation (nominal rollout + forward-mode derivatives of the
// dynamics and the cost) and the line-search rollout.  One thread owns one problem (linearise) or
// one (problem, alpha) pair (rollout); time is sequential inside the thread, state lives in
// registers, and with PDDP_BATCH_INNER layout every global access is coalesced across problems.
//
// Roofline: HBM.  Per trajectory-step the linearise kernel writes 2nz^2+2nz*nu+2nz+nu+nu^2+1
// elements and reads nu; the rollout reads nz+2nu+nu*nz (shared by all alphas through L1/L2) and
// writes nz+nu for the winner (SURVEY.md 8d).
#include "core.cuh"
#include "kernels.h"

namespace pddp {

// ------------------------------------------------------------------------------------------
// cost value / gradient / Hessian w.r.t. the encoded state, one thread
// ------------------------------------------------------------------------------------------
template <class T, int GEO, int ENC, class EmitH>
__device__ __forceinline__ void cost_derivs_thread(const CostParams<T>& cp, const T* xg, const T* z, bool terminal,
                                                   T& l, T* lz, EmitH&& emit_h) {
    constexpr int D = Geo<GEO>::D;
    constexpr int NZ = enc_size(D, ENC);
    if (ENC == ENC_IGNORE && D <= 4) {
        // one evaluation on a full second-order jet: value, D gradients, D(D+1)/2 Hessian entries
        typedef Jet2<T, D> S;
        S zj[NZ];
#pragma unroll
        for (int k = 0; k < NZ; ++k) {
            zj[k] = S(z[k]);
            zj[k].g[k] = T(1);
        }
        S r = cost_state<GEO, ENC, T, S>(cp, xg, zj, terminal);
        l = r.v;
#pragma unroll
        for (int i = 0; i < D; ++i) lz[i] = r.g[i];
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = i; j < D; ++j) emit_h(i, j, r.h[tri<D>(i, j)]);
    } else {
        // hyper-dual sweep over the upper triangle: seeds (e_i, e_j) -> h(0,1) = d2l/dz_i dz_j
        typedef Jet2<T, 2> S;
        for (int i = 0; i < NZ; ++i)
            for (int j = i; j < NZ; ++j) {
                S zj[NZ];
#pragma unroll
                for (int k = 0; k < NZ; ++k) {
                    zj[k] = S(z[k]);
                    zj[k].g[0] = k == i ? T(1) : T(0);
                    zj[k].g[1] = k == j ? T(1) : T(0);
                }
                S r = cost_state<GEO, ENC, T, S>(cp, xg, zj, terminal);
                if (i == j) {
                    l = r.v;
                    lz[i] = r.g[0];
                }
                emit_h(i, j, r.h[1]);   // for i == j both seeds coincide and h(0,1) == d2/dz_i^2
            }
    }
}

// ------------------------------------------------------------------------------------------
// linearise
// ------------------------------------------------------------------------------------------
// STEP: the cost reads per-step goals (CostParams::xg_bt / ug_bt).  A separate instantiation, launched only when they
// are given, so the shared and per-problem goals keep the code (and the registers) they had without them.
// PB: the dynamics read problem b's row of p_b (per-problem parameters), likewise a separate instantiation.
template <class T, int GEO, int ENC, bool STEP, bool PB>
__global__ void __launch_bounds__(128) linearize_known_kernel(const LinKnownArgs<T> a) {
    typedef Geo<GEO> G;
    constexpr int D = G::D, NU = G::NU, NZ = enc_size(D, ENC);
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    if (a.active && a.active[b] != 1) return;   // 1 = (re)linearise, 2 = retry with the old one
    auto goal = problem_goal<GEO>(a.cost, b);
    KnownParams<T> pb;
    if (PB) pb = problem_params<GEO>(a.p_b, b);
    const KnownParams<T>& dyn = PB ? pb : a.dyn;

    T z[NZ];
#pragma unroll
    for (int e = 0; e < NZ; ++e) z[e] = a.z0[(int64_t)b * NZ + e];
    const bool bounded = a.u_min != nullptr && a.u_max != nullptr;
    T lo = bounded ? a.u_min[0] : T(0), hi = bounded ? a.u_max[0] : T(0);
    T J = T(0);

    for (int t = 0; t <= a.N; ++t) {
        const bool terminal = t == a.N;
#pragma unroll
        for (int e = 0; e < NZ; ++e) a.Z[a.lZ.at(b, t, e)] = z[e];
        if (STEP) step_goal_x(a.cost, b, t, goal);

        // ---- cost (fused for IGNORE_UNCERTAINTY; the uncertain encodings run the
        //      (problem, time, Hessian-pair)-parallel cost_pairs_kernel on Z afterwards) ----
        T l = T(0);
        if (ENC == ENC_IGNORE) {
            T lz[NZ];
            cost_derivs_thread<T, GEO, ENC>(a.cost, goal.x, z, terminal, l, lz, [&](int i, int j, T h) {
                a.L_zz[a.lLzz.at(b, t, i * NZ + j)] = h;
                if (i != j) a.L_zz[a.lLzz.at(b, t, j * NZ + i)] = h;
            });
#pragma unroll
            for (int e = 0; e < NZ; ++e) a.L_z[a.lLz.at(b, t, e)] = lz[e];
        }
        if (terminal) {
            if (ENC == ENC_IGNORE) a.L[a.lL.at(b, t, 0)] = l;
            J += l;
            break;
        }
        T u = a.U[a.lU.at(b, t, 0)];
        if (bounded) u = clampv(u, lo, hi);      // ref: ilqr.py:459-462, derivatives w.r.t. the clamped u
        if (a.U_clamped) a.U_clamped[a.lU.at(b, t, 0)] = u;
        if (ENC == ENC_IGNORE) {
            if (STEP) step_goal_u(a.cost, b, t, goal);
            T la, lu, luu;
            cost_action(a.cost, goal.u[0], u, la, lu, luu);
            l += la;
            J += l;
            a.L[a.lL.at(b, t, 0)] = l;
            a.L_u[a.lLu.at(b, t, 0)] = lu;
            a.L_uu[a.lLuu.at(b, t, 0)] = luu;
#pragma unroll
            for (int e = 0; e < NZ; ++e) a.L_uz[a.lLuz.at(b, t, e)] = T(0);
        }

        // ---- dynamics: mean on first-order jets over (x, u) ----
        typedef Jet1<T, D + NU> S1;
        S1 x[D], xn[D], uj = S1::variable(u, D);
#pragma unroll
        for (int i = 0; i < D; ++i) x[i] = S1::variable(z[i], i);
        known_mean_step<GEO, T, S1>(dyn, x, uj, xn);
        T zn[NZ];
#pragma unroll
        for (int i = 0; i < D; ++i) zn[i] = xn[i].v;
        known_uncertainty_step<D, ENC, T>(z, zn);

        if (NZ > D) {
#pragma unroll 1
            for (int e = 0; e < NZ * NZ; ++e) a.F_z[a.lFz.at(b, t, e)] = T(0);
#pragma unroll 1
            for (int e = D; e < NZ; ++e) a.F_u[a.lFu.at(b, t, e)] = T(0);
        }
#pragma unroll
        for (int r = 0; r < D; ++r) {
#pragma unroll
            for (int c = 0; c < D; ++c) a.F_z[a.lFz.at(b, t, r * NZ + c)] = xn[r].d[c];
            a.F_u[a.lFu.at(b, t, r)] = xn[r].d[D];
        }
        known_uncertainty_jacobian<D, ENC, T>(z, zn, [&](int r, int c, T v) {
            a.F_z[a.lFz.at(b, t, r * NZ + c)] = v;
        });
#pragma unroll
        for (int e = 0; e < NZ; ++e) z[e] = zn[e];
    }
    if (ENC == ENC_IGNORE) {
        a.J_opt[b] = J;
        if (a.status && !isfinite(J)) a.status[b] |= 2;
    }
}

// ------------------------------------------------------------------------------------------
// rollout + line search.  GA lanes (16 or 32) share one problem, lane = alpha.
// pass 1: every alpha rolls the control law and accumulates its trajectory cost
//         (ref: ilqr.py:677-723 + 764-791); group argmin by shuffles (first minimum wins, any NaN
//         wins outright like torch.argmin).
// pass 2: the winning lane replays its rollout and stores Z_new / U_new.
// ------------------------------------------------------------------------------------------
template <class T, int GEO, int ENC, bool STORE, bool STEP = false, bool PB = false>
__device__ __forceinline__ T roll_one(const RollKnownArgs<T>& a, int b, T alpha, bool bounded, T lo, T hi) {
    typedef Geo<GEO> G;
    constexpr int D = G::D, NZ = enc_size(D, ENC);
    auto goal = problem_goal<GEO>(a.cost, b);                 // (dead in the STORE pass, which evaluates no cost)
    // per-problem parameters: the GA lanes of the problem read the same row, a broadcast load
    KnownParams<T> pb;
    if (PB) pb = problem_params<GEO>(a.p_b, b);
    const KnownParams<T>& dyn = PB ? pb : a.dyn;
    T z[NZ];
#pragma unroll
    for (int e = 0; e < NZ; ++e) z[e] = a.Z[a.lZ.at(b, 0, e)];
    T J = T(0);
    // running pointers into the step records (the loop is bound by instruction issue: the 64-bit index arithmetic of
    // six Layout::at() calls per step was a quarter of it)
    const T* pZ = a.Z + a.lZ.at(b, 0, 0);
    const T* pK = a.K + a.lK.at(b, 0, 0);
    const T* pk = a.k + a.lk.at(b, 0, 0);
    const T* pU = a.U + a.lU.at(b, 0, 0);
    T* pZn = STORE ? a.Z_new + a.lZ.at(b, 0, 0) : nullptr;
    T* pUn = STORE ? a.U_new + a.lU.at(b, 0, 0) : nullptr;
    const int64_t seZ = a.lZ.se, seK = a.lK.se;
    // per-step goals (NULL unless given): rows shared by the GA lanes of the problem, a broadcast load
    const T* pXg = STEP && !STORE && a.cost.xg_bt ? a.cost.xg_bt + a.cost.lXg.at(b, 0, 0) : nullptr;
    const T* pUg = STEP && !STORE && a.cost.ug_bt ? a.cost.ug_bt + a.cost.lUg.at(b, 0, 0) : nullptr;
    for (int t = 0; t < a.N; ++t) {
        T du = alpha * pk[0];
#pragma unroll
        for (int e = 0; e < NZ; ++e) du += (z[e] - pZ[e * seZ]) * pK[e * seK];
        T u = pU[0] + du;
        if (bounded) u = clampv(u, lo, hi);
        if (STORE) {
#pragma unroll
            for (int e = 0; e < NZ; ++e) pZn[e * seZ] = z[e];
            pUn[0] = u;
            pZn += a.lZ.st; pUn += a.lU.st;
        }
        pZ += a.lZ.st; pK += a.lK.st; pk += a.lk.st; pU += a.lU.st;
        StateTrig<GEO, T> tr;                               // shared by the cost and the dynamics of this step
        state_trig<GEO, T>(z, tr);
        if (!STORE) {
            if (pXg) {
#pragma unroll
                for (int j = 0; j < G::DA; ++j) goal.x[j] = pXg[j * a.cost.lXg.se];
                pXg += a.cost.lXg.st;
            }
            if (pUg) {
                goal.u[0] = pUg[0];
                pUg += a.cost.lUg.st;
            }
            T la, lu, luu;
            cost_action(a.cost, goal.u[0], u, la, lu, luu);
            J += cost_state<GEO, ENC, T, T>(a.cost, goal.x, z, false, tr) + la;
        }
        T zn[NZ];
        known_mean_step<GEO, T, T>(dyn, z, u, zn, tr);
        known_uncertainty_step<D, ENC, T>(z, zn);
#pragma unroll
        for (int e = 0; e < NZ; ++e) z[e] = zn[e];
    }
    if (STORE) {
#pragma unroll
        for (int e = 0; e < NZ; ++e) pZn[e * seZ] = z[e];
    } else {
        if (pXg) {
#pragma unroll
            for (int j = 0; j < G::DA; ++j) goal.x[j] = pXg[j * a.cost.lXg.se];     // row N
        }
        J += cost_state<GEO, ENC, T, T>(a.cost, goal.x, z, true);
    }
    return J;
}

// GA lanes = the alphas of one problem, 32/GA problems per warp (GA = 10: three problems on 30 lanes,
// the reference's default line search has 10 alphas; GA = 16 / 32 for longer searches).
template <class T, int GEO, int ENC, int GA, bool STEP, bool PB = false>
__global__ void __launch_bounds__(128) rollout_known_kernel(const RollKnownArgs<T> a) {
    constexpr int GPW = 32 / GA;                           // problems per warp
    const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int lane32 = threadIdx.x & 31, grp = lane32 / GA, lane = lane32 - grp * GA;
    const int64_t b64 = (tid >> 5) * GPW + grp;
    const int b = (int)b64;
    const bool live = grp < GPW && b64 < a.B && (!a.active || a.active[b] != 0) && (!a.bw_status || a.bw_status[b] == 0);
    const bool bounded = a.u_min != nullptr && a.u_max != nullptr;
    T lo = bounded ? a.u_min[0] : T(0), hi = bounded ? a.u_max[0] : T(0);
    const bool has_alpha = live && lane < a.A;
    T alpha = has_alpha ? a.alphas[lane] : T(0);
    T J = has_alpha ? roll_one<T, GEO, ENC, false, STEP, PB>(a, b, alpha, bounded, lo, hi) : T(INFINITY);
    if (has_alpha) a.J_all[(int64_t)b * a.A + lane] = J;

    // argmin with torch semantics (NaN beats everything, ties -> lowest index): every lane scans
    // its group's candidates in index order
    const unsigned full = 0xffffffffu;
    T best = T(INFINITY);
    int idx = 0;
    bool nan = false, any = false;
#pragma unroll
    for (int c = 0; c < GA; ++c) {
        const int src = (grp < GPW ? grp : 0) * GA + c;
        const T oJ = __shfl_sync(full, J, src);
        if (c >= a.A) continue;
        const bool on = oJ != oJ;
        const bool take = !any || (!nan && (on || oJ < best));
        if (take) { best = oJ; idx = c; nan = on; any = true; }
    }
    if (!live) return;
    if (lane == 0) {
        a.amin[b] = idx;
        a.J_new[b] = best;
    }
}

// Second pass: ONE THREAD PER PROBLEM re-rolls the winning alpha and stores its trajectory.  Done
// inside the kernel above, only one lane of each alpha group would be busy: the same warp-level
// instruction count as the all-alpha pass for 1/16 of the useful work.  Here every lane works, and
// with the BATCH_INNER layout every store is a coalesced line.
template <class T, int GEO, int ENC, bool PB = false>
__global__ void __launch_bounds__(128) rollout_known_store_kernel(const RollKnownArgs<T> a) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    if ((a.active && a.active[b] == 0) || (a.bw_status && a.bw_status[b] != 0)) return;
    const bool bounded = a.u_min != nullptr && a.u_max != nullptr;
    const T lo = bounded ? a.u_min[0] : T(0), hi = bounded ? a.u_max[0] : T(0);
    roll_one<T, GEO, ENC, true, false, PB>(a, b, a.alphas[a.amin[b]], bounded, lo, hi);
}

// ------------------------------------------------------------------------------------------
// host dispatch
// ------------------------------------------------------------------------------------------
template <class T, int GEO, int ENC, bool PB>
static void launch_lin_pb(const LinKnownArgs<T>& a, cudaStream_t s) {
    const int threads = 128, grid = (a.B + threads - 1) / threads;
    // (the uncertain encodings evaluate the cost in cost_pairs_kernel: their linearisation reads no goal)
    if (ENC == ENC_IGNORE && (a.cost.xg_bt || a.cost.ug_bt))
        linearize_known_kernel<T, GEO, ENC, ENC == ENC_IGNORE, PB><<<grid, threads, 0, s>>>(a);
    else
        linearize_known_kernel<T, GEO, ENC, false, PB><<<grid, threads, 0, s>>>(a);
}
template <class T, int GEO, int ENC>
static cudaError_t launch_lin(const LinKnownArgs<T>& a, cudaStream_t s) {
    if (a.p_b) launch_lin_pb<T, GEO, ENC, true>(a, s);
    else launch_lin_pb<T, GEO, ENC, false>(a, s);
    return cudaGetLastError();
}
template <class T, int GEO, int ENC>
static cudaError_t launch_roll(const RollKnownArgs<T>& a, cudaStream_t s) {
    const int threads = 128;
    const bool step = a.cost.xg_bt || a.cost.ug_bt;
    if (a.p_b) {                                 // per-problem parameters: GA = 10 or 32, with or without per-step goals
        const int64_t total = a.A <= 10 ? ((int64_t)a.B + 2) / 3 * 32 : (int64_t)a.B * 32;
        const unsigned grid = (unsigned)((total + threads - 1) / threads);
        if (a.A <= 10) {
            if (step) rollout_known_kernel<T, GEO, ENC, 10, true, true><<<grid, threads, 0, s>>>(a);
            else rollout_known_kernel<T, GEO, ENC, 10, false, true><<<grid, threads, 0, s>>>(a);
        } else {
            if (step) rollout_known_kernel<T, GEO, ENC, 32, true, true><<<grid, threads, 0, s>>>(a);
            else rollout_known_kernel<T, GEO, ENC, 32, false, true><<<grid, threads, 0, s>>>(a);
        }
        rollout_known_store_kernel<T, GEO, ENC, true><<<(a.B + threads - 1) / threads, threads, 0, s>>>(a);
        return cudaGetLastError();
    }
    if (step) {                                  // per-step goals: GA = 10 or 32 (no third instantiation for 16)
        const int64_t total = a.A <= 10 ? ((int64_t)a.B + 2) / 3 * 32 : (int64_t)a.B * 32;
        const unsigned grid = (unsigned)((total + threads - 1) / threads);
        if (a.A <= 10) rollout_known_kernel<T, GEO, ENC, 10, true><<<grid, threads, 0, s>>>(a);
        else rollout_known_kernel<T, GEO, ENC, 32, true><<<grid, threads, 0, s>>>(a);
    } else if (a.A <= 10) {
        const int64_t total = ((int64_t)a.B + 2) / 3 * 32;
        rollout_known_kernel<T, GEO, ENC, 10, false><<<(unsigned)((total + threads - 1) / threads), threads, 0, s>>>(a);
    } else if (a.A <= 16) {
        const int64_t total = (int64_t)a.B * 16;
        rollout_known_kernel<T, GEO, ENC, 16, false><<<(unsigned)((total + threads - 1) / threads), threads, 0, s>>>(a);
    } else {
        const int64_t total = (int64_t)a.B * 32;
        rollout_known_kernel<T, GEO, ENC, 32, false><<<(unsigned)((total + threads - 1) / threads), threads, 0, s>>>(a);
    }
    rollout_known_store_kernel<T, GEO, ENC><<<(a.B + threads - 1) / threads, threads, 0, s>>>(a);
    return cudaGetLastError();
}

#define PDDP_DISPATCH_GEO_ENC(FN, geo, enc, ...)                                                  \
    switch ((geo) * 8 + (enc)) {                                                                  \
        case GEO_PENDULUM * 8 + ENC_FULL: return FN<T, GEO_PENDULUM, ENC_FULL>(__VA_ARGS__);      \
        case GEO_PENDULUM * 8 + ENC_UT: return FN<T, GEO_PENDULUM, ENC_UT>(__VA_ARGS__);          \
        case GEO_PENDULUM * 8 + ENC_IGNORE: return FN<T, GEO_PENDULUM, ENC_IGNORE>(__VA_ARGS__);  \
        case GEO_PENDULUM * 8 + ENC_VAR: return FN<T, GEO_PENDULUM, ENC_VAR>(__VA_ARGS__);        \
        case GEO_PENDULUM * 8 + ENC_STD: return FN<T, GEO_PENDULUM, ENC_STD>(__VA_ARGS__);        \
        case GEO_CARTPOLE * 8 + ENC_VAR: return FN<T, GEO_CARTPOLE, ENC_VAR>(__VA_ARGS__);        \
        case GEO_CARTPOLE * 8 + ENC_STD: return FN<T, GEO_CARTPOLE, ENC_STD>(__VA_ARGS__);        \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_VAR: return FN<T, GEO_DOUBLE_CARTPOLE, ENC_VAR>(__VA_ARGS__); \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_STD: return FN<T, GEO_DOUBLE_CARTPOLE, ENC_STD>(__VA_ARGS__); \
        case GEO_CARTPOLE * 8 + ENC_FULL: return FN<T, GEO_CARTPOLE, ENC_FULL>(__VA_ARGS__);      \
        case GEO_CARTPOLE * 8 + ENC_UT: return FN<T, GEO_CARTPOLE, ENC_UT>(__VA_ARGS__);          \
        case GEO_CARTPOLE * 8 + ENC_IGNORE: return FN<T, GEO_CARTPOLE, ENC_IGNORE>(__VA_ARGS__);  \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_FULL: return FN<T, GEO_DOUBLE_CARTPOLE, ENC_FULL>(__VA_ARGS__); \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_UT: return FN<T, GEO_DOUBLE_CARTPOLE, ENC_UT>(__VA_ARGS__);     \
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_IGNORE: return FN<T, GEO_DOUBLE_CARTPOLE, ENC_IGNORE>(__VA_ARGS__); \
        default: return cudaErrorInvalidValue;                                                    \
    }

// ------------------------------------------------------------------------------------------
// ground-truth simulator step of the example environments, thread = environment instance
// (ref: examples/*/env.py step(): x' = model(x, u, 0, IGNORE_UNCERTAINTY))
// ------------------------------------------------------------------------------------------
// PB: instance b simulates the system of row b of p_b
template <class T, int GEO, bool PB>
__global__ void __launch_bounds__(128) env_step_kernel(int B, KnownParams<T> dyn, const T* p_b, const T* x, const T* u,
                                                       T* xn) {
    constexpr int D = Geo<GEO>::D;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    KnownParams<T> pb;
    if (PB) pb = problem_params<GEO>(p_b, b);
    T xi[D], xo[D];
#pragma unroll
    for (int i = 0; i < D; ++i) xi[i] = x[(int64_t)b * D + i];
    known_mean_step<GEO, T, T>(PB ? pb : dyn, xi, u[b], xo);
#pragma unroll
    for (int i = 0; i < D; ++i) xn[(int64_t)b * D + i] = xo[i];
}
template <class T, int GEO>
static void launch_env_step(int B, const KnownParams<T>& dyn, const T* p_b, const T* x, const T* u, T* xn, cudaStream_t s) {
    const int th = 128, grid = (B + th - 1) / th;
    if (p_b) env_step_kernel<T, GEO, true><<<grid, th, 0, s>>>(B, dyn, p_b, x, u, xn);
    else env_step_kernel<T, GEO, false><<<grid, th, 0, s>>>(B, dyn, p_b, x, u, xn);
}
template <class T>
cudaError_t env_step_known(int geo, int B, const KnownParams<T>& dyn, const T* p_b, const T* x, const T* u, T* xn,
                           cudaStream_t s) {
    switch (geo) {
        case GEO_PENDULUM: launch_env_step<T, GEO_PENDULUM>(B, dyn, p_b, x, u, xn, s); break;
        case GEO_CARTPOLE: launch_env_step<T, GEO_CARTPOLE>(B, dyn, p_b, x, u, xn, s); break;
        case GEO_DOUBLE_CARTPOLE: launch_env_step<T, GEO_DOUBLE_CARTPOLE>(B, dyn, p_b, x, u, xn, s); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}
template cudaError_t env_step_known<PDDP_KNOWN_T>(int, int, const KnownParams<PDDP_KNOWN_T>&, const PDDP_KNOWN_T*,
                                                  const PDDP_KNOWN_T*, const PDDP_KNOWN_T*, PDDP_KNOWN_T*, cudaStream_t);

template <class T>
cudaError_t linearize_known(int geo, int enc, const LinKnownArgs<T>& a, cudaStream_t s) {
    PDDP_DISPATCH_GEO_ENC(launch_lin, geo, enc, a, s)
}
template <class T>
cudaError_t rollout_known(int geo, int enc, const RollKnownArgs<T>& a, cudaStream_t s) {
    PDDP_DISPATCH_GEO_ENC(launch_roll, geo, enc, a, s)
}
template cudaError_t linearize_known<PDDP_KNOWN_T>(int, int, const LinKnownArgs<PDDP_KNOWN_T>&, cudaStream_t);
template cudaError_t rollout_known<PDDP_KNOWN_T>(int, int, const RollKnownArgs<PDDP_KNOWN_T>&, cudaStream_t);

}  // namespace pddp
