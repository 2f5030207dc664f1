// Backward Riccati pass for action_size > 1 (ref: pddp/controllers/ilqr.py:489-674, default
// V_zz_reg=False branch; pddp/utils/constraint.py:150-266 for the box-constrained feed-forward term).
//
// Same organisation as backward_warp_kernel (backward.cu): a TEAM of threads (a warp, or a CTA for
// nz >= 24) owns one problem, V_zz / F_z / V_zz.F_z live in shared memory, time runs from N-1 down to
// 0.  What changes with nu > 1 is the small dense algebra on Q_uu (nu x nu, nu <= 4):
//   * eigen-clipping (ilqr.py:631-634): cyclic Jacobi rotations on the symmetrised Q_uu, in registers,
//     every thread of the team redundantly (the inputs are team-uniform, so are the results);
//   * unconstrained gains [k|K] = -(E/e)E^T [Q_u|Q_uz], NaN -> the reference raises (ilqr.py:636-640);
//   * with bounds: Q_uu_reg = E diag(e) E^T, k = boxqp(warm start k[t+1], ...), K[free] =
//     -Q_uu_reg[free,free]^-1 Q_uz[free], clamped rows of K stay zero (ilqr.py:642-662).
// The box-QP works on the full nu x nu system with clamped dimensions decoupled (unit diagonal, zero
// off-diagonal): the Cholesky factor restricted to the free dimensions is then exactly the factor of
// Q[free][:, free] the reference computes, without gathering index lists.
// Roofline: HBM -- per trajectory-step 2nz^2+2nz*nu+nz+nu+nu^2 elements read, nu+nu*nz written.
#include "core.cuh"
#include "kernels.h"

namespace pddp {

constexpr int MNU = MAX_NU;

// TEAM threads own one problem: a whole CTA (256), a warp (32), or a SUB-WARP team of 4 / 8 lanes -- several
// problems per warp, so the team-uniform scalar algebra (Jacobi sweeps, box-QP Newton iterations) that every lane
// executes redundantly is paid once per 8 / 4 problems instead of once per problem, and with the
// BATCH_INNER layout the lanes that hold the same element of consecutive problems read full 32-byte sectors.
template <int TEAM>
__device__ __forceinline__ unsigned nu_team_mask() {
    return TEAM >= 32 ? 0xffffffffu : (((1u << (TEAM & 31)) - 1u) << ((threadIdx.x & 31) / TEAM * TEAM));
}
// Sub-warp teams synchronise with a FULL-warp barrier: it is also the point where the teams of a warp re-converge
// after the data-dependent scalar part (Jacobi sweeps, box-QP iterations).  With per-team masks the teams stayed
// diverged and the warp issued the matrix code once per team (17 k instructions per warp and time step).  Teams
// that left the time loop (not positive definite) or the kernel are exited threads and do not take part.
template <int TEAM>
__device__ __forceinline__ void nu_team_sync() {
    if (TEAM <= 32) __syncwarp(); else __syncthreads();
}
template <int TEAM>
__device__ __forceinline__ bool nu_team_any(bool x) {
    if (TEAM <= 32) return __any_sync(nu_team_mask<TEAM>(), x);
    return __syncthreads_or(x) != 0;
}

// Eigen-decomposition of a symmetric n x n matrix (n <= MNU) by cyclic Jacobi: A = E diag(e) E^T.
// Static loops over MNU with n guards keep everything in registers.
template <class T>
__device__ __forceinline__ void jacobi_eig(int n, T (&A)[MNU][MNU], T (&E)[MNU][MNU], T (&e)[MNU]) {
#pragma unroll
    for (int i = 0; i < MNU; ++i)
#pragma unroll
        for (int j = 0; j < MNU; ++j) E[i][j] = i == j ? T(1) : T(0);
    for (int sweep = 0; sweep < 16; ++sweep) {
        T off = T(0), dia = T(0);
#pragma unroll
        for (int p = 0; p < MNU; ++p) {
            if (p < n) dia += A[p][p] * A[p][p];
#pragma unroll
            for (int q = p + 1; q < MNU; ++q)
                if (q < n) off += A[p][q] * A[p][q];
        }
        const T eps = sizeof(T) == 4 ? T(1e-14) : T(1e-32);       // (machine epsilon)^2
        if (!(off > eps * dia)) break;
#pragma unroll
        for (int p = 0; p < MNU; ++p)
#pragma unroll
            for (int q = p + 1; q < MNU; ++q) {
                if (q >= n || A[p][q] == T(0)) continue;
                const T theta = (A[q][q] - A[p][p]) / (T(2) * A[p][q]);
                const T tt = (theta >= T(0) ? T(1) : T(-1)) / (fabs(theta) + jsqrt(theta * theta + T(1)));
                const T c = T(1) / jsqrt(tt * tt + T(1)), s = tt * c;
#pragma unroll
                for (int k = 0; k < MNU; ++k) {                    // columns p, q of A and E
                    const T akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - s * akq;
                    A[k][q] = s * akp + c * akq;
                    const T ekp = E[k][p], ekq = E[k][q];
                    E[k][p] = c * ekp - s * ekq;
                    E[k][q] = s * ekp + c * ekq;
                }
#pragma unroll
                for (int k = 0; k < MNU; ++k) {                    // rows p, q of A
                    const T apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - s * aqk;
                    A[q][k] = s * apk + c * aqk;
                }
            }
    }
#pragma unroll
    for (int i = 0; i < MNU; ++i) e[i] = A[i][i];
}

// Upper Cholesky factor of Q with the non-free dimensions decoupled; false where potrf would fail.
template <class T>
__device__ __forceinline__ bool masked_chol(const T (&Q)[MNU][MNU], unsigned free, T (&U)[MNU][MNU]) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i < MNU; ++i) {
        const bool fi = (free >> i) & 1u;
#pragma unroll
        for (int j = 0; j < MNU; ++j) {
            if (j < i) { U[i][j] = T(0); continue; }
            const bool fj = (free >> j) & 1u;
            T s = (fi && fj) ? Q[i][j] : (i == j ? T(1) : T(0));
#pragma unroll
            for (int k = 0; k < i; ++k) s -= U[k][i] * U[k][j];
            if (i == j) {
                if (!(s > T(0))) ok = false;
                U[i][i] = jsqrt(s);
            } else {
                U[i][j] = s / U[i][i];
            }
        }
    }
    return ok;
}
// x = (U^T U)^-1 r  (potrs with the upper factor); r must be zero on the non-free dimensions.
template <class T>
__device__ __forceinline__ void chol_solve(const T (&U)[MNU][MNU], const T (&r)[MNU], T (&x)[MNU]) {
    T y[MNU];
#pragma unroll
    for (int i = 0; i < MNU; ++i) {
        T s = r[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s -= U[k][i] * y[k];
        y[i] = s / U[i][i];
    }
#pragma unroll
    for (int i = MNU - 1; i >= 0; --i) {
        T s = y[i];
#pragma unroll
        for (int k = i + 1; k < MNU; ++k) s -= U[i][k] * x[k];
        x[i] = s / U[i][i];
    }
}

template <class T>
__device__ __forceinline__ T qp_objective(int n, const T (&Q)[MNU][MNU], const T (&c)[MNU], const T (&x)[MNU]) {
    T quad = T(0), lin = T(0);
#pragma unroll
    for (int i = 0; i < MNU; ++i) {
        if (i >= n) continue;
        T row = T(0);
#pragma unroll
        for (int j = 0; j < MNU; ++j)
            if (j < n) row += x[j] * Q[j][i];
        quad += row * x[i];
        lin += x[i] * c[i];
    }
    return T(0.5) * quad + lin;
}

// Projected-Newton box QP, a restatement of the reference loop (constraint.py:150-266) on an n x n
// problem.  Returns the reference's result code; x = solution, free = bit mask of the dimensions that
// were not clamped at exit, Uf = the Cholesky factor belonging to that set.
template <class T>
__device__ __forceinline__ int boxqp_n(int n, const T (&x0)[MNU], const T (&Q)[MNU][MNU], const T (&c)[MNU],
                                       const T (&lo)[MNU], const T (&hi)[MNU], T (&x)[MNU], unsigned& free,
                                       T (&Uf)[MNU][MNU]) {
    const T min_grad = T(1e-8), tol = T(1e-8), step_dec = T(0.6), min_step = T(1e-22), armijo = T(0.1);
    const unsigned all = (1u << n) - 1u;
#pragma unroll
    for (int i = 0; i < MNU; ++i) {
        x[i] = i < n ? clampv(x0[i], lo[i], hi[i]) : T(0);
        if (isinf(x[i])) x[i] = T(0);
    }
    T f = qp_objective(n, Q, c, x);
    int result = 0;
    T old_f = T(0);
    unsigned clamped = 0u;
    free = all;
#pragma unroll
    for (int i = 0; i < MNU; ++i)
#pragma unroll
        for (int j = 0; j < MNU; ++j) Uf[i][j] = i == j ? T(1) : T(0);
    for (int it = 0; it < 100; ++it) {
        if (result != 0) break;
        if (it > 0 && (old_f - f) < tol * fabs(old_f)) { result = 4; break; }
        old_f = f;
        T g[MNU];
#pragma unroll
        for (int i = 0; i < MNU; ++i) {
            T s = i < n ? c[i] : T(0);
#pragma unroll
            for (int j = 0; j < MNU; ++j)
                if (i < n && j < n) s += Q[i][j] * x[j];
            g[i] = s;
        }
        const unsigned was = clamped;
        clamped = 0u;
#pragma unroll
        for (int i = 0; i < MNU; ++i)
            if (i < n && ((x[i] == lo[i] && g[i] > T(0)) || (x[i] == hi[i] && g[i] < T(0)))) clamped |= 1u << i;
        free = all & ~clamped;
        if (clamped == all) { result = 6; break; }
        if (it == 0 || was != clamped) {
            if (!masked_chol(Q, free, Uf)) { result = -1; break; }
        }
        T gn = T(0);
#pragma unroll
        for (int i = 0; i < MNU; ++i)
            if ((free >> i) & 1u) gn += g[i] * g[i];
        if (jsqrt(gn) < min_grad) { result = 5; break; }
        T gc[MNU], sol[MNU], search[MNU];                          // g_clamped = Q (x o clamped) + c on the free dims
#pragma unroll
        for (int i = 0; i < MNU; ++i) {
            T s = T(0);
            if ((free >> i) & 1u) {
                s = c[i];
#pragma unroll
                for (int j = 0; j < MNU; ++j)
                    if ((clamped >> j) & 1u) s += Q[i][j] * x[j];
            }
            gc[i] = s;
        }
        chol_solve(Uf, gc, sol);
        T sdotg = T(0);
#pragma unroll
        for (int i = 0; i < MNU; ++i) {
            search[i] = ((free >> i) & 1u) ? -sol[i] - x[i] : T(0);
            sdotg += search[i] * g[i];
        }
        T step = T(1);
        T xc[MNU];
#pragma unroll
        for (int i = 0; i < MNU; ++i) xc[i] = i < n ? clampv(x[i] + step * search[i], lo[i], hi[i]) : T(0);
        T fc = qp_objective(n, Q, c, xc);
        while ((fc - old_f) / (step * sdotg) < armijo) {
            step *= step_dec;
            bool same = true, unchanged = true;
#pragma unroll
            for (int i = 0; i < MNU; ++i) {
                const T prev = xc[i];
                xc[i] = i < n ? clampv(x[i] + step * search[i], lo[i], hi[i]) : T(0);
                same = same && (xc[i] == x[i]);
                unchanged = unchanged && (xc[i] == prev);
            }
            // the candidate has rounded back onto x and stays there for every smaller step: the reference
            // shrinks the step down to min_step and leaves x unchanged with result 2 (see boxqp1)
            if (same) { fc = old_f; result = 2; break; }
            // a saturated Newton step (the direction is orders of magnitude longer than the box): every moving
            // dimension sits on its bound for many consecutive step sizes, the candidate -- and so its objective --
            // does not change, and only `step` in the Armijo ratio does.  Same iterations, same comparisons, without
            // re-evaluating the objective (the loop was 23 % of the rendezvous backward pass's instructions).
            if (!unchanged) fc = qp_objective(n, Q, c, xc);
            if (step < min_step) { result = 2; break; }
        }
#pragma unroll
        for (int i = 0; i < MNU; ++i) x[i] = xc[i];
        f = fc;
    }
    return result;
}

// The small dense part of one time step (team-uniform inputs): eigen-clipped regularised Q_uu, feed-forward term kt
// (unconstrained: -Q_uu_reg^-1 Q_u; bounded: box QP warm-started at k[t+1]) and M with K = -M Q_uz (the regularised
// inverse restricted to the free dimensions).  false where the reference raises (ilqr.py:636-640, 653-655).
template <class T>
__device__ __forceinline__ bool solve_small(int nu, bool bounded, const T (&Quu)[MNU][MNU], const T (&Qu)[MNU], T reg,
                                            const T (&lot)[MNU], const T (&hit)[MNU], const T (&k_next)[MNU],
                                            T (&kt)[MNU], T (&M)[MNU][MNU]) {
    T A[MNU][MNU], E[MNU][MNU], ev[MNU];
    bool finite = true, ok = true;
#pragma unroll
    for (int i = 0; i < MNU; ++i)
#pragma unroll
        for (int j = 0; j < MNU; ++j) {
            A[i][j] = Quu[i][j];
            finite = finite && isfinite(Quu[i][j]);
        }
    if (!finite) return false;                             // linalg.eig raises on NaN / Inf
    // (A Cholesky test for "Q_uu is already positive definite, skip the eigen-decomposition" was tried and
    // measured SLOWER on the rendezvous workload: 40.6 vs 30.5 ms.  With R = 0.1 I the symmetric problem's Q_uu is
    // diagonal up to rounding and the Jacobi loop exits before its first rotation, while the extra factorisation
    // costs square roots, divisions and registers.)
    jacobi_eig(nu, A, E, ev);
#pragma unroll
    for (int i = 0; i < MNU; ++i) {
        if (ev[i] < T(0)) ev[i] = T(1e-12);                // ref: ilqr.py:633-634
        ev[i] += reg;
    }
    if (!bounded) {
#pragma unroll
        for (int i = 0; i < MNU; ++i)
#pragma unroll
            for (int j = 0; j < MNU; ++j) {
                T sum = T(0);
#pragma unroll
                for (int m = 0; m < MNU; ++m)
                    if (m < nu) sum += (E[i][m] / ev[m]) * E[j][m];
                M[i][j] = (i < nu && j < nu) ? sum : T(0);
            }
#pragma unroll
        for (int i = 0; i < MNU; ++i) {
            T sum = T(0);
#pragma unroll
            for (int j = 0; j < MNU; ++j) sum += M[i][j] * Qu[j];
            kt[i] = -sum;
            if (kt[i] != kt[i]) ok = false;
        }
    } else {
        T Qreg[MNU][MNU], Uf[MNU][MNU];
#pragma unroll
        for (int i = 0; i < MNU; ++i)
#pragma unroll
            for (int j = 0; j < MNU; ++j) {
                T sum = T(0);
#pragma unroll
                for (int m = 0; m < MNU; ++m)
                    if (m < nu) sum += (E[i][m] * ev[m]) * E[j][m];
                Qreg[i][j] = sum;
            }
        unsigned free;
        const int result = boxqp_n(nu, k_next, Qreg, Qu, lot, hit, kt, free, Uf);
        if (result < 1) ok = false;                        // ref: ilqr.py:653-655
        // M = (Q_uu_reg[free, free])^-1 scattered back, zero rows / columns for the clamped dims
#pragma unroll
        for (int j = 0; j < MNU; ++j) {
            T r[MNU], x[MNU];
#pragma unroll
            for (int i = 0; i < MNU; ++i) r[i] = (i == j && ((free >> j) & 1u)) ? T(1) : T(0);
            chol_solve(Uf, r, x);
#pragma unroll
            for (int i = 0; i < MNU; ++i) M[i][j] = (((free >> i) & 1u) && ((free >> j) & 1u)) ? x[i] : T(0);
        }
    }
    return ok;
}

// shared memory per team: three nz x LD matrices, two LD vectors, four nu x LD matrices, 64 small values
// (Q_uu 16, Q_u 4 | hand-off results: kt 4, M 16, ok 1)
__host__ __device__ inline int backward_nu_elems(int nz, int nu) {
    const int LD = (nz + 3) & ~3;
    return 3 * nz * LD + 2 * LD + 4 * nu * LD + 64;
}
// stride between the teams of a CTA: == TEAM (mod 32) words, so that the 32 / TEAM teams of a warp, whose lanes read
// TEAM consecutive words (or one broadcast word) at the same offset of their own region, hit 32 different banks
// (an unpadded 368-word stride put the 8 teams of a warp on 2 bank groups: 73 % of the wavefronts were conflicts)
__host__ __device__ inline int backward_nu_stride(int nz, int nu, int team) {
    const int e = backward_nu_elems(nz, nu);
    return team >= 32 ? e : ((e + 31) & ~31) + team;
}

// NZC / NUC > 0: state / action sizes known at compile time (the loops unroll and the index divisions become shifts:
// with run-time sizes the matrix phases of the rendezvous problem were 9.6 k instructions per warp and time step).
//
// HO (hand-off, sub-warp teams): the small dense part is data dependent (Jacobi sweeps, box-QP iterations) and
// team-uniform, so a warp of 32 / TEAM teams would pay the union of its problems' paths once per 32 / TEAM problems:
// for the rendezvous shape 6.8 k of the 10 k instructions per warp and time step.  Instead every team parks Q_uu / Q_u
// in its shared-memory region and ONE warp of the CTA solves all of the CTA's problems, a problem per lane (the warm
// start k[t+1] stays in that lane's registers); the other warps wait at the CTA barrier (other CTAs of the SM run
// their matrix phases meanwhile).  Teams without work (b >= B, inactive, failed) keep taking part in the barriers.
template <class T, int TEAM, int NZC = 0, int NUC = 0>
__global__ void __launch_bounds__(TEAM <= 32 ? 128 : TEAM, (TEAM < 32 && sizeof(T) == 4) ? 4 : 1) backward_nu_kernel(const BackwardArgs<T> a) {
    constexpr bool HO = TEAM < 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x % TEAM, warp = threadIdx.x / TEAM, wpb = blockDim.x / TEAM;
    const int b = blockIdx.x * wpb + warp;
    const bool alive = b < a.B && !(a.active && a.active[b] == 0);
    if (!HO && !alive) return;
    const int nz = NZC > 0 ? NZC : a.nz, nu = NUC > 0 ? NUC : a.nu, nn = nz * nz, LD = (nz + 3) & ~3, nl = nz * LD;
    const int stride = backward_nu_stride(nz, nu, TEAM);
    T* base = reinterpret_cast<T*>(smem_raw) + (size_t)warp * stride;
    T *V = base, *Fz = base + nl, *W = base + 2 * nl;
    T *v = base + 3 * nl, *Qz = v + LD;
    T *FuT = Qz + LD, *WuT = FuT + nu * LD, *Quz = WuT + nu * LD, *Kt = Quz + nu * LD;   // [nu][LD], row = control dim
    T *sQuu = Kt + nu * LD, *sQu = sQuu + 16, *sKt = sQu + 4, *sM = sKt + 4, *sOk = sM + 16;
    const int small_off = (int)(sQuu - base);
    const bool bounded = a.u_min != nullptr && a.u_max != nullptr;
    const T reg = alive ? (T)a.mu[b] : T(0);
    T lo[MNU], hi[MNU], k_next[MNU];
#pragma unroll
    for (int i = 0; i < MNU; ++i) {
        lo[i] = bounded && i < nu ? a.u_min[i] : T(0);
        hi[i] = bounded && i < nu ? a.u_max[i] : T(0);
        k_next[i] = T(0);                                     // ref: ilqr.py:649 -- k[-1] is still zero at t = N-1
    }
    // hand-off: the problem this thread SOLVES (threads 0 .. wpb-1 of the CTA), its regularisation and warm start
    const int sb = blockIdx.x * wpb + (int)threadIdx.x;
    const bool solver = HO && (int)threadIdx.x < wpb;
    const bool s_alive = solver && sb < a.B && !(a.active && a.active[sb] == 0);
    const T s_reg = s_alive ? (T)a.mu[sb] : T(0);
    T* s_small = reinterpret_cast<T*>(smem_raw) + (size_t)(solver ? threadIdx.x : 0) * stride + small_off;
    if (alive) {
        for (int e = lane; e < nn; e += TEAM) V[(e / nz) * LD + e % nz] = a.L_zz[a.lLzz.at(b, a.N, e)];
        for (int e = lane; e < nz; e += TEAM) v[e] = a.L_z[a.lLz.at(b, a.N, e)];
    }
    if (HO && lane == 0) sOk[1] = alive ? T(1) : T(0);        // "this team has work at the next hand-off"
    nu_team_sync<TEAM>();
    bool ok = true;
    for (int t = a.N - 1; t >= 0; --t) {
        const bool work = alive && ok;                        // (without hand-off a team without work has left)
        if (work) {
            for (int e = lane; e < nn; e += TEAM) Fz[(e / nz) * LD + e % nz] = a.F_z[a.lFz.at(b, t, e)];
            for (int e = lane; e < nz * nu; e += TEAM) FuT[(e % nu) * LD + e / nu] = a.F_u[a.lFu.at(b, t, e)];
        }
        nu_team_sync<TEAM>();
        // W = V Fz ; WuT[i] = V Fu[:, i]
        if (work) {
            for (int e = lane; e < nn; e += TEAM) {
                const int i = e / nz, j = e - i * nz;
                T s = T(0);
                for (int kk = 0; kk < nz; ++kk) s += V[i * LD + kk] * Fz[kk * LD + j];
                W[i * LD + j] = s;
            }
            for (int e = lane; e < nz * nu; e += TEAM) {
                const int i = e / nz, r = e - i * nz;
                T s = T(0);
                for (int kk = 0; kk < nz; ++kk) s += V[r * LD + kk] * FuT[i * LD + kk];
                WuT[i * LD + r] = s;
            }
        }
        nu_team_sync<TEAM>();
        // Q_z, Q_uz, Q_u, Q_uu   (ref: ilqr.py:489-526)
        if (work) {
            for (int i = lane; i < nz; i += TEAM) {
                T sz = a.L_z[a.lLz.at(b, t, i)];
                for (int kk = 0; kk < nz; ++kk) sz += Fz[kk * LD + i] * v[kk];
                Qz[i] = sz;
            }
            for (int e = lane; e < nz * nu; e += TEAM) {
                const int i = e / nz, c = e - i * nz;
                T s = a.L_uz[a.lLuz.at(b, t, i * nz + c)];
                for (int kk = 0; kk < nz; ++kk) s += FuT[i * LD + kk] * W[kk * LD + c];
                Quz[i * LD + c] = s;
            }
            for (int e = lane; e < nu * nu + nu; e += TEAM) {
                if (e < nu * nu) {
                    const int i = e / nu, j = e - i * nu;
                    T s = a.L_uu[a.lLuu.at(b, t, e)];
                    for (int kk = 0; kk < nz; ++kk) s += FuT[i * LD + kk] * WuT[j * LD + kk];
                    sQuu[i * MNU + j] = s;
                } else {
                    const int i = e - nu * nu;
                    T s = a.L_u[a.lLu.at(b, t, i)];
                    for (int kk = 0; kk < nz; ++kk) s += FuT[i * LD + kk] * v[kk];
                    sQu[i] = s;
                }
            }
        }
        nu_team_sync<TEAM>();
        // Q_zz = L_zz + Fz^T W -> overwrites V (dead once W and WuT exist)
        if (work) {
            for (int e = lane; e < nn; e += TEAM) {
                const int i = e / nz, j = e - i * nz;
                T s = a.L_zz[a.lLzz.at(b, t, e)];
                for (int kk = 0; kk < nz; ++kk) s += Fz[kk * LD + i] * W[kk * LD + j];
                V[i * LD + j] = s;
            }
        }
        // ---- small dense part ----
        T Quu[MNU][MNU], Qu[MNU], kt[MNU], M[MNU][MNU];
        if (HO) {
            __syncthreads();                                   // every team's Q_uu / Q_u (and work flag) is parked
            if (solver && s_alive && s_small[41] != T(0)) {    // s_small: Q_uu 0..15, Q_u 16..19, kt 20..23, M 24..39, ok 40, work 41
                T sQ[MNU][MNU], sq[MNU], lot[MNU], hit[MNU], skt[MNU], sMm[MNU][MNU];
#pragma unroll
                for (int i = 0; i < MNU; ++i) {
                    sq[i] = i < nu ? s_small[16 + i] : T(0);
                    const T ut = (bounded && i < nu) ? a.U[a.lU.at(sb, t, i)] : T(0);
                    lot[i] = lo[i] - ut;
                    hit[i] = hi[i] - ut;
#pragma unroll
                    for (int j = 0; j < MNU; ++j)
                        sQ[i][j] = (i < nu && j < nu) ? T(0.5) * (s_small[i * MNU + j] + s_small[j * MNU + i]) : T(0);
                }
                const bool sok = solve_small(nu, bounded, sQ, sq, s_reg, lot, hit, k_next, skt, sMm);
#pragma unroll
                for (int i = 0; i < MNU; ++i) {
                    k_next[i] = skt[i];
                    s_small[20 + i] = skt[i];
#pragma unroll
                    for (int j = 0; j < MNU; ++j) s_small[24 + i * MNU + j] = sMm[i][j];
                }
                s_small[40] = sok ? T(1) : T(0);
            }
            __syncthreads();
            if (work) {
#pragma unroll
                for (int i = 0; i < MNU; ++i) {
                    Qu[i] = i < nu ? sQu[i] : T(0);
                    kt[i] = sKt[i];
#pragma unroll
                    for (int j = 0; j < MNU; ++j) {
                        Quu[i][j] = (i < nu && j < nu) ? T(0.5) * (sQuu[i * MNU + j] + sQuu[j * MNU + i]) : T(0);
                        M[i][j] = sM[i * MNU + j];
                    }
                }
                ok = sOk[0] != T(0);
            }
        } else {
            T lot[MNU], hit[MNU];
#pragma unroll
            for (int i = 0; i < MNU; ++i) {
                Qu[i] = i < nu ? sQu[i] : T(0);
                const T ut = (bounded && i < nu) ? a.U[a.lU.at(b, t, i)] : T(0);
                lot[i] = lo[i] - ut;
                hit[i] = hi[i] - ut;
#pragma unroll
                for (int j = 0; j < MNU; ++j)
                    Quu[i][j] = (i < nu && j < nu) ? T(0.5) * (sQuu[i * MNU + j] + sQuu[j * MNU + i]) : T(0);
            }
            ok = solve_small(nu, bounded, Quu, Qu, reg, lot, hit, k_next, kt, M);
#pragma unroll
            for (int i = 0; i < MNU; ++i) k_next[i] = kt[i];
            if (!ok) break;
        }
        const bool work2 = work && ok;
        bool bad = false;
        if (work2) {
            for (int e = lane; e < nz * nu; e += TEAM) {
                const int i = e / nz, c = e - i * nz;
                T s = T(0);
#pragma unroll
                for (int j = 0; j < MNU; ++j)
                    if (j < nu) s += M[i][j] * Quz[j * LD + c];      // M[i][j] indexed with a runtime i: small local array
                s = -s;
                Kt[i * LD + c] = s;
                bad |= (s != s);
            }
        }
        if (HO) {
            if (work2) ok = !(__any_sync(nu_team_mask<TEAM>(), bad && !bounded));
        } else {
            ok = ok && !nu_team_any<TEAM>(bad && !bounded);    // the NaN test is on the unconstrained branch only
            if (!ok) break;
        }
        if (HO && lane == 0) sOk[1] = (alive && ok) ? T(1) : T(0);   // work flag for the next hand-off
        nu_team_sync<TEAM>();
        if (alive && ok && work) {
            for (int l = lane; l < nu; l += TEAM) {
                T kv = T(0);
#pragma unroll
                for (int i = 0; i < MNU; ++i) if (i == l) kv = kt[i];
                a.k[a.lk.at(b, t, l)] = kv;
            }
            for (int e = lane; e < nz * nu; e += TEAM) {
                const int i = e / nz, c = e - i * nz;
                a.K[a.lK.at(b, t, i * nz + c)] = Kt[i * LD + c];
            }
            // value update with the UN-regularised Q_uu (ref: ilqr.py:664-672)
            T Quuk[MNU];                                           // Q_uu k
#pragma unroll
            for (int i = 0; i < MNU; ++i) {
                T s = T(0);
#pragma unroll
                for (int j = 0; j < MNU; ++j) s += Quu[i][j] * kt[j];
                Quuk[i] = s;
            }
            for (int c = lane; c < nz; c += TEAM) {
                T s = Qz[c];
#pragma unroll
                for (int i = 0; i < MNU; ++i)
                    if (i < nu) s += Kt[i * LD + c] * (Qu[i] + Quuk[i]) + Quz[i * LD + c] * kt[i];
                v[c] = s;
            }
        }
        nu_team_sync<TEAM>();                                  // V (= Q_zz) complete before it is symmetrised
        if (alive && ok && work) {
            for (int e = lane; e < nn; e += TEAM) {
                const int i = e / nz, j = e - i * nz;
                if (j < i) continue;
                T val = T(0.5) * (V[i * LD + j] + V[j * LD + i]);
                T kqk = T(0), cross = T(0);
#pragma unroll
                for (int p = 0; p < MNU; ++p) {
                    if (p >= nu) continue;
                    T qk = T(0);                                   // (Q_uu K)[p][j]
#pragma unroll
                    for (int q = 0; q < MNU; ++q)
                        if (q < nu) qk += Quu[p][q] * Kt[q * LD + j];
                    kqk += Kt[p * LD + i] * qk;
                    cross += Kt[p * LD + i] * Quz[p * LD + j] + Quz[p * LD + i] * Kt[p * LD + j];
                }
                // 0.5 (X + X^T) of X = K^T Q_uu K + K^T Q_uz + Q_uz^T K: the first term is symmetric because the
                // symmetrised Q_uu is, the other two are each other's transpose
                val += kqk + cross;
                V[i * LD + j] = val;
                V[j * LD + i] = val;
            }
        }
        nu_team_sync<TEAM>();
    }
    if (lane == 0 && alive) a.status[b] = ok ? 0 : 1;
}

template <class T, int TEAM, int NZC = 0, int NUC = 0>
static cudaError_t launch_nu_teams(const BackwardArgs<T>& a, cudaStream_t s) {
    const size_t per_team = (size_t)backward_nu_stride(a.nz, a.nu, TEAM) * sizeof(T);
    int tpb = 128 / TEAM;                                   // teams (problems) per CTA
    while (tpb > 1 && per_team * tpb > 200 * 1024) tpb >>= 1;
    const size_t smem = per_team * tpb;
    auto kern = backward_nu_kernel<T, TEAM, NZC, NUC>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<(a.B + tpb - 1) / tpb, tpb * TEAM, smem, s>>>(a);
    return cudaGetLastError();
}

template <class T>
cudaError_t backward_pass_nu(const BackwardArgs<T>& a, cudaStream_t s) {
    if (a.nu < 1 || a.nu > MNU) return cudaErrorInvalidValue;
    const size_t per_team = (size_t)backward_nu_elems(a.nz, a.nu) * sizeof(T);
    if (a.nz >= 24) {
        if (per_team > 227 * 1024) return cudaErrorInvalidValue;
        cudaError_t e = cudaFuncSetAttribute(backward_nu_kernel<T, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)per_team);
        if (e != cudaSuccess) return e;
        backward_nu_kernel<T, 256><<<a.B, 256, per_team, s>>>(a);
        return cudaGetLastError();
    }
    // small states: sub-warp teams (nz <= 8: 4 lanes, 8 problems per warp; nz <= 12: 8 lanes), else a warp per problem
    if (a.nz == 8 && a.nu == 4) return launch_nu_teams<T, 4, 8, 4>(a, s);    // rendezvous, IGNORE_UNCERTAINTY
    if (a.nz <= 8) return launch_nu_teams<T, 4>(a, s);
    if (a.nz <= 12) return launch_nu_teams<T, 8>(a, s);
    return launch_nu_teams<T, 32>(a, s);
}
template cudaError_t backward_pass_nu<float>(const BackwardArgs<float>&, cudaStream_t);
template cudaError_t backward_pass_nu<double>(const BackwardArgs<double>&, cudaStream_t);

}  // namespace pddp
