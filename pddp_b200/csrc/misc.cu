// Per-problem controller state machine (accept / reject / regularisation schedule) and the
// stand-alone cost linearisation used by the BNN path.
#include "core.cuh"
#include "kernels.h"

namespace pddp {

// ref: pddp/controllers/ilqr.py:364-390 (Tassa schedule, python floats -> doubles here)
__device__ __forceinline__ bool increase_reg(double& mu, double& delta, double max_reg) {
    delta = fmax(1.0, delta) * 2.0;
    mu = fmax(1e-6, mu * delta);
    return mu < max_reg;
}
__device__ __forceinline__ void decrease_reg(double& mu, double& delta) {
    delta = fmin(1.0, delta) / 2.0;
    mu *= delta;
    if (mu <= 1e-6) mu = 0.0;
}

// ref: pddp/controllers/ilqr.py:140-181 (tail of _step), one thread per problem.
// active[b]: 0 finished, 1 needs a fresh linearisation, 2 retry backward+rollout on the old one.
template <class T>
__global__ void accept_state_kernel(const AcceptArgs<T> a, int32_t* accepted) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    accepted[b] = 0;
    if (a.active[b] == 0) return;
    double mu = a.mu[b], delta = a.delta[b];
    int state;
    if (a.bw_status && a.bw_status[b] != 0) {
        state = increase_reg(mu, delta, a.max_reg) ? ST_NOT_PD : ST_MAX_REG;
    } else {
        const T Jn = a.J_new[b], Jo = a.J_opt[b];
        if (Jn < Jo) {
            accepted[b] = 1;
            decrease_reg(mu, delta);
            T change = fabs(Jo - Jn) / Jo;
            state = change < (T)a.tol ? ST_CONVERGED : ST_ACCEPTED;
            a.J_opt[b] = Jn;
        } else {
            state = increase_reg(mu, delta, a.max_reg) ? ST_REJECTED : ST_MAX_REG;
        }
    }
    a.mu[b] = mu;
    a.delta[b] = delta;
    a.state[b] = state;
    int act;
    if (state == ST_CONVERGED || state == ST_MAX_REG) act = 0;
    else if (state == ST_ACCEPTED) {
        int left = a.iters_left[b] - 1;
        a.iters_left[b] = left;
        act = left > 0 ? 1 : 0;
    } else act = 2;
    a.active[b] = act;
    if (act != 0 && a.n_active) atomicAdd(a.n_active, 1);
}

// copy the accepted candidates into the nominal trajectory (self._Z_nominal/_U_nominal)
template <class T>
__global__ void accept_copy_kernel(const AcceptArgs<T> a, const int32_t* accepted) {
    const int64_t nK = a.K_nominal ? (int64_t)a.N * a.nu * a.nz : 0;
    const int64_t per = (int64_t)(a.N + 1) * a.nz + (int64_t)a.N * a.nu + nK;
    const int64_t total = per * a.B;
    for (int64_t id = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; id < total;
         id += (int64_t)gridDim.x * blockDim.x) {
        // id enumerates (slot, b) with b fastest for BATCH_INNER-friendly coalescing; for
        // PROBLEM_MAJOR the layout strides make consecutive slots contiguous instead.
        int64_t b, slot;
        if (a.lZ.sb == 1) { b = id % a.B; slot = id / a.B; }
        else { b = id / per; slot = id % per; }
        if (!accepted[b]) continue;
        if (slot < (int64_t)(a.N + 1) * a.nz) {
            int64_t t = slot / a.nz, e = slot % a.nz;
            a.Z[a.lZ.at(b, t, e)] = a.Z_new[a.lZ.at(b, t, e)];
        } else if ((slot -= (int64_t)(a.N + 1) * a.nz) < (int64_t)a.N * a.nu) {
            int64_t t = slot / a.nu, e = slot % a.nu;
            a.U[a.lU.at(b, t, e)] = a.U_new[a.lU.at(b, t, e)];
        } else {
            slot -= (int64_t)a.N * a.nu;
            const int64_t E = (int64_t)a.nu * a.nz, t = slot / E, e = slot % E;
            a.K_nominal[a.lK.at(b, t, e)] = a.K[a.lK.at(b, t, e)];
        }
    }
}

// BATCH_INNER: Z, U and K are flat [row][B] arrays (row = t * E + e), so the copy is three masked row copies.  A thread
// owns ONE problem (a warp's accesses are one coalesced line whatever the acceptance mask looks like) and walks the rows
// with a stride of gridDim.y, 8 rows in flight: no index arithmetic per element (the generic kernel's 64-bit divisions
// made it instruction bound: 2.0 TB/s at 2^20 pendulums).
template <class T>
__global__ void __launch_bounds__(256) accept_copy_inner_kernel(const AcceptArgs<T> a, const int32_t* accepted) {
    const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (b >= a.B || !accepted[b]) return;
    const int64_t rowsZ = (int64_t)(a.N + 1) * a.nz, rowsU = (int64_t)a.N * a.nu;
    const int64_t rowsK = a.K_nominal ? (int64_t)a.N * a.nu * a.nz : 0;
    constexpr int UR = 8;
    auto copy_rows = [&](const T* src, T* dst, int64_t nrows) {
        for (int64_t r0 = (int64_t)blockIdx.y * UR; r0 < nrows; r0 += (int64_t)gridDim.y * UR) {
            T tmp[UR];
#pragma unroll
            for (int u = 0; u < UR; ++u)
                if (r0 + u < nrows) tmp[u] = __ldg(src + (r0 + u) * a.B + b);
#pragma unroll
            for (int u = 0; u < UR; ++u)
                if (r0 + u < nrows) dst[(r0 + u) * a.B + b] = tmp[u];
        }
    };
    copy_rows(a.Z_new, a.Z, rowsZ);
    copy_rows(a.U_new, a.U, rowsU);
    if (rowsK) copy_rows(a.K, a.K_nominal, rowsK);
}

template <class T>
cudaError_t accept_update(const AcceptArgs<T>& a, int32_t* accepted_scratch, cudaStream_t s) {
    accept_state_kernel<T><<<(a.B + 127) / 128, 128, 0, s>>>(a, accepted_scratch);
    if (a.lZ.sb == 1) {                                     // BATCH_INNER
        const int64_t rows = (int64_t)(a.N + 1) * a.nz + (int64_t)a.N * a.nu + (a.K_nominal ? (int64_t)a.N * a.nu * a.nz : 0);
        const unsigned gx = (unsigned)(((int64_t)a.B + 255) / 256);
        int64_t gy = (148 * 16 + gx - 1) / gx;              // ~16 CTAs per SM in flight, each thread several rows
        if (gy > (rows + 7) / 8) gy = (rows + 7) / 8;
        if (gy > 65535) gy = 65535;
        if (gy < 1) gy = 1;
        accept_copy_inner_kernel<T><<<dim3(gx, (unsigned)gy), 256, 0, s>>>(a, accepted_scratch);
        return cudaGetLastError();
    }
    const int64_t total = ((int64_t)(a.N + 1) * a.nz + (int64_t)a.N * a.nu +
                           (a.K_nominal ? (int64_t)a.N * a.nu * a.nz : 0)) * a.B;
    int grid = (int)((total + 255) / 256);
    if (grid > 148 * 16) grid = 148 * 16;
    accept_copy_kernel<T><<<grid, 256, 0, s>>>(a, accepted_scratch);
    return cudaGetLastError();
}
template cudaError_t accept_update<float>(const AcceptArgs<float>&, int32_t*, cudaStream_t);
template cudaError_t accept_update<double>(const AcceptArgs<double>&, int32_t*, cudaStream_t);

// ------------------------------------------------------------------------------------------
// Stand-alone cost linearisation: one thread per (problem, time, Hessian pair).
// Replaces batch_eval_cost (pddp/utils/evaluation.py:134-239) for a whole nominal trajectory.
// ------------------------------------------------------------------------------------------
// Pair order for FULL_COVARIANCE_MATRIX: the cost is LINEAR in most covariance entries (trace term and the
// cross blocks of the augmented covariance, core.cuh cost_state), so most of the nz(nz+1)/2 Hessian pairs
// are structurally zero.  c_pair_order lists the pairs that can be non-zero first -- every diagonal pair
// (it also carries the gradient), pairs inside {means, C[ang][ang]}, and C[ang_i][*] / C[*][ang_i] against
// {m_ang_i, C[ang_i][ang_i]} -- then the rest, which only get zeros written (double cartpole: 119 of 903
// pairs are evaluated).  Entry = i * 256 + j.
// __constant__ memory is PER DEVICE: the table is uploaded once per (device, geometry), the pair count is
// device independent.
__constant__ uint16_t c_pair_order[3][1024];
static int g_pair_nnz[3] = {-1, -1, -1};
static bool g_pair_uploaded[64][3] = {};

template <int GEO>
static cudaError_t fill_pair_order(int* nnz_out) {
    typedef Geo<GEO> G;
    constexpr int D = G::D, NZ = D + D * D;
    int dev = 0;
    cudaError_t de = cudaGetDevice(&dev);
    if (de != cudaSuccess) return de;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (g_pair_uploaded[dev][GEO]) { *nnz_out = g_pair_nnz[GEO]; return cudaSuccess; }
    auto is_ang = [](int a) { for (int i = 0; i < G::NANG; ++i) if (G::ang(i) == a) return true; return false; };
    // class of a variable: 0 mean, 1 C[ang][ang], 2 C with exactly one angular index, 3 C[nonang][nonang]
    auto cls = [&](int v, int& angle) {
        angle = -1;
        if (v < D) { if (is_ang(v)) angle = v; return 0; }
        const int a = (v - D) / D, b = (v - D) % D;
        if (is_ang(a) && is_ang(b)) { if (a == b) angle = a; return 1; }
        if (is_ang(a) || is_ang(b)) { angle = is_ang(a) ? a : b; return 2; }
        return 3;
    };
    uint16_t order[1024];
    int n = 0;
    for (int pass = 0; pass < 2; ++pass)
        for (int i = 0; i < NZ; ++i)
            for (int j = i; j < NZ; ++j) {
                int ai, aj;
                const int ci = cls(i, ai), cj = cls(j, aj);
                bool nonzero = i == j || (ci <= 1 && cj <= 1);
                if (ci == 2 && cj <= 1 && aj == ai) nonzero = true;      // C[ang_i][.] x {m_ang_i, C[ang_i][ang_i]}
                if (cj == 2 && ci <= 1 && ai == aj) nonzero = true;
                if ((pass == 0) == nonzero) order[n++] = (uint16_t)(i * 256 + j);
                if (pass == 0 && i == NZ - 1 && j == NZ - 1) g_pair_nnz[GEO] = n;
            }
    cudaError_t e = cudaMemcpyToSymbol(c_pair_order, order, sizeof(uint16_t) * n, sizeof(uint16_t) * 1024 * GEO);
    if (e != cudaSuccess) return e;
    g_pair_uploaded[dev][GEO] = true;
    *nnz_out = g_pair_nnz[GEO];
    return cudaSuccess;
}

// zero L_zz (and L_uz) of every active site with coalesced stores; the structurally non-zero pairs are
// then written by cost_pairs_kernel (FULL_COVARIANCE_MATRIX only)
template <class T>
__global__ void __launch_bounds__(256) cost_zero_kernel(const CostDerivArgs<T> a, int NZ) {
    const int64_t site = blockIdx.x;
    const int b = (int)(site / (a.N + 1)), t = (int)(site - (int64_t)b * (a.N + 1));
    if (a.active && a.active[b] != 1) return;
    for (int e = threadIdx.x; e < NZ * NZ; e += blockDim.x) a.L_zz[a.lLzz.at(b, t, e)] = T(0);
    if (a.L_uz && t < a.N)
        for (int e = threadIdx.x; e < NZ; e += blockDim.x) a.L_uz[a.lLuz.at(b, t, e)] = T(0);
}

template <class T, int GEO, int ENC>
__global__ void __launch_bounds__(128) cost_pairs_kernel(const CostDerivArgs<T> a, int nnz) {
    typedef Geo<GEO> G;
    constexpr int D = G::D, NZ = enc_size(D, ENC);
    const int NP = ENC == ENC_FULL ? nnz : NZ * (NZ + 1) / 2;      // threads per site
    const int64_t id = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t site = id / NP;
    if (site >= (int64_t)a.B * (a.N + 1)) return;
    int p = (int)(id - site * NP);
    const int b = (int)(site / (a.N + 1)), t = (int)(site - (int64_t)b * (a.N + 1));
    if (a.active && a.active[b] != 1) return;
    int i = 0, j;
    const bool terminal = t == a.N;
    if (ENC == ENC_FULL) {
        const int e = c_pair_order[GEO][p];
        i = e >> 8;
        j = e & 255;
    } else {
        while (p >= NZ - i) { p -= NZ - i; ++i; }
        j = i + p;
    }
    const auto goal = site_goal<GEO>(a.cost, b, t, terminal);
    typedef Jet2<T, 2> S;
    S zj[NZ];
#pragma unroll
    for (int k = 0; k < NZ; ++k) {
        zj[k] = S(a.Z[a.lZ.at(b, t, k)]);
        zj[k].g[0] = k == i ? T(1) : T(0);
        zj[k].g[1] = k == j ? T(1) : T(0);
    }
    S r = cost_state<GEO, ENC, T, S>(a.cost, goal.x, zj, terminal);
    a.L_zz[a.lLzz.at(b, t, i * NZ + j)] = r.h[1];
    if (i != j) a.L_zz[a.lLzz.at(b, t, j * NZ + i)] = r.h[1];
    else a.L_z[a.lLz.at(b, t, i)] = r.g[0];
    if (ENC != ENC_FULL && i == 0) a.L_uz && !terminal ? (void)(a.L_uz[a.lLuz.at(b, t, j)] = T(0)) : (void)0;
    if (i == 0 && j == 0) {
        T l = r.v;
        if (!terminal) {
            T la, lu, luu;
            cost_action(a.cost, goal.u[0], a.U[a.lU.at(b, t, 0)], la, lu, luu);
            l += la;
            a.L_u[a.lLu.at(b, t, 0)] = lu;
            a.L_uu[a.lLuu.at(b, t, 0)] = luu;
        }
        a.L[a.lL.at(b, t, 0)] = l;
    }
}

template <class T>
__global__ void cost_sum_kernel(const CostDerivArgs<T> a) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    if (a.active && a.active[b] != 1) return;
    T J = T(0);
    for (int t = 0; t <= a.N; ++t) J += a.L[a.lL.at(b, t, 0)];
    a.J_opt[b] = J;
}

template <class T, int GEO, int ENC>
static cudaError_t launch_cost(const CostDerivArgs<T>& a, cudaStream_t s) {
    constexpr int NZ = enc_size(Geo<GEO>::D, ENC), NP = NZ * (NZ + 1) / 2;
    int nnz = NP;
    if (ENC == ENC_FULL) {
        cudaError_t e = fill_pair_order<GEO>(&nnz);
        if (e != cudaSuccess) return e;
        cost_zero_kernel<T><<<(unsigned)((int64_t)a.B * (a.N + 1)), 256, 0, s>>>(a, NZ);
    }
    const int64_t total = (int64_t)a.B * (a.N + 1) * nnz;
    cost_pairs_kernel<T, GEO, ENC><<<(unsigned)((total + 127) / 128), 128, 0, s>>>(a, nnz);
    if (a.J_opt) cost_sum_kernel<T><<<(a.B + 127) / 128, 128, 0, s>>>(a);
    return cudaGetLastError();
}

template <class T>
cudaError_t cost_derivatives(int geo, int enc, const CostDerivArgs<T>& a, cudaStream_t s) {
    switch (geo * 8 + enc) {
        case GEO_PENDULUM * 8 + ENC_FULL: return launch_cost<T, GEO_PENDULUM, ENC_FULL>(a, s);
        case GEO_PENDULUM * 8 + ENC_UT: return launch_cost<T, GEO_PENDULUM, ENC_UT>(a, s);
        case GEO_PENDULUM * 8 + ENC_IGNORE: return launch_cost<T, GEO_PENDULUM, ENC_IGNORE>(a, s);
        case GEO_PENDULUM * 8 + ENC_VAR: return launch_cost<T, GEO_PENDULUM, ENC_VAR>(a, s);
        case GEO_PENDULUM * 8 + ENC_STD: return launch_cost<T, GEO_PENDULUM, ENC_STD>(a, s);
        case GEO_CARTPOLE * 8 + ENC_VAR: return launch_cost<T, GEO_CARTPOLE, ENC_VAR>(a, s);
        case GEO_CARTPOLE * 8 + ENC_STD: return launch_cost<T, GEO_CARTPOLE, ENC_STD>(a, s);
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_VAR: return launch_cost<T, GEO_DOUBLE_CARTPOLE, ENC_VAR>(a, s);
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_STD: return launch_cost<T, GEO_DOUBLE_CARTPOLE, ENC_STD>(a, s);
        case GEO_CARTPOLE * 8 + ENC_FULL: return launch_cost<T, GEO_CARTPOLE, ENC_FULL>(a, s);
        case GEO_CARTPOLE * 8 + ENC_UT: return launch_cost<T, GEO_CARTPOLE, ENC_UT>(a, s);
        case GEO_CARTPOLE * 8 + ENC_IGNORE: return launch_cost<T, GEO_CARTPOLE, ENC_IGNORE>(a, s);
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_FULL: return launch_cost<T, GEO_DOUBLE_CARTPOLE, ENC_FULL>(a, s);
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_UT: return launch_cost<T, GEO_DOUBLE_CARTPOLE, ENC_UT>(a, s);
        case GEO_DOUBLE_CARTPOLE * 8 + ENC_IGNORE: return launch_cost<T, GEO_DOUBLE_CARTPOLE, ENC_IGNORE>(a, s);
        default: return cudaErrorInvalidValue;
    }
}
template cudaError_t cost_derivatives<float>(int, int, const CostDerivArgs<float>&, cudaStream_t);
template cudaError_t cost_derivatives<double>(int, int, const CostDerivArgs<double>&, cudaStream_t);

}  // namespace pddp
