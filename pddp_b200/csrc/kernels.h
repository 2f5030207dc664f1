// Internal (C++) launch interfaces between capi.cu and the kernel translation units.
#pragma once
#include "../../include/pddp_b200.h"
#include "core.cuh"

namespace pddp {

template <class T>
struct LinKnownArgs {
    int B, N;
    CostParams<T> cost;
    KnownParams<T> dyn;
    const T* z0; const T* U; const T* u_min; const T* u_max; const int32_t* active;
    T* Z; T* F_z; T* F_u; T* L; T* L_z; T* L_u; T* L_zz; T* L_uz; T* L_uu; T* J_opt;
    T* U_clamped;   // scratch [B,N,nu] (same layout as U) for the separate cost pass, or NULL
    int32_t* status;
    Layout lZ, lU, lFz, lFu, lL, lLz, lLu, lLzz, lLuz, lLuu;
    const T* p_b;   // [B, 8] per-problem dynamics parameters, or NULL: dyn (pddp_known_dynamics::p_b)
};

template <class T>
struct RollKnownArgs {
    int B, N, A;
    CostParams<T> cost;
    KnownParams<T> dyn;
    const T* Z; const T* U; const T* k; const T* K; const T* alphas; const T* u_min; const T* u_max;
    const int32_t* active; const int32_t* bw_status;
    T* J_all; int32_t* amin; T* J_new; T* Z_new; T* U_new;
    Layout lZ, lU, lk, lK;
    const T* p_b;   // [B, 8] per-problem dynamics parameters, or NULL: dyn
};

template <class T>
struct BackwardArgs {
    int B, N, nz, nu;
    const T* F_z; const T* F_u; const T* L_z; const T* L_u; const T* L_zz; const T* L_uz; const T* L_uu;
    const double* mu; const T* U; const T* u_min; const T* u_max; const int32_t* active;
    T* k; T* K; int32_t* status;
    Layout lFz, lFu, lLz, lLu, lLzz, lLuz, lLuu, lU, lk, lK;
};

template <class T>
struct AcceptArgs {
    int B, N, nz, nu;
    const T* J_new; const int32_t* bw_status; const T* Z_new; const T* U_new;
    double tol, max_reg;
    double* mu; double* delta; T* J_opt; int32_t* state; int32_t* iters_left; int32_t* active;
    T* Z; T* U; int32_t* n_active;
    const T* K; T* K_nominal;      // optional: gains kept only for accepted steps (ilqr.py:166-171)
    Layout lZ, lU, lK;
};

template <class T>
struct CostDerivArgs {
    int B, N;
    CostParams<T> cost;
    const T* Z; const T* U; const int32_t* active;
    T* L; T* L_z; T* L_u; T* L_zz; T* L_uz; T* L_uu; T* J_opt;
    Layout lZ, lU, lL, lLz, lLu, lLzz, lLuz, lLuu;
};

// pddp_cost (host, doubles) -> the kernels' CostParams, with the per-step goals' layouts from the shape (capi.cu)
template <class T> void fill_cost(const pddp_cost* c, const pddp_shape* s, CostParams<T>& out);

template <class T> cudaError_t linearize_known(int geo, int enc, const LinKnownArgs<T>&, cudaStream_t);
template <class T> cudaError_t rollout_known(int geo, int enc, const RollKnownArgs<T>&, cudaStream_t);
// p_b: [B, 8] parameters of every instance, or NULL: the shared ones
template <class T> cudaError_t env_step_known(int geo, int B, const KnownParams<T>&, const T* p_b, const T* x, const T* u, T* xn,
                                              cudaStream_t);
template <class T> cudaError_t env_step_lq(int B, const KnownParams<T>&, const T* p_b, const T* x, const T* u, T* xn, cudaStream_t);
template <class T> cudaError_t linearize_lq(int enc, const LinKnownArgs<T>&, cudaStream_t);      // known_lq.cu (rendezvous)
template <class T> cudaError_t rollout_lq(int enc, const RollKnownArgs<T>&, cudaStream_t);
template <class T> cudaError_t cost_derivatives_lq(int enc, const CostDerivArgs<T>&, cudaStream_t);
template <class T> cudaError_t backward_pass(const BackwardArgs<T>&, int layout, cudaStream_t);
template <class T> cudaError_t backward_pass_nu(const BackwardArgs<T>&, cudaStream_t);      // backward_nu.cu, nu <= MAX_NU
template <class T> cudaError_t accept_update(const AcceptArgs<T>&, int32_t* accepted_scratch, cudaStream_t);
template <class T> cudaError_t cost_derivatives(int geo, int enc, const CostDerivArgs<T>&, cudaStream_t);

}  // namespace pddp
