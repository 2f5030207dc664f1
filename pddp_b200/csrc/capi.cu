// extern "C" entry points (declared in include/pddp_b200.h): argument checking, host-side
// conversion of the by-value parameter structs, dtype dispatch.  No allocation, no synchronisation.
#include "../../include/pddp_b200.h"
#include "kernels.h"
#include "profile.h"
#include <stdio.h>
#include <string.h>

using namespace pddp;

static thread_local char g_err[256] = "";

static int fail(int code, const char* msg) {
    snprintf(g_err, sizeof(g_err), "%s", msg);
    return code;
}
static int cuda_result(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return 0;
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return (int)e;
}

static int geo_D(int geo) { return geo == GEO_PENDULUM ? 2 : geo == GEO_CARTPOLE ? 4 : geo == GEO_DOUBLE_CARTPOLE ? 6 : geo == GEO_RENDEZVOUS ? 8 : -1; }
static int geo_DA(int geo) { return geo == GEO_PENDULUM ? 3 : geo == GEO_CARTPOLE ? 5 : 8; }
static int geo_nu(int geo) { return geo == GEO_RENDEZVOUS ? 4 : 1; }

static int check_shape(const pddp_shape* s) {
    if (!s) return fail(PDDP_E_BADARG, "shape is NULL");
    if (s->dtype != PDDP_F32 && s->dtype != PDDP_F64) return fail(PDDP_E_BADARG, "dtype must be PDDP_F32 or PDDP_F64");
    if (s->layout != PDDP_PROBLEM_MAJOR && s->layout != PDDP_BATCH_INNER) return fail(PDDP_E_BADARG, "bad layout");
    if (geo_D(s->geo) < 0) return fail(PDDP_E_UNSUPPORTED, "unsupported geometry (pendulum, cartpole, double_cartpole, rendezvous)");
    if (s->enc < 0 || s->enc > 4) return fail(PDDP_E_BADARG, "bad encoding");
    if (s->nu != geo_nu(s->geo)) return fail(PDDP_E_BADARG, "nu does not match the geometry's action size");
    if (s->nz != enc_size(geo_D(s->geo), s->enc)) return fail(PDDP_E_BADARG, "nz does not match the encoding size of this geometry");
    if (s->B < 1 || s->N < 1) return fail(PDDP_E_BADARG, "B and N must be positive");
    return 0;
}

// a goal comes from one source: per problem ([B, .]) or per problem and step ([B, Nt, .]), not both
static int check_cost(const pddp_cost* c) {
    if (c->x_goal_b && c->x_goal_bt) return fail(PDDP_E_BADARG, "pddp_cost: x_goal_b and x_goal_bt are exclusive");
    if (c->u_goal_b && c->u_goal_bt) return fail(PDDP_E_BADARG, "pddp_cost: u_goal_b and u_goal_bt are exclusive");
    return 0;
}

template <class T>
void pddp::fill_cost(const pddp_cost* c, const pddp_shape* s, CostParams<T>& out) {
    const int DA = geo_DA(s->geo);
    memset(&out, 0, sizeof(out));
    for (int i = 0; i < DA * DA; ++i) { out.Q[i] = (T)c->Q[i]; out.Qt[i] = (T)c->Q_term[i]; }
    for (int i = 0; i < DA; ++i) out.xg[i] = (T)c->x_goal[i];
    for (int i = 0; i < MAX_NU * MAX_NU; ++i) out.R[i] = (T)c->R[i];
    for (int i = 0; i < MAX_NU; ++i) out.ug[i] = (T)c->u_goal[i];
    out.xg_b = (const T*)c->x_goal_b;
    out.ug_b = (const T*)c->u_goal_b;
    out.xg_bt = (const T*)c->x_goal_bt;
    out.ug_bt = (const T*)c->u_goal_bt;
    out.lXg = make_layout(s->layout, s->B, (int64_t)s->N + 1, DA);
    out.lUg = make_layout(s->layout, s->B, s->N, s->nu);
}
template void pddp::fill_cost<float>(const pddp_cost*, const pddp_shape*, CostParams<float>&);
template void pddp::fill_cost<double>(const pddp_cost*, const pddp_shape*, CostParams<double>&);

// pddp_backward only sees derivative tensors: no geometry / encoding constraints
static int check_shape_backward(const pddp_shape* s) {
    if (!s) return fail(PDDP_E_BADARG, "shape is NULL");
    if (s->dtype != PDDP_F32 && s->dtype != PDDP_F64) return fail(PDDP_E_BADARG, "dtype must be PDDP_F32 or PDDP_F64");
    if (s->layout != PDDP_PROBLEM_MAJOR && s->layout != PDDP_BATCH_INNER) return fail(PDDP_E_BADARG, "bad layout");
    if (s->nu < 1 || s->nu > PDDP_MAX_NU) return fail(PDDP_E_UNSUPPORTED, "pddp_backward: 1 <= action_size <= PDDP_MAX_NU");
    if (s->nz < 1 || s->nz > 96) return fail(PDDP_E_UNSUPPORTED, "pddp_backward: 1 <= nz <= 96");
    if (s->B < 1 || s->N < 1) return fail(PDDP_E_BADARG, "B and N must be positive");
    return 0;
}

int pddp_capi_fail(int code, const char* msg) { return fail(code, msg); }
int pddp_capi_cuda(cudaError_t e, const char* what) { return cuda_result(e, what); }
int pddp_capi_check_shape(const pddp_shape* s) { return check_shape(s); }
int pddp_capi_check_cost(const pddp_cost* c) { return check_cost(c); }

extern "C" const char* pddp_version(void) { return "pddp_b200 0.2 (sm_100a)"; }
extern "C" const char* pddp_last_error(void) { return g_err; }

// ---------------------------------------------------------------------------------------------
template <class T>
static int linearize_known_t(const pddp_shape* s, const pddp_known_dynamics* dyn, const pddp_cost* cost,
                             const void* z0, const void* U, const void* u_min, const void* u_max,
                             const int32_t* active, void* Z, void* F_z, void* F_u, void* L, void* L_z,
                             void* L_u, void* L_zz, void* L_uz, void* L_uu, void* J_opt, int32_t* status,
                             cudaStream_t st) {
    LinKnownArgs<T> a;
    a.B = s->B; a.N = s->N;
    fill_cost(cost, s, a.cost);
    for (int i = 0; i < 8; ++i) a.dyn.p[i] = (T)dyn->p[i];
    a.p_b = (const T*)dyn->p_b;
    a.z0 = (const T*)z0; a.U = (const T*)U; a.u_min = (const T*)u_min; a.u_max = (const T*)u_max;
    a.active = active;
    a.Z = (T*)Z; a.F_z = (T*)F_z; a.F_u = (T*)F_u; a.L = (T*)L; a.L_z = (T*)L_z; a.L_u = (T*)L_u;
    a.L_zz = (T*)L_zz; a.L_uz = (T*)L_uz; a.L_uu = (T*)L_uu; a.J_opt = (T*)J_opt; a.status = status;
    const int64_t B = s->B, N = s->N, nz = s->nz, nu = s->nu, ly = s->layout;
    a.lZ = make_layout(ly, B, N + 1, nz); a.lU = make_layout(ly, B, N, nu);
    a.lFz = make_layout(ly, B, N, nz * nz); a.lFu = make_layout(ly, B, N, nz * nu);
    a.lL = make_layout(ly, B, N + 1, 1); a.lLz = make_layout(ly, B, N + 1, nz);
    a.lLu = make_layout(ly, B, N, nu); a.lLzz = make_layout(ly, B, N + 1, nz * nz);
    a.lLuz = make_layout(ly, B, N, nu * nz); a.lLuu = make_layout(ly, B, N, nu * nu);
    // uncertain encodings: the kernel rolls the nominal trajectory + dynamics Jacobians and parks
    // the clamped controls in the L_u buffer; the pair-parallel cost kernel then reads them back
    // (the only thread that reads U[b,t] is the one that overwrites L_u[b,t]).
    if (s->geo == GEO_RENDEZVOUS) {             // linear-quadratic: dynamics and cost derivatives in one kernel
        a.U_clamped = nullptr;
        note_launches(1);
        prof_begin(PROF_LIN_KNOWN, st);
        cudaError_t e = linearize_lq<T>(s->enc, a, st);
        prof_end(PROF_LIN_KNOWN, st);
        return cuda_result(e, "pddp_linearize_known(rendezvous)");
    }
    a.U_clamped = s->enc == PDDP_ENC_IGNORE_UNCERTAINTY ? nullptr : (T*)L_u;
    prof_begin(PROF_LIN_KNOWN, st);
    cudaError_t le = linearize_known<T>(s->geo, s->enc, a, st);
    prof_end(PROF_LIN_KNOWN, st);
    if (int e = cuda_result(le, "pddp_linearize_known")) return e;
    note_launches(s->enc == PDDP_ENC_IGNORE_UNCERTAINTY ? 1 : 3);
    if (s->enc == PDDP_ENC_IGNORE_UNCERTAINTY) return 0;
    CostDerivArgs<T> c;
    c.B = s->B; c.N = s->N; c.cost = a.cost; c.Z = a.Z; c.U = (const T*)L_u; c.active = active;
    c.L = a.L; c.L_z = a.L_z; c.L_u = a.L_u; c.L_zz = a.L_zz; c.L_uz = a.L_uz; c.L_uu = a.L_uu; c.J_opt = a.J_opt;
    c.lZ = a.lZ; c.lU = a.lU; c.lL = a.lL; c.lLz = a.lLz; c.lLu = a.lLu; c.lLzz = a.lLzz; c.lLuz = a.lLuz; c.lLuu = a.lLuu;
    prof_begin(PROF_COST, st);
    cudaError_t ce = cost_derivatives<T>(s->geo, s->enc, c, st);
    prof_end(PROF_COST, st);
    return cuda_result(ce, "pddp_linearize_known(cost)");
}

extern "C" int pddp_linearize_known(const pddp_shape* s, const pddp_known_dynamics* dyn, const pddp_cost* cost,
                                    const void* z0, const void* U, const void* u_min, const void* u_max,
                                    const int32_t* active, void* Z, void* F_z, void* F_u, void* L, void* L_z,
                                    void* L_u, void* L_zz, void* L_uz, void* L_uu, void* J_opt,
                                    int32_t* status, void* stream) {
    if (int e = check_shape(s)) return e;
    if (!dyn || !cost || !z0 || !U || !Z || !F_z || !F_u || !L || !L_z || !L_u || !L_zz || !L_uz || !L_uu || !J_opt)
        return fail(PDDP_E_BADARG, "pddp_linearize_known: NULL argument");
    if (int e = check_cost(cost)) return e;
    if ((u_min == nullptr) != (u_max == nullptr)) return fail(PDDP_E_BADARG, "u_min and u_max must be given together");
    cudaStream_t st = (cudaStream_t)stream;
    if (s->dtype == PDDP_F32)
        return linearize_known_t<float>(s, dyn, cost, z0, U, u_min, u_max, active, Z, F_z, F_u, L, L_z, L_u, L_zz, L_uz, L_uu, J_opt, status, st);
    return linearize_known_t<double>(s, dyn, cost, z0, U, u_min, u_max, active, Z, F_z, F_u, L, L_z, L_u, L_zz, L_uz, L_uu, J_opt, status, st);
}

// ---------------------------------------------------------------------------------------------
template <class T>
static int env_step_t(const pddp_shape* s, const pddp_known_dynamics* dyn, const void* x, const void* u, void* xn,
                      cudaStream_t st) {
    KnownParams<T> kp;
    for (int i = 0; i < 8; ++i) kp.p[i] = (T)dyn->p[i];
    const T* p_b = (const T*)dyn->p_b;
    note_launches(1);
    if (s->geo == GEO_RENDEZVOUS)
        return cuda_result(env_step_lq<T>(s->B, kp, p_b, (const T*)x, (const T*)u, (T*)xn, st), "pddp_env_step_known");
    return cuda_result(env_step_known<T>(s->geo, s->B, kp, p_b, (const T*)x, (const T*)u, (T*)xn, st), "pddp_env_step_known");
}

extern "C" int pddp_env_step_known(const pddp_shape* s, const pddp_known_dynamics* dyn, const void* x, const void* u,
                                   void* x_next, void* stream) {
    if (!s) return fail(PDDP_E_BADARG, "shape is NULL");
    if (geo_D(s->geo) < 0) return fail(PDDP_E_UNSUPPORTED, "unsupported geometry");
    if (s->dtype != PDDP_F32 && s->dtype != PDDP_F64) return fail(PDDP_E_BADARG, "dtype must be PDDP_F32 or PDDP_F64");
    if (s->B < 1 || !dyn || !x || !u || !x_next) return fail(PDDP_E_BADARG, "pddp_env_step_known: NULL argument / B < 1");
    cudaStream_t st = (cudaStream_t)stream;
    if (s->dtype == PDDP_F32) return env_step_t<float>(s, dyn, x, u, x_next, st);
    return env_step_t<double>(s, dyn, x, u, x_next, st);
}

// ---------------------------------------------------------------------------------------------
template <class T>
static int backward_t(const pddp_shape* s, const void* F_z, const void* F_u, const void* L_z, const void* L_u,
                      const void* L_zz, const void* L_uz, const void* L_uu, const double* mu, const void* U,
                      const void* u_min, const void* u_max, const int32_t* active, void* k, void* K,
                      int32_t* status, cudaStream_t st) {
    BackwardArgs<T> a;
    a.B = s->B; a.N = s->N; a.nz = s->nz; a.nu = s->nu;
    a.F_z = (const T*)F_z; a.F_u = (const T*)F_u; a.L_z = (const T*)L_z; a.L_u = (const T*)L_u;
    a.L_zz = (const T*)L_zz; a.L_uz = (const T*)L_uz; a.L_uu = (const T*)L_uu; a.mu = mu;
    a.U = (const T*)U; a.u_min = (const T*)u_min; a.u_max = (const T*)u_max; a.active = active;
    a.k = (T*)k; a.K = (T*)K; a.status = status;
    const int64_t B = s->B, N = s->N, nz = s->nz, nu = s->nu, ly = s->layout;
    a.lFz = make_layout(ly, B, N, nz * nz); a.lFu = make_layout(ly, B, N, nz * nu);
    a.lLz = make_layout(ly, B, N + 1, nz); a.lLu = make_layout(ly, B, N, nu);
    a.lLzz = make_layout(ly, B, N + 1, nz * nz); a.lLuz = make_layout(ly, B, N, nu * nz);
    a.lLuu = make_layout(ly, B, N, nu * nu); a.lU = make_layout(ly, B, N, nu);
    a.lk = make_layout(ly, B, N, nu); a.lK = make_layout(ly, B, N, nu * nz);
    note_launches(1);
    prof_begin(PROF_BACKWARD, st);
    cudaError_t e = backward_pass<T>(a, s->layout, st);
    prof_end(PROF_BACKWARD, st);
    return cuda_result(e, "pddp_backward");
}

extern "C" int pddp_backward(const pddp_shape* s, const void* F_z, const void* F_u, const void* L_z,
                             const void* L_u, const void* L_zz, const void* L_uz, const void* L_uu,
                             const double* mu, const void* U, const void* u_min, const void* u_max,
                             const int32_t* active, void* k, void* K, int32_t* status, void* stream) {
    if (int e = check_shape_backward(s)) return e;
    if (!F_z || !F_u || !L_z || !L_u || !L_zz || !L_uz || !L_uu || !mu || !k || !K || !status)
        return fail(PDDP_E_BADARG, "pddp_backward: NULL argument");
    if ((u_min == nullptr) != (u_max == nullptr)) return fail(PDDP_E_BADARG, "u_min and u_max must be given together");
    if (u_min && !U) return fail(PDDP_E_BADARG, "pddp_backward: U is required with bounds");
    cudaStream_t st = (cudaStream_t)stream;
    if (s->dtype == PDDP_F32)
        return backward_t<float>(s, F_z, F_u, L_z, L_u, L_zz, L_uz, L_uu, mu, U, u_min, u_max, active, k, K, status, st);
    return backward_t<double>(s, F_z, F_u, L_z, L_u, L_zz, L_uz, L_uu, mu, U, u_min, u_max, active, k, K, status, st);
}

// ---------------------------------------------------------------------------------------------
template <class T>
static int rollout_known_t(const pddp_shape* s, const pddp_known_dynamics* dyn, const pddp_cost* cost,
                           const void* Z, const void* U, const void* k, const void* K, const void* alphas,
                           int32_t A, const void* u_min, const void* u_max, const int32_t* active,
                           const int32_t* bw_status, void* J_all, int32_t* amin, void* J_new, void* Z_new,
                           void* U_new, cudaStream_t st) {
    RollKnownArgs<T> a;
    a.B = s->B; a.N = s->N; a.A = A;
    fill_cost(cost, s, a.cost);
    for (int i = 0; i < 8; ++i) a.dyn.p[i] = (T)dyn->p[i];
    a.p_b = (const T*)dyn->p_b;
    a.Z = (const T*)Z; a.U = (const T*)U; a.k = (const T*)k; a.K = (const T*)K; a.alphas = (const T*)alphas;
    a.u_min = (const T*)u_min; a.u_max = (const T*)u_max; a.active = active; a.bw_status = bw_status;
    a.J_all = (T*)J_all; a.amin = amin; a.J_new = (T*)J_new; a.Z_new = (T*)Z_new; a.U_new = (T*)U_new;
    const int64_t B = s->B, N = s->N, nz = s->nz, nu = s->nu, ly = s->layout;
    a.lZ = make_layout(ly, B, N + 1, nz); a.lU = make_layout(ly, B, N, nu);
    a.lk = make_layout(ly, B, N, nu); a.lK = make_layout(ly, B, N, nu * nz);
    note_launches(2);
    prof_begin(PROF_ROLL_KNOWN, st);
    cudaError_t e = s->geo == GEO_RENDEZVOUS ? rollout_lq<T>(s->enc, a, st) : rollout_known<T>(s->geo, s->enc, a, st);
    prof_end(PROF_ROLL_KNOWN, st);
    return cuda_result(e, "pddp_rollout_known");
}

extern "C" int pddp_rollout_known(const pddp_shape* s, const pddp_known_dynamics* dyn, const pddp_cost* cost,
                                  const void* Z, const void* U, const void* k, const void* K,
                                  const void* alphas, int32_t A, const void* u_min, const void* u_max,
                                  const int32_t* active, const int32_t* bw_status, void* J_all,
                                  int32_t* amin, void* J_new, void* Z_new, void* U_new, void* stream) {
    if (int e = check_shape(s)) return e;
    if (!dyn || !cost || !Z || !U || !k || !K || !alphas || !J_all || !amin || !J_new || !Z_new || !U_new)
        return fail(PDDP_E_BADARG, "pddp_rollout_known: NULL argument");
    if (int e = check_cost(cost)) return e;
    if (A < 1 || A > 32) return fail(PDDP_E_UNSUPPORTED, "1 <= A <= 32 line-search candidates");
    if ((u_min == nullptr) != (u_max == nullptr)) return fail(PDDP_E_BADARG, "u_min and u_max must be given together");
    cudaStream_t st = (cudaStream_t)stream;
    if (s->dtype == PDDP_F32)
        return rollout_known_t<float>(s, dyn, cost, Z, U, k, K, alphas, A, u_min, u_max, active, bw_status, J_all, amin, J_new, Z_new, U_new, st);
    return rollout_known_t<double>(s, dyn, cost, Z, U, k, K, alphas, A, u_min, u_max, active, bw_status, J_all, amin, J_new, Z_new, U_new, st);
}

// ---------------------------------------------------------------------------------------------
template <class T>
static int accept_t(const pddp_shape* s, const void* J_new, const int32_t* bw_status, const void* Z_new,
                    const void* U_new, double tol, double max_reg, double* mu, double* delta, void* J_opt,
                    int32_t* state, int32_t* iters_left, int32_t* active, void* Z, void* U,
                    int32_t* accepted, int32_t* n_active, const void* K, void* K_nominal, cudaStream_t st) {
    AcceptArgs<T> a;
    a.B = s->B; a.N = s->N; a.nz = s->nz; a.nu = s->nu;
    a.J_new = (const T*)J_new; a.bw_status = bw_status; a.Z_new = (const T*)Z_new; a.U_new = (const T*)U_new;
    a.tol = tol; a.max_reg = max_reg; a.mu = mu; a.delta = delta; a.J_opt = (T*)J_opt; a.state = state;
    a.iters_left = iters_left; a.active = active; a.Z = (T*)Z; a.U = (T*)U; a.n_active = n_active;
    a.lZ = make_layout(s->layout, s->B, s->N + 1, s->nz);
    a.lU = make_layout(s->layout, s->B, s->N, s->nu);
    a.K = (const T*)K; a.K_nominal = (T*)K_nominal;
    a.lK = make_layout(s->layout, s->B, s->N, s->nu * s->nz);
    note_launches(2);
    prof_begin(PROF_ACCEPT, st);
    cudaError_t e = accept_update<T>(a, accepted, st);
    prof_end(PROF_ACCEPT, st);
    return cuda_result(e, "pddp_accept_update");
}

extern "C" int pddp_accept_update(const pddp_shape* s, const void* J_new, const int32_t* bw_status,
                                  const void* Z_new, const void* U_new, double tol, double max_reg,
                                  double* mu, double* delta, void* J_opt, int32_t* state,
                                  int32_t* iters_left, int32_t* active, void* Z, void* U,
                                  int32_t* accepted, int32_t* n_active, const void* K, void* K_nominal,
                                  void* stream) {
    if (int e = check_shape(s)) return e;
    if (!J_new || !Z_new || !U_new || !mu || !delta || !J_opt || !state || !iters_left || !active || !Z || !U || !accepted)
        return fail(PDDP_E_BADARG, "pddp_accept_update: NULL argument");
    if ((K == nullptr) != (K_nominal == nullptr)) return fail(PDDP_E_BADARG, "pddp_accept_update: K and K_nominal go together");
    cudaStream_t st = (cudaStream_t)stream;
    if (s->dtype == PDDP_F32)
        return accept_t<float>(s, J_new, bw_status, Z_new, U_new, tol, max_reg, mu, delta, J_opt, state, iters_left, active, Z, U, accepted, n_active, K, K_nominal, st);
    return accept_t<double>(s, J_new, bw_status, Z_new, U_new, tol, max_reg, mu, delta, J_opt, state, iters_left, active, Z, U, accepted, n_active, K, K_nominal, st);
}

// ---------------------------------------------------------------------------------------------
template <class T>
static int cost_derivs_t(const pddp_shape* s, const pddp_cost* cost, const void* Z, const void* U,
                         const int32_t* active, void* L, void* L_z, void* L_u, void* L_zz, void* L_uz,
                         void* L_uu, void* J_opt, cudaStream_t st) {
    CostDerivArgs<T> a;
    a.B = s->B; a.N = s->N;
    fill_cost(cost, s, a.cost);
    a.Z = (const T*)Z; a.U = (const T*)U; a.active = active;
    a.L = (T*)L; a.L_z = (T*)L_z; a.L_u = (T*)L_u; a.L_zz = (T*)L_zz; a.L_uz = (T*)L_uz; a.L_uu = (T*)L_uu;
    a.J_opt = (T*)J_opt;
    const int64_t B = s->B, N = s->N, nz = s->nz, nu = s->nu, ly = s->layout;
    a.lZ = make_layout(ly, B, N + 1, nz); a.lU = make_layout(ly, B, N, nu);
    a.lL = make_layout(ly, B, N + 1, 1); a.lLz = make_layout(ly, B, N + 1, nz);
    a.lLu = make_layout(ly, B, N, nu); a.lLzz = make_layout(ly, B, N + 1, nz * nz);
    a.lLuz = make_layout(ly, B, N, nu * nz); a.lLuu = make_layout(ly, B, N, nu * nu);
    if (s->geo == GEO_RENDEZVOUS) {
        note_launches(a.J_opt ? 2 : 1);
        return cuda_result(cost_derivatives_lq<T>(s->enc, a, st), "pddp_cost_derivatives(rendezvous)");
    }
    note_launches((a.J_opt ? 2 : 1) + (s->enc == PDDP_ENC_FULL_COVARIANCE_MATRIX ? 1 : 0));
    return cuda_result(cost_derivatives<T>(s->geo, s->enc, a, st), "pddp_cost_derivatives");
}

extern "C" int pddp_cost_derivatives(const pddp_shape* s, const pddp_cost* cost, const void* Z, const void* U,
                                     const int32_t* active, void* L, void* L_z, void* L_u, void* L_zz,
                                     void* L_uz, void* L_uu, void* J_opt, void* stream) {
    if (int e = check_shape(s)) return e;
    if (!cost || !Z || !U || !L || !L_z || !L_u || !L_zz || !L_uz || !L_uu)
        return fail(PDDP_E_BADARG, "pddp_cost_derivatives: NULL argument");
    if (int e = check_cost(cost)) return e;
    cudaStream_t st = (cudaStream_t)stream;
    if (s->dtype == PDDP_F32) return cost_derivs_t<float>(s, cost, Z, U, active, L, L_z, L_u, L_zz, L_uz, L_uu, J_opt, st);
    return cost_derivs_t<double>(s, cost, Z, U, active, L, L_z, L_u, L_zz, L_uz, L_uu, J_opt, st);
}
