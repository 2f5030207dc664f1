// Leaf math shared by every kernel: problem geometry, state encodings, closed-form angular moment
// matching, the QR cost and the three known-dynamics models -- each a template over the scalar
// type S so the same code runs on plain T (rollout / line search), Jet1 (dynamics Jacobian) and
// Jet2 (cost gradient + Hessian).  Citations `ref:` are relative to /root/reference/pddp/.
#pragma once
#include "jet.cuh"
#include <stdint.h>

namespace pddp {

// ---- enums shared with include/pddp_b200.h -------------------------------------------------
enum { ENC_FULL = 0, ENC_UT = 1, ENC_VAR = 2, ENC_STD = 3, ENC_IGNORE = 4 };      // ref: utils/encoding.py:25-33
enum { GEO_PENDULUM = 0, GEO_CARTPOLE = 1, GEO_DOUBLE_CARTPOLE = 2, GEO_RENDEZVOUS = 3 };
enum { ST_UNDEFINED = 0, ST_ACCEPTED = 1, ST_REJECTED = 2, ST_NOT_PD = 3, ST_MAX_REG = 4,
       ST_CONVERGED = 5 };                                                       // ref: controllers/ilqr.py:35-64
enum { LAYOUT_PROBLEM_MAJOR = 0, LAYOUT_BATCH_INNER = 1 };

constexpr int MAX_DA = 8;
constexpr int MAX_NU = 4;   // rendezvous (ref: examples/rendezvous/model.py) has action_size 4

// ---- geometry: which state dims are angles (ref: examples/*/model.py angular_indices) -------
template <int GEO> struct Geo;
template <> struct Geo<GEO_PENDULUM> {
    static constexpr int D = 2, NU = 1, NANG = 1, NNA = 1, DA = 3;
    PDDP_HD static constexpr int ang(int) { return 0; }
    PDDP_HD static constexpr int nonang(int) { return 1; }
};
template <> struct Geo<GEO_CARTPOLE> {
    static constexpr int D = 4, NU = 1, NANG = 1, NNA = 3, DA = 5;
    PDDP_HD static constexpr int ang(int) { return 2; }
    PDDP_HD static constexpr int nonang(int i) { return i == 0 ? 0 : (i == 1 ? 1 : 3); }
};
template <> struct Geo<GEO_DOUBLE_CARTPOLE> {
    static constexpr int D = 6, NU = 1, NANG = 2, NNA = 4, DA = 8;
    PDDP_HD static constexpr int ang(int i) { return i == 0 ? 2 : 4; }
    PDDP_HD static constexpr int nonang(int i) { return i == 0 ? 0 : (i == 1 ? 1 : (i == 2 ? 3 : 5)); }
};
// two point masses in the plane (ref: examples/rendezvous/model.py): no angles, so the augmented state is the state.
// The known-dynamics path (known_lq.cu) does not use this struct; the BNN path does, with the QR cost of rdv_cost.cuh.
template <> struct Geo<GEO_RENDEZVOUS> {
    static constexpr int D = 8, NU = 4, NANG = 0, NNA = 8, DA = 8;
    PDDP_HD static constexpr int ang(int) { return 0; }      // (never called: NANG == 0)
    PDDP_HD static constexpr int nonang(int i) { return i; }
};

PDDP_HD constexpr int enc_size(int D, int enc) {          // ref: utils/encoding.py:46-67
    return enc == ENC_FULL ? D + D * D
         : enc == ENC_UT   ? (3 * D + D * D) / 2
         : enc == ENC_IGNORE ? D : 2 * D;
}

// ---- memory layout of a [B, Nt, E] tensor ---------------------------------------------------
// PROBLEM_MAJOR: ((b*Nt + t)*E + e)   -- the reference layout with a leading problem dim; a warp /
//                CTA that owns one problem streams contiguous records.
// BATCH_INNER:   ((t*E + e)*B + b)    -- SoA over problems; thread-per-problem kernels coalesce.
struct Layout {
    int64_t sb, st, se;
    PDDP_HD int64_t at(int64_t b, int64_t t, int64_t e) const { return b * sb + t * st + e * se; }
};
PDDP_HD Layout make_layout(int layout, int64_t B, int64_t Nt, int64_t E) {
    Layout l;
    if (layout == LAYOUT_BATCH_INNER) { l.sb = 1; l.st = E * B; l.se = B; }
    else { l.sb = Nt * E; l.st = E; l.se = 1; }
    return l;
}

// ---- cost constants (by-value kernel parameter) ---------------------------------------------
template <class T>
struct CostParams {          // ref: costs/quadratic.py:39-58 ; Q acts on the AUGMENTED state
    T Q[MAX_DA * MAX_DA];
    T Qt[MAX_DA * MAX_DA];
    T R[MAX_NU * MAX_NU];
    T xg[MAX_DA];
    T ug[MAX_NU];
};

// ---- decoders (ref: utils/encoding.py:144-362) ----------------------------------------------
template <int D, int ENC, class S, class T>
PDDP_HD void decode_covar(const S* z, S (&C)[D][D]) {
    if (ENC == ENC_FULL) {
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = 0; b < D; ++b) C[a][b] = z[D + a * D + b];
    } else if (ENC == ENC_UT) {                          // C = U^T U, U upper, row-major triu order
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = a; b < D; ++b) {
                S acc = z[D + tri<D>(0, a)] * z[D + tri<D>(0, b)];
#pragma unroll
                for (int k = 1; k <= a; ++k) acc = acc + z[D + tri<D>(k, a)] * z[D + tri<D>(k, b)];
                C[a][b] = acc;
                C[b][a] = acc;
            }
    } else {
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = 0; b < D; ++b) C[a][b] = S(T(0));
#pragma unroll
        for (int a = 0; a < D; ++a)
            C[a][a] = ENC == ENC_VAR ? z[D + a] : (ENC == ENC_STD ? z[D + a] * z[D + a] : S(T(1e-6)));
    }
}

template <int D, int ENC, class S, class T>
PDDP_HD void decode_var(const S* z, S (&V)[D]) {
#pragma unroll
    for (int a = 0; a < D; ++a) {
        if (ENC == ENC_FULL) V[a] = z[D + a * D + a];
        else if (ENC == ENC_UT) {                        // column sums of U^2
            S acc = z[D + tri<D>(0, a)] * z[D + tri<D>(0, a)];
#pragma unroll
            for (int k = 1; k <= a; ++k) acc = acc + z[D + tri<D>(k, a)] * z[D + tri<D>(k, a)];
            V[a] = acc;
        } else if (ENC == ENC_VAR) V[a] = z[D + a];
        else if (ENC == ENC_STD) V[a] = z[D + a] * z[D + a];
        else V[a] = S(T(1e-6));
    }
}

// ---- expected QR cost of the angle-augmented Gaussian ---------------------------------------
// ref: examples/*/cost.py forward -> utils/angular.py:47-84,161-248 -> costs/quadratic.py:60-99.
// The reference re-encodes the augmented moments (a Cholesky for UT) and decodes them again inside
// QRCost; U^T U == C (+1e-12 I jitter) so the round trip is the identity and is not replayed here.
// l_x(z) only; the action term du^T R du is separable (L_uz == 0) and handled by the caller.
// sine / cosine of the angular components of a state: evaluated ONCE per state and shared by the cost and the
// dynamics of the same step (the rollout of the closed-form models is bound by instruction issue, and the three
// separate sinf / cosf calls per pendulum step were a third of it)
template <int GEO, class S>
struct StateTrig { S s[Geo<GEO>::NANG > 0 ? Geo<GEO>::NANG : 1], c[Geo<GEO>::NANG > 0 ? Geo<GEO>::NANG : 1]; };
template <int GEO, class S>
PDDP_HD void state_trig(const S* z, StateTrig<GEO, S>& tr) {
#pragma unroll
    for (int i = 0; i < Geo<GEO>::NANG; ++i) jsincos(z[Geo<GEO>::ang(i)], tr.s[i], tr.c[i]);
}

template <int GEO, int ENC, class T, class S>
PDDP_HD S cost_state(const CostParams<T>& cp, const S* z, bool terminal, const StateTrig<GEO, S>& tr) {
    typedef Geo<GEO> G;
    constexpr int D = G::D, DA = G::DA, NNA = G::NNA, NANG = G::NANG;
    const T* Q = terminal ? cp.Qt : cp.Q;
    S Ma[DA];
    S sn[NANG > 0 ? NANG : 1], cs[NANG > 0 ? NANG : 1];
    if (ENC == ENC_IGNORE) {                              // ref: utils/angular.py:251-286
#pragma unroll
        for (int i = 0; i < NNA; ++i) Ma[i] = z[G::nonang(i)];
#pragma unroll
        for (int i = 0; i < NANG; ++i) {
            Ma[NNA + 2 * i] = tr.s[i];
            Ma[NNA + 2 * i + 1] = tr.c[i];
        }
        S val = S(T(0));
#pragma unroll
        for (int i = 0; i < DA; ++i) {
            S row = S(T(0));
#pragma unroll
            for (int j = 0; j < DA; ++j) row = row + (Ma[j] - cp.xg[j]) * Q[i * DA + j];
            val = val + (Ma[i] - cp.xg[i]) * row;
        }
        return val;
    }
    S C[D][D];
    decode_covar<D, ENC, S, T>(z, C);
#pragma unroll
    for (int i = 0; i < NNA; ++i) Ma[i] = z[G::nonang(i)];
#pragma unroll
    for (int i = 0; i < NANG; ++i) {
        S damp = jexp(C[G::ang(i)][G::ang(i)] * T(-0.5));
        sn[i] = damp * tr.s[i];
        cs[i] = damp * tr.c[i];
        Ma[NNA + 2 * i] = sn[i];
        Ma[NNA + 2 * i + 1] = cs[i];
    }
    S val = S(T(0));
#pragma unroll
    for (int i = 0; i < DA; ++i) {
        S row = S(T(0));
#pragma unroll
        for (int j = 0; j < DA; ++j) row = row + (Ma[j] - cp.xg[j]) * Q[i * DA + j];
        val = val + (Ma[i] - cp.xg[i]) * row;
    }
    // trace term sum_ij Ca[i][j] * Q[j][i], block by block
#pragma unroll
    for (int i = 0; i < NNA; ++i)
#pragma unroll
        for (int j = 0; j < NNA; ++j) val = val + C[G::nonang(i)][G::nonang(j)] * Q[j * DA + i];
    if (ENC == ENC_FULL || ENC == ENC_UT) {
        // cross blocks: Ca[jn][NNA+2i] = c[ang_i][nonang_jn]*cos_i ; [..+1] = -c*sin_i ; and transpose
#pragma unroll
        for (int i = 0; i < NANG; ++i)
#pragma unroll
            for (int jn = 0; jn < NNA; ++jn) {
                S cr = C[G::ang(i)][G::nonang(jn)];
                T qs = Q[(NNA + 2 * i) * DA + jn] + Q[jn * DA + NNA + 2 * i];
                T qc = Q[(NNA + 2 * i + 1) * DA + jn] + Q[jn * DA + NNA + 2 * i + 1];
                val = val + cr * (cs[i] * qs - sn[i] * qc);
            }
    }
#pragma unroll
    for (int i = 0; i < NANG; ++i)
#pragma unroll
        for (int j = 0; j < NANG; ++j) {
            if ((ENC == ENC_VAR || ENC == ENC_STD) && i != j) continue;   // _augment_var keeps the diagonal
            S cii = C[G::ang(i)][G::ang(i)], cjj = C[G::ang(j)][G::ang(j)];
            S cij = C[G::ang(i)][G::ang(j)];
            S lq = (cii + cjj) * T(-0.5);
            S q = jexp(lq);
            S ep = jexp(lq + cij) - q, em = jexp(lq - cij) - q;
            S dm = z[G::ang(i)] - z[G::ang(j)], sm = z[G::ang(i)] + z[G::ang(j)];
            S sdm, cdm, ssm, csm;
            jsincos(dm, sdm, cdm);
            jsincos(sm, ssm, csm);
            S U3 = ep * cdm, U4 = em * csm;
            const int si = NNA + 2 * i, ci = si + 1, sj = NNA + 2 * j, cj = sj + 1;
            // Va[si][sj] = .5(U3-U4), Va[ci][cj] = .5(U3+U4); multiplied by Q[sj][si], Q[cj][ci]
            val = val + (U3 - U4) * (T(0.5) * Q[sj * DA + si]) + (U3 + U4) * (T(0.5) * Q[cj * DA + ci]);
            if (ENC == ENC_FULL || ENC == ENC_UT) {
                S U1 = ep * sdm, U2 = em * ssm;
                // Va[si][cj] = .5(U1+U2)[i][j] times Q[cj][si]; Va[cj][si] (transpose) times Q[si][cj]
                val = val + (U1 + U2) * (T(0.5) * (Q[cj * DA + si] + Q[si * DA + cj]));
            }
        }
    return val;
}

template <int GEO, int ENC, class T, class S>
PDDP_HD S cost_state(const CostParams<T>& cp, const S* z, bool terminal) {
    StateTrig<GEO, S> tr;
    state_trig<GEO, S>(z, tr);
    return cost_state<GEO, ENC, T, S>(cp, z, terminal, tr);
}

// action part of the cost: value, gradient, Hessian (NU == 1)   ref: costs/quadratic.py:86-89
template <class T>
PDDP_HD void cost_action(const CostParams<T>& cp, T u, T& l, T& l_u, T& l_uu) {
    T du = u - cp.ug[0];
    l = du * cp.R[0] * du;
    l_u = T(2) * cp.R[0] * du;
    l_uu = T(2) * cp.R[0];
}

// ---- known dynamics, mean part (ref: examples/*/model.py) -----------------------------------
template <class T>
struct KnownParams { T p[8]; };   // pendulum: dt,m,l,mu,g | cartpole: dt,mc,mp,l,mu,g | double: dt,mc,mp1,mp2,l1,l2,mu,g

template <int GEO, class T, class S>
PDDP_HD void known_mean_step(const KnownParams<T>& kp, const S* x, const S& u, S* xn, const StateTrig<GEO, S>& tr) {
    const T* p = kp.p;
    if (GEO == GEO_PENDULUM) {                            // ref: examples/pendulum/model.py:84-119
        T dt = p[0], m = p[1], l = p[2], mu = p[3], g = p[4];
        T ml = m * l;
        S acc = (u - x[1] * mu - tr.s[0] * (T(0.5) * ml * g)) * (T(3) / (ml * l));
        xn[0] = x[0] + x[1] * dt;
        xn[1] = x[1] + acc * dt;
    } else if (GEO == GEO_CARTPOLE) {                     // ref: examples/cartpole/model.py:88-141
        T dt = p[0], mc = p[1], mp = p[2], l = p[3], mu = p[4], g = p[5];
        S s = tr.s[0], c = tr.c[0];
        S a0 = x[3] * x[3] * s * (mp * l);
        S a1 = s * g;
        S a2 = u - x[1] * mu;
        S a3 = T(4) * (mc + mp) - c * c * (T(3) * mp);
        S thdd = (a0 * c + (a1 * (mc + mp) + a2 * c) * T(2)) * T(-3) / (a3 * l);
        S acc = (a0 * T(2) + a1 * c * (T(3) * mp) + a2 * T(4)) / a3;
        S nvel = x[1] + acc * dt, nthd = x[3] + thdd * dt;
        xn[0] = x[0] + nvel * dt;
        xn[1] = nvel;
        xn[2] = x[2] + nthd * dt;
        xn[3] = nthd;
    } else {                                              // ref: examples/double_cartpole/model.py:100-195
        T dt = p[0], mc = p[1], mp1 = p[2], mp2 = p[3], l1 = p[4], l2 = p[5], mu = p[6], g = p[7];
        S s1 = tr.s[0], c1 = tr.c[0], s2 = tr.s[1], c2 = tr.c[1];
        S sd, cd;
        jsincos(x[2] - x[4], sd, cd);
        T a0 = mp2 + T(2) * mc, a1 = mc * l2;
        S a2 = x[3] * x[3] * l1, a3 = x[5] * x[5] * a1;
        // A sol = b, rows as in the reference
        S A00 = S(T(2) * (mp1 + mp2 + mc)), A01 = c1 * (-a0 * l1), A02 = c2 * (-a1);
        S A10 = c1 * (T(-3) * a0), A11 = S((T(2) * a0 + T(2) * mc) * l1), A12 = cd * (T(3) * a1);
        S A20 = c2 * T(-3), A21 = cd * (T(3) * l1), A22 = S(T(2) * l2);
        S b0 = u * T(2) - x[1] * (T(2) * mu) - a2 * s1 * a0 - a3 * s2;
        S b1 = s1 * (T(3) * a0 * g) - a3 * sd * T(3);
        S b2 = a2 * sd * T(3) + s2 * (T(3) * g);
        // Cramer / adjugate solve (the reference uses LU; A is 3x3 and well conditioned)
        S m00 = A11 * A22 - A12 * A21, m01 = A10 * A22 - A12 * A20, m02 = A10 * A21 - A11 * A20;
        S det = A00 * m00 - A01 * m01 + A02 * m02;
        S x0 = b0 * m00 - A01 * (b1 * A22 - A12 * b2) + A02 * (b1 * A21 - A11 * b2);
        S x1 = A00 * (b1 * A22 - A12 * b2) - b0 * m01 + A02 * (A10 * b2 - b1 * A20);
        S x2 = A00 * (A11 * b2 - b1 * A21) - A01 * (A10 * b2 - b1 * A20) + b0 * m02;
        S nvel = x[1] + x0 / det * dt, n1 = x[3] + x1 / det * dt, n2 = x[5] + x2 / det * dt;
        xn[0] = x[0] + nvel * dt;
        xn[1] = nvel;
        xn[2] = x[2] + n1 * dt;
        xn[3] = n1;
        xn[4] = x[4] + n2 * dt;
        xn[5] = n2;
    }
}

template <int GEO, class T, class S>
PDDP_HD void known_mean_step(const KnownParams<T>& kp, const S* x, const S& u, S* xn) {
    StateTrig<GEO, S> tr;
    state_trig<GEO, S>(x, tr);
    known_mean_step<GEO, T, S>(kp, x, u, xn, tr);
}

// Known models pass the variance through unchanged and drop off-diagonal covariance
// (SURVEY quirk 15; ref: examples/pendulum/model.py:103,119).  Writes the uncertainty part of z'.
template <int D, int ENC, class T>
PDDP_HD void known_uncertainty_step(const T* z, T* zn) {
    if (ENC == ENC_IGNORE) return;
    T V[D];
    decode_var<D, ENC, T, T>(z, V);
    if (ENC == ENC_FULL) {
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = 0; b < D; ++b) zn[D + a * D + b] = a == b ? V[a] : T(0);
    } else if (ENC == ENC_UT) {                           // chol(diag(V) + 1e-12 I), ref: utils/encoding.py:536-564
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = a; b < D; ++b) zn[D + tri<D>(a, b)] = a == b ? jsqrt(V[a] + T(1e-12)) : T(0);
    } else if (ENC == ENC_VAR) {
#pragma unroll
        for (int a = 0; a < D; ++a) zn[D + a] = V[a];
    } else {
#pragma unroll
        for (int a = 0; a < D; ++a) zn[D + a] = jsqrt(V[a]);
    }
}

// d(uncertainty part of z') / d z  for the pass-through above; only non-zero entries are visited.
template <int D, int ENC, class T, class F>
PDDP_HD void known_uncertainty_jacobian(const T* z, const T* zn, F&& emit /* (row, col, value) */) {
    if (ENC == ENC_FULL) {
#pragma unroll
        for (int a = 0; a < D; ++a) emit(D + a * D + a, D + a * D + a, T(1));
    } else if (ENC == ENC_UT) {
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int k = 0; k <= a; ++k)
                emit(D + tri<D>(a, a), D + tri<D>(k, a), z[D + tri<D>(k, a)] / zn[D + tri<D>(a, a)]);
    } else if (ENC == ENC_VAR) {
#pragma unroll
        for (int a = 0; a < D; ++a) emit(D + a, D + a, T(1));
    } else if (ENC == ENC_STD) {
#pragma unroll
        for (int a = 0; a < D; ++a) emit(D + a, D + a, z[D + a] / zn[D + a]);
    }
}

PDDP_HD float clampv(float u, float lo, float hi) { return fminf(fmaxf(u, lo), hi); }
PDDP_HD double clampv(double u, double lo, double hi) { return fmin(fmax(u, lo), hi); }

}  // namespace pddp
