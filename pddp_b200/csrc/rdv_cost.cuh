// QR cost of the rendezvous problem on the un-augmented state (D = 8, action_size = 4, no angles), shared by the
// known-dynamics path (known_lq.cu) and the BNN line search (bnn.cu).
// ref: pddp/examples/rendezvous/cost.py:29-43 + pddp/costs/quadratic.py:60-99
#pragma once
#include "core.cuh"

namespace pddp {

constexpr int RDV_D = 8, RDV_NU = 4;

// state part of the QR cost: (m - xg)^T Q (m - xg) + sum_ij C_ij Q_ji   ref: costs/quadratic.py:80-97
template <int ENC, class T>
__device__ __forceinline__ T rdv_cost_state(const CostParams<T>& cp, const T* z, bool terminal) {
    constexpr int D = RDV_D;
    const T* Q = terminal ? cp.Qt : cp.Q;
    T val = T(0);
#pragma unroll
    for (int i = 0; i < D; ++i) {
        T row = T(0);
#pragma unroll
        for (int j = 0; j < D; ++j) row += (z[j] - cp.xg[j]) * Q[j * D + i];
        val += row * (z[i] - cp.xg[i]);
    }
    if (ENC == ENC_FULL) {
#pragma unroll 1
        for (int i = 0; i < D; ++i)
            for (int j = 0; j < D; ++j) val += z[D + i * D + j] * Q[j * D + i];
    } else if (ENC == ENC_UT) {
        for (int i = 0; i < D; ++i)
            for (int j = 0; j < D; ++j) {
                T c = T(0);
                const int m = i < j ? i : j;
                for (int k = 0; k <= m; ++k) c += z[D + tri<D>(k, i)] * z[D + tri<D>(k, j)];
                val += c * Q[j * D + i];
            }
    } else if (ENC == ENC_VAR) {
#pragma unroll
        for (int a = 0; a < D; ++a) val += z[D + a] * Q[a * D + a];
    } else if (ENC == ENC_STD) {
#pragma unroll
        for (int a = 0; a < D; ++a) val += z[D + a] * z[D + a] * Q[a * D + a];
    }
    return val;
}

template <class T>
__device__ __forceinline__ T rdv_cost_action(const CostParams<T>& cp, const T* u) {
    T val = T(0);
#pragma unroll
    for (int i = 0; i < RDV_NU; ++i) {
        T row = T(0);
#pragma unroll
        for (int j = 0; j < RDV_NU; ++j) row += (u[j] - cp.ug[j]) * cp.R[j * RDV_NU + i];
        val += row * (u[i] - cp.ug[i]);
    }
    return val;
}

}  // namespace pddp
