// Shared by spline_deriv.cu (decode of orders 0..2) and spline_deriv_grad.cu (its adjoint): the grid object and the
// in-kernel Cox-de Boor recursion with its derivative form.
#pragma once
#include "common.cuh"

namespace beast {

struct Grid {
    const Plan* plan;
    int Tq, max_order;
    float* dev_block;     // times [Tq], rows_j [(max_order+1)][Tq][nc], rows_g [(max_order+1)][Tq][nb] (grippers only)
    float* times_d;
    float* rows_j_d;
    float* rows_g_d;
    int* bands_d;         // [joint | gripper][Tq][lo, hi): union over the orders of the non-zero columns of each row
    int* list_d;          // dec_list of the grid: token positions some row reads, k | slot << 16 | gripper << 31
    int* colsup_d;        // [joint | gripper][nb][lo, hi): the rows t whose band holds column k (first, last + 1)
    int n_dec;
    int band_max;
};

// d/du of the degree-q basis from the degree-(q-1) values `in` (n entries out); in place when out == in.
__device__ inline void deriv_step(const float* __restrict__ kn, int q, const float* in, float* out, int n) {
    const float fq = (float)q;
    for (int i = 0; i < n; ++i) {
        const float d1 = __fsub_rn(kn[i + q], kn[i]);
        const float d2 = __fsub_rn(kn[i + q + 1], kn[i + 1]);
        const bool h1 = d1 != 0.0f, h2 = d2 != 0.0f;
        const float a = h1 ? __fdiv_rn(in[i], d1) : 0.0f;
        const float b = h2 ? __fdiv_rn(in[i + 1], d2) : 0.0f;
        const float v = (h1 && h2) ? __fsub_rn(a, b) : (h1 ? a : (h2 ? -b : 0.0f));
        out[i] = __fmul_rn(v, fq);
    }
}

// Cox-de Boor exactly as deboor_basis (spline_decode.cu): N[0..nb) <- basis values at u; D1 / D2 [0..nb) <- d/du and
// d2/du2 when max_order >= 1 / 2, taken from levels p-1 / p-2 before they are overwritten.
__device__ inline void deboor_deriv(const float* __restrict__ kn, int nb, int p, float u, int max_order, float* N,
                                    float* D1, float* D2) {
    const int n0 = nb + p;
    for (int i = 0; i < n0; ++i) {
        const bool in = (u >= kn[i]) && (i == nb - 1 ? (u <= kn[i + 1]) : (u < kn[i + 1]));
        N[i] = in ? 1.0f : 0.0f;
    }
    if (max_order >= 1 && p < 1)
        for (int i = 0; i < nb; ++i) D1[i] = 0.0f;
    if (max_order >= 2 && p < 2)
        for (int i = 0; i < nb; ++i) D2[i] = 0.0f;
    for (int k = 1; k <= p; ++k) {
        if (k == p - 1 && max_order >= 2) {
            deriv_step(kn, p - 1, N, D2, n0 - (p - 1));      // d/du of level p-1
            deriv_step(kn, p, D2, D2, nb);                   // d2/du2 of level p
        }
        if (k == p && max_order >= 1) deriv_step(kn, p, N, D1, nb);
        for (int i = 0; i < n0 - k; ++i) {
            const float d1 = __fsub_rn(kn[i + k], kn[i]);
            const float d2 = __fsub_rn(kn[i + k + 1], kn[i + 1]);
            const bool h1 = d1 != 0.0f, h2 = d2 != 0.0f;
            const float t1 = h1 ? __fmul_rn(__fdiv_rn(__fsub_rn(u, kn[i]), d1), N[i]) : 0.0f;
            const float t2 = h2 ? __fmul_rn(__fdiv_rn(__fsub_rn(kn[i + k + 1], u), d2), N[i + 1]) : 0.0f;
            N[i] = (h1 && h2) ? __fadd_rn(t1, t2) : (h1 ? t1 : t2);
        }
    }
}

}  // namespace beast
