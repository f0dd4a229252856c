// ocd_hessian.cuh -- second derivatives of the horizon-summed features with respect to the controls.
//
// What the reference's second-order inverse optimal control (LocalCIOC, interact_drive/reward_design/
// second_order_ioc.py:80-152) takes from TensorFlow as `t.jacobian(gradients, controls)`: the Hessian of
// sum_t phi_k(s_{t+1}(u)) in the 2H controls of one window.  The reward is linear in the weights, so the K
// per-feature Hessians (and the K rows of ocd_feature_jacobian_batch) are everything CIOC's likelihood and its
// weight gradient need -- no third derivatives.
//
// Method: hyper-dual numbers  a + b e1 + c e2 + d e1 e2  (e1^2 = e2^2 = 0): one rollout of
// naive_planner.py:32-79 in that arithmetic, seeded with e1 on control i and e2 on control j, returns
// d^2 Phi_k / du_i du_j for every feature k at once in the e1 e2 component -- exact second derivatives (no
// differencing), float32 throughout.  One thread per (problem, pair i <= j).  Piecewise operations (clip, Minimum,
// reduce_min / reduce_max, where, abs) follow the branch TensorFlow's gradients follow (SURVEY.md A.3); exactly
// at a kink the second derivative is that of the selected branch (first of several tied branches).
// Same formulas and reference lines as ocd_device.cuh's PRECISE back-end:
//   dynamics   interact_drive/simulation_utils.py:9-21      smooth helpers  interact_drive/math_utils.py:7-31, 59-97, 135-180
//   features   experiments/merging.py:32-83                 other cars      interact_drive/planner/naive_planner.py:47-67
#pragma once

#include "ocd_device.cuh"

namespace ocd {

struct HD {              // value, d/de1, d/de2, d2/de1 de2
    float v, a, b, ab;
};
__device__ __forceinline__ HD hd_const(float c) { return HD{c, 0.0f, 0.0f, 0.0f}; }
__device__ __forceinline__ HD operator+(HD x, HD y) { return HD{x.v + y.v, x.a + y.a, x.b + y.b, x.ab + y.ab}; }
__device__ __forceinline__ HD operator-(HD x, HD y) { return HD{x.v - y.v, x.a - y.a, x.b - y.b, x.ab - y.ab}; }
__device__ __forceinline__ HD operator-(HD x) { return HD{-x.v, -x.a, -x.b, -x.ab}; }
__device__ __forceinline__ HD operator+(HD x, float c) { return HD{x.v + c, x.a, x.b, x.ab}; }
__device__ __forceinline__ HD operator-(HD x, float c) { return HD{x.v - c, x.a, x.b, x.ab}; }
__device__ __forceinline__ HD operator*(HD x, float c) { return HD{x.v * c, x.a * c, x.b * c, x.ab * c}; }
__device__ __forceinline__ HD operator*(HD x, HD y) {
    return HD{x.v * y.v, fmaf(x.a, y.v, x.v * y.a), fmaf(x.b, y.v, x.v * y.b),
              fmaf(x.ab, y.v, fmaf(x.a, y.b, fmaf(x.b, y.a, x.v * y.ab)))};
}
// g(x) for a scalar function with first and second derivative g1, g2 at x.v
__device__ __forceinline__ HD hd_chain(HD x, float g, float g1, float g2) {
    return HD{g, g1 * x.a, g1 * x.b, fmaf(g2, x.a * x.b, g1 * x.ab)};
}
__device__ __forceinline__ HD hd_sin(HD x) { const float s = sinf(x.v), c = cosf(x.v); return hd_chain(x, s, c, -s); }
__device__ __forceinline__ HD hd_cos(HD x) { const float s = sinf(x.v), c = cosf(x.v); return hd_chain(x, c, -s, -c); }
__device__ __forceinline__ HD hd_exp(HD x) { const float e = expf(x.v); return hd_chain(x, e, e, e); }
__device__ __forceinline__ HD hd_rcp(HD x) {
    const float r = __fdiv_rn(1.0f, x.v), r2 = r * r;
    return hd_chain(x, r, -r2, 2.0f * r2 * r);
}

// _f (math_utils.py:7-31): exp(-1/(shape q)) for q > 0, else 0 (where() routes no derivative to the other branch)
__device__ __forceinline__ HD hd_f(HD q, float shape) {
    if (q.v > 0.0f) return hd_exp(-hd_rcp(q * shape));
    return hd_const(0.0f);
}
// smooth_threshold(threshold, width)(z) (math_utils.py:59-97)
__device__ __forceinline__ HD hd_threshold(const KParams &k, HD z) {
    const HD q = z - k.thr_lo;
    const HD u2 = hd_const(k.thr_w) - q;
    const HD F1 = hd_f(q, k.fshape), F2 = hd_f(u2, k.fshape);
    return F1 * hd_rcp(F1 + F2);
}
// smooth_bump(c - hw, c + hw)(z) (math_utils.py:135-180)
__device__ __forceinline__ HD hd_bump(HD z, float c, float hw) {
    const float start = __fsub_rn(c, hw), end = __fadd_rn(c, hw);
    const float width = __fmul_rn(__fsub_rn(end, start), 0.5f), center = __fmul_rn(__fadd_rn(start, end), 0.5f);
    const HD n = (z - center) * __fdiv_rn(1.0f, width);
    if (n.v * n.v < 1.0f) {
        const HD om = hd_const(1.0f) - n * n;
        return hd_exp(hd_const(1.0f) - hd_rcp(om));
    }
    return hd_const(0.0f);
}

#ifndef OCD_HD_ONLY   // translation units that only use the hyper-dual arithmetic (ocd_vjp.cuh in ocd_inst.cu)
// One thread: problem b, control pair (i, j) with i <= j (flat indices into [H][2]).  hess [K][2H][2H][B].
__global__ void __launch_bounds__(128)
k_feature_hessian(const __grid_constant__ KParams k, const float *world, const float *controls,
                  const float *other_controls, long long Bo, float *hess, long long B) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int n = 2 * k.H;
    // pair index -> (i, j), i <= j, rows of the upper triangle in order
    int i = 0, rem = (int)blockIdx.y;
    while (rem >= n - i) { rem -= n - i; ++i; }
    const int j = i + rem;

    HD x = hd_const(world[b]), y = hd_const(world[B + b]), v = hd_const(world[2 * B + b]), th = hd_const(world[3 * B + b]);
    float os[OCD_MAX_OTHER][4];                       // the other cars' states under the planner's model
    for (int c = 0; c < k.NO; ++c)
        for (int q = 0; q < 4; ++q) os[c][q] = world[(size_t)((c + 1) * 4 + q) * B + b];
    HD phi_sum[OCD_MAX_LANES + 4];
#pragma unroll
    for (int q = 0; q < OCD_MAX_LANES + 4; ++q) phi_sum[q] = hd_const(0.0f);

    for (int t = 0; t < k.H; ++t) {
        HD a = hd_const(controls[(size_t)(t * 2 + 0) * B + b]), om = hd_const(controls[(size_t)(t * 2 + 1) * B + b]);
        if (2 * t == i) a.a = 1.0f;
        if (2 * t == j) a.b = 1.0f;
        if (2 * t + 1 == i) om.a = 1.0f;
        if (2 * t + 1 == j) om.b = 1.0f;
        // clip_by_value: outside [lo, hi] the value is the bound and nothing flows (inclusive masks)
        const HD ac = a.v > 4.0f ? hd_const(4.0f) : (a.v < -8.0f ? hd_const(-8.0f) : a);
        const HD oc = om.v > 4.0f ? hd_const(4.0f) : (om.v < -4.0f ? hd_const(-4.0f) : om);
        const HD total = ac - (v * v) * k.mu;
        const HD dist = v * k.dt + (total * 0.5f) * k.dt2;
        const HD cs = hd_cos(th), sn = hd_sin(th);
        x = x + cs * dist;
        y = y + sn * dist;
        v = v + total * k.dt;
        th = th + oc * k.dt;
        for (int c = 0; c < k.NO; ++c) {              // naive_planner.py:53-66
            float oa = 0.0f, oo = 0.0f;
            if (k.other_mode == 1) {
                const float *ocp = other_controls + (size_t)(c * k.H + t) * 2 * Bo + (Bo == 1 ? 0 : b);
                oa = ocp[0];
                oo = ocp[Bo];
            }
            other_model_step<true>(os[c][0], os[c][1], os[c][2], os[c][3], k.other_mode == 1, oa, oo, k.dt, k.dt2);
        }
        // features at the new state (merging.py:51-83)
        {
            const HD e = v * hd_sin(th) - k.ts;
            const HD e2 = e * e;
            phi_sum[0] = phi_sum[0] + (e2.v <= k.bound ? e2 : hd_const(k.bound));
        }
        HD fmin = hd_const(0.0f);
        for (int l = 0; l < k.L; ++l) {
            const HD d = x - k.lane_x[l];
            const HD f = (d * d) * 10.0f;
            phi_sum[1 + l] = phi_sum[1 + l] + f;
            if (l == 0 || f.v < fmin.v) fmin = f;
        }
        HD best = hd_const(0.0f);
        for (int c = 0; c < k.NO; ++c) {
            const HD val = hd_bump(x, os[c][0], OCD_BUMP_HX) * hd_bump(y, os[c][1], OCD_BUMP_HY);
            if (c == 0 || val.v > best.v) best = val;
        }
        const HD ax = x.v < 0.0f ? -x : x;
        const HD fence = (hd_threshold(k, x) + hd_threshold(k, -x)) * ax;
#pragma unroll
        for (int l = 1; l <= OCD_MAX_LANES; ++l)      // static indices: the sums stay in registers
            if (l == k.L) {
                phi_sum[1 + l] = phi_sum[1 + l] + fmin;
                if (l + 2 < OCD_MAX_LANES + 4) phi_sum[2 + l] = phi_sum[2 + l] + best;
                if (l + 3 < OCD_MAX_LANES + 4) phi_sum[3 + l] = phi_sum[3 + l] + fence;
            }
    }
#pragma unroll
    for (int q = 0; q < OCD_MAX_LANES + 4; ++q)
        if (q < k.K) {
            hess[((size_t)(q * n + i) * n + j) * B + b] = phi_sum[q].ab;
            hess[((size_t)(q * n + j) * n + i) * B + b] = phi_sum[q].ab;
        }
}
#endif

}  // namespace ocd
