// ocd_vjp.cuh -- the reverse pass through the fixed-budget SGD solve: ocd_solve_vjp_batch.
//
// For one problem the planner runs the start s it finally picks as (naive_planner.py:107-164)
//   u^0 = start_s,   u^{n+1} = u^n + lr G(u^n; w, s0)   (n = 0 .. N-1),   plan = u^N
// with G = dR/du under TensorFlow's conventions (clip masks, min / max selections: sgd_iteration in ocd_device.cuh) and
// s0 the whole initial world [C][4] -- the other cars through the planner's prediction of them (predict_other).  The
// argmin over starts is piecewise constant and is not differentiated; clip masks and selections have zero derivative
// almost everywhere.  Given plan_bar = ubar^N, the vector-Jacobian product walks the iterations backwards:
//   phi_n(u, w, s0) = G(u; w, s0) . ubar^{n+1}
//   wbar += lr grad_w phi_n,   s0bar += lr grad_s0 phi_n,   ubar^n = ubar^{n+1} + lr grad_u phi_n
// and at the end adds the start's dependence on the robot's speed (a0 = friction v0^2 of the extra-init starts, when
// cur_speed is NULL).
//
// phi_n is the derivative of R along the masked direction d = M ubar^{n+1} of the clipped controls, so all three
// gradients come from one forward-over-reverse sweep at u^n: the rollout in dual numbers (value, tangent along d), then
// sgd_iteration's closed-form adjoint in dual numbers.  The tangent of the adjoint at control t is grad_u phi (the
// Hessian-vector product M H M ubar), at the initial robot state grad_s0 phi, and the tangent of sum_t phi(s_{t+1}) is
// grad_w phi (R is linear in w).  The feature gradient at a state and its tangent -- a state-Hessian-vector product --
// come from ocd_hessian.cuh's hyper-dual numbers: e1 on one state component (or one coordinate of another car's predicted
// position), e2 on the tangent state.  The predicted positions do not depend on the controls: their gradients are
// summed per (car, step) over all iterations and chained through the prediction model once, at the end.
//
// One thread per problem.  It first re-runs the winning start with the forward's own iteration code -- the same
// specialisation (horizon, car count, lanes) and math mode as ocd_solve_batch, so the derivative is taken along the
// trajectory the forward produced, bit for bit -- and stores u^0 .. u^{N-1} in the caller's workspace [N][H][2][B]
// (thread b touches element b).  The reverse pass then reads them back in reverse order; it runs in precise arithmetic
// (libdevice sin / cos / exp, IEEE division) whatever the math mode, like the Hessian and L-BFGS kernels.  Outputs are
// per problem, weights_bar [K][B] and world_bar [C][4][B]: no reduction across problems, no atomics.
#pragma once

#include "ocd_kernels.cuh"
#include "ocd_hessian.cuh"

namespace ocd {

struct VjpArgs {
    const float *world;            // [C][4][B]
    const float *other_controls;   // [NO][H][2][Bo] or null
    long long    Bo;
    const float *weights;          // [K][Bw]
    long long    Bw;
    const int32_t *weight_idx;     // [B] or null
    const float *cur_speed;        // [B] or null
    const int32_t *best;           // [B] (ocd_solve_batch's)
    const float *plan_bar;         // [H][2][B]
    float       *weights_bar;      // [K][B]
    float       *world_bar;        // [C][4][B] or null
    float       *iters;            // [n_iter][H][2][B] workspace
    long long    B;
};

static constexpr int kVjpThreads = 128;
static constexpr int kVjpK = OCD_MAX_LANES + 4;

// smooth_bump(c - hw, c + hw)(z) with the centre c a hyper-dual number as well (an other car's predicted position)
__device__ __forceinline__ HD hd_bump_at(HD z, HD c, float hw) {
    const float start = __fsub_rn(c.v, hw), end = __fadd_rn(c.v, hw);
    const float width = __fmul_rn(__fsub_rn(end, start), 0.5f), center = __fmul_rn(__fadd_rn(start, end), 0.5f);
    const HD n = (z - HD{center, c.a, c.b, c.ab}) * __fdiv_rn(1.0f, width);
    if (n.v * n.v < 1.0f) {
        const HD om = hd_const(1.0f) - n * n;
        return hd_exp(hd_const(1.0f) - hd_rcp(om));
    }
    return hd_const(0.0f);
}

// The K features at one state (merging.py:51-83; k_feature_hessian's formulas), other car c at (ox[c], oy[c]).
__device__ __forceinline__ void hd_features(const KParams &k, HD x, HD y, HD v, HD th, const HD *ox, const HD *oy,
                                            HD (&phi)[kVjpK]) {
    {
        const HD e = v * hd_sin(th) - k.ts;
        const HD e2 = e * e;
        phi[0] = e2.v <= k.bound ? e2 : hd_const(k.bound);
    }
    HD fmin = hd_const(0.0f);
#pragma unroll
    for (int l = 0; l < OCD_MAX_LANES; ++l)
        if (l < k.L) {
            const HD d = x - k.lane_x[l];
            const HD f = (d * d) * 10.0f;
            phi[1 + l] = f;
            if (l == 0 || f.v < fmin.v) fmin = f;
        }
    HD best = hd_const(0.0f);
    for (int c = 0; c < k.NO; ++c) {
        const HD val = hd_bump_at(x, ox[c], OCD_BUMP_HX) * hd_bump_at(y, oy[c], OCD_BUMP_HY);
        if (c == 0 || val.v > best.v) best = val;
    }
    const HD ax = x.v < 0.0f ? -x : x;
    const HD fence = (hd_threshold(k, x) + hd_threshold(k, -x)) * ax;
#pragma unroll
    for (int l = 1; l <= OCD_MAX_LANES; ++l)      // static indices: phi stays in registers
        if (l == k.L) {
            phi[1 + l] = fmin;
            if (l + 2 < kVjpK) phi[2 + l] = best;
            if (l + 3 < kVjpK) phi[3 + l] = fence;
        }
}

// At the state s (tangent sd along the direction of the sweep), other cars at op[2c], op[2c + 1]:
//   g[i]  = d(w . phi)/d z_i      z = (x, y, v, th, ox_0, oy_0, ox_1, ...)
//   gd[i] = its tangent           (sum_j d^2(w . phi)/dz_i ds_j sd_j)
//   phid[q] = tangent of feature q
// One hyper-dual evaluation per component: e1 on z_i, e2 on the tangent state.
__device__ __forceinline__ void grad_and_tangent(const KParams &k, const float *w, int ws, const float (&s)[4],
                                                 const float (&sd)[4], const float *op, float *g, float *gd,
                                                 float (&phid)[kVjpK]) {
    const int nz = 4 + 2 * k.NO;
    HD ox[OCD_MAX_OTHER], oy[OCD_MAX_OTHER];
    for (int i = 0; i < nz; ++i) {
        const HD x{s[0], i == 0 ? 1.0f : 0.0f, sd[0], 0.0f}, y{s[1], i == 1 ? 1.0f : 0.0f, sd[1], 0.0f};
        const HD v{s[2], i == 2 ? 1.0f : 0.0f, sd[2], 0.0f}, th{s[3], i == 3 ? 1.0f : 0.0f, sd[3], 0.0f};
        for (int c = 0; c < k.NO; ++c) {
            ox[c] = HD{op[2 * c], i == 4 + 2 * c ? 1.0f : 0.0f, 0.0f, 0.0f};
            oy[c] = HD{op[2 * c + 1], i == 5 + 2 * c ? 1.0f : 0.0f, 0.0f, 0.0f};
        }
        HD phi[kVjpK];
        hd_features(k, x, y, v, th, ox, oy, phi);
        float ga = 0.0f, gab = 0.0f;
#pragma unroll
        for (int q = 0; q < kVjpK; ++q)
            if (q < k.K) {
                const float wq = w[(size_t)q * ws];
                ga = fmaf(wq, phi[q].a, ga);
                gab = fmaf(wq, phi[q].ab, gab);
                if (i == 0) phid[q] = phi[q].b;
            }
        g[i] = ga;
        gd[i] = gab;
    }
}

// One iteration of the reverse pass at the iterate u = u^n ([2H], flat index 2t + c).  On entry ubar holds ubar^{n+1},
// on exit ubar^n; wbar [K], s0bar [4] (robot) and obar [H][NO][2] (the other cars' predicted positions) gain
// lr * grad phi_n.  oth: the predicted positions [H][NO][2] (precise).
__device__ __forceinline__ void vjp_iteration(const KParams &k, const float *w, int ws, const float (&s0)[4],
                                              const float *oth, const float *u, float *ubar, float *wbar,
                                              float *s0bar, float *obar) {
    const int H = k.H;
    float S[OCD_MAX_H + 1][4], Sd[OCD_MAX_H + 1][4], D[OCD_MAX_H], Dd[OCD_MAX_H];
    for (int q = 0; q < 4; ++q) {
        S[0][q] = s0[q];
        Sd[0][q] = 0.0f;
    }
    // rollout in dual numbers, tangent d = M ubar on the clipped controls (simulation_utils.py:9-21)
    for (int t = 0; t < H; ++t) {
        const float a = u[2 * t], om = u[2 * t + 1];
        const bool in_a = (a >= -8.0f) && (a <= 4.0f), in_w = fabsf(om) <= 4.0f;
        const float ac = fmaxf(fminf(a, 4.0f), -8.0f), oc = fmaxf(fminf(om, 4.0f), -4.0f);
        const float acd = in_a ? ubar[2 * t] : 0.0f, ocd = in_w ? ubar[2 * t + 1] : 0.0f;
        const float x = S[t][0], y = S[t][1], v = S[t][2], th = S[t][3];
        const float xd = Sd[t][0], yd = Sd[t][1], vd = Sd[t][2], thd = Sd[t][3];
        const float sn = sinf(th), cs = cosf(th), snd = cs * thd, csd = -sn * thd;
        const float total = ac - k.mu * (v * v), totd = acd - 2.0f * k.mu * v * vd;
        const float dist = v * k.dt + k.hdt2 * total, distd = vd * k.dt + k.hdt2 * totd;
        S[t + 1][0] = x + cs * dist;
        S[t + 1][1] = y + sn * dist;
        S[t + 1][2] = v + total * k.dt;
        S[t + 1][3] = th + oc * k.dt;
        Sd[t + 1][0] = xd + csd * dist + cs * distd;
        Sd[t + 1][1] = yd + snd * dist + sn * distd;
        Sd[t + 1][2] = vd + totd * k.dt;
        Sd[t + 1][3] = thd + ocd * k.dt;
        D[t] = dist;
        Dd[t] = distd;
    }
    // the closed-form adjoint (sgd_iteration) in dual numbers
    float lx = 0.0f, ly = 0.0f, lv = 0.0f, lth = 0.0f, lxd = 0.0f, lyd = 0.0f, lvd = 0.0f, lthd = 0.0f;
    float g[4 + 2 * OCD_MAX_OTHER], gd[4 + 2 * OCD_MAX_OTHER], phid[kVjpK];
    for (int t = H - 1; t >= 0; --t) {
        const float st[4] = {S[t + 1][0], S[t + 1][1], S[t + 1][2], S[t + 1][3]};
        const float sdt[4] = {Sd[t + 1][0], Sd[t + 1][1], Sd[t + 1][2], Sd[t + 1][3]};
        grad_and_tangent(k, w, ws, st, sdt, oth + (size_t)t * k.NO * 2, g, gd, phid);
#pragma unroll
        for (int q = 0; q < kVjpK; ++q)
            if (q < k.K) wbar[q] = fmaf(k.lr, phid[q], wbar[q]);
        for (int c = 0; c < 2 * k.NO; ++c) obar[(size_t)t * k.NO * 2 + c] = fmaf(k.lr, gd[4 + c], obar[(size_t)t * k.NO * 2 + c]);
        const float mx = g[0] + lx, my = g[1] + ly, mv = g[2] + lv, mth = g[3] + lth;
        const float mxd = gd[0] + lxd, myd = gd[1] + lyd, mvd = gd[2] + lvd, mthd = gd[3] + lthd;
        const float v = S[t][2], vd = Sd[t][2], th = S[t][3], thd = Sd[t][3];
        const float sn = sinf(th), cs = cosf(th), snd = cs * thd, csd = -sn * thd;
        const float ld = cs * mx + sn * my;                       // adjoint of the step length
        const float ldd = csd * mx + cs * mxd + snd * my + sn * myd;
        const float lt = k.hdt2 * ld + k.dt * mv;                 // adjoint of the clipped acceleration
        const float ltd = k.hdt2 * ldd + k.dt * mvd;
        const float cr = cs * my - sn * mx;
        const float crd = csd * my + cs * myd - snd * mx - sn * mxd;
        lv = mv + k.dt * ld - 2.0f * k.mu * v * lt;
        lvd = mvd + k.dt * ldd - 2.0f * k.mu * (vd * lt + v * ltd);
        lth = mth + D[t] * cr;
        lthd = mthd + Dd[t] * cr + D[t] * crd;
        lx = mx; ly = my; lxd = mxd; lyd = myd;
        const float a = u[2 * t], om = u[2 * t + 1];
        if ((a >= -8.0f) && (a <= 4.0f)) ubar[2 * t] = fmaf(k.lr, ltd, ubar[2 * t]);
        if (fabsf(om) <= 4.0f) ubar[2 * t + 1] = fmaf(k.lr, k.dt * mthd, ubar[2 * t + 1]);
    }
    s0bar[0] = fmaf(k.lr, lxd, s0bar[0]);
    s0bar[1] = fmaf(k.lr, lyd, s0bar[1]);
    s0bar[2] = fmaf(k.lr, lvd, s0bar[2]);
    s0bar[3] = fmaf(k.lr, lthd, s0bar[3]);
}

// The reverse pass of problem b (start s, iterates already in the workspace); writes weights_bar and world_bar.
static __device__ __noinline__ void vjp_reverse(const KParams &k, const VjpArgs &a, long long b, int s) {
    const long long B = a.B;
    const int H = k.H, NO = k.NO;
    float oth[OCD_MAX_H * OCD_MAX_OTHER * 2], obar[OCD_MAX_H * OCD_MAX_OTHER * 2];
    for (int j = 0; j < NO; ++j) {
        const float *st = a.world + (size_t)(j + 1) * 4 * B + b;
        const float *oc = nullptr;
        long long ocs = 0;
        if (k.other_mode == 1) {
            ocs = a.Bo;
            oc = a.other_controls + (size_t)j * H * 2 * a.Bo + (a.Bo == 1 ? 0 : b);
        }
        predict_other<true>(k, st[0], st[B], st[2 * B], st[3 * B], oc, ocs, oth, j, 1);
    }
    for (int i = 0; i < H * NO * 2; ++i) obar[i] = 0.0f;
    const float s0[4] = {a.world[b], a.world[B + b], a.world[2 * B + b], a.world[3 * B + b]};
    const float *w = a.weights + weight_column(a.weight_idx, a.Bw, b);
    const int ws = (int)a.Bw;
    float u[2 * OCD_MAX_H], ubar[2 * OCD_MAX_H], wbar[kVjpK], s0bar[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    for (int i = 0; i < 2 * H; ++i) ubar[i] = a.plan_bar[(size_t)i * B + b];
#pragma unroll
    for (int q = 0; q < kVjpK; ++q) wbar[q] = 0.0f;
    for (int n = k.n_iter - 1; n >= 0; --n) {
        for (int i = 0; i < 2 * H; ++i) u[i] = a.iters[((size_t)n * 2 * H + i) * B + b];
        vjp_iteration(k, w, ws, s0, oth, u, ubar, wbar, s0bar, obar);
    }
    // the start: a0 = friction * cur_speed^2 for the extra-init starts (naive_planner.py:114-116), cur_speed = v0
    if (s >= 3 && !a.cur_speed) {
        float sa = 0.0f;
        for (int t = 0; t < H; ++t) sa += ubar[2 * t];
        s0bar[2] = fmaf(sa, 2.0f * k.mu * s0[2], s0bar[2]);
    }
#pragma unroll
    for (int q = 0; q < kVjpK; ++q)
        if (q < k.K) a.weights_bar[(size_t)q * B + b] = wbar[q];
    if (!a.world_bar) return;
    for (int q = 0; q < 4; ++q) a.world_bar[(size_t)q * B + b] = s0bar[q];
    // other car j: obar through the prediction model (naive_planner.py:53-66) in forward mode, one seed per component
    for (int j = 0; j < NO; ++j) {
        const float *st = a.world + (size_t)(j + 1) * 4 * B + b;
        const float *oc = (k.other_mode == 1) ? a.other_controls + (size_t)j * H * 2 * a.Bo + (a.Bo == 1 ? 0 : b)
                                              : nullptr;
        for (int q = 0; q < 4; ++q) {
            float x = st[0], y = st[B], v = st[2 * B], th = st[3 * B];
            float xd = q == 0, yd = q == 1, vd = q == 2, thd = q == 3;
            float acc = 0.0f;
            for (int t = 0; t < H; ++t) {
                const float sn = sinf(th), cs = cosf(th);
                if (oc) {
                    const float oa = oc[(size_t)(t * 2 + 0) * a.Bo], oo = oc[(size_t)(t * 2 + 1) * a.Bo];
                    const float dist = v * k.dt + 0.5f * oa * k.dt2, distd = vd * k.dt;
                    x += cs * dist;
                    y += sn * dist;
                    xd += -sn * thd * dist + cs * distd;
                    yd += cs * thd * dist + sn * distd;
                    v += oa * k.dt;
                    th += oo * k.dt;
                } else {
                    x += cs * v * k.dt;
                    y += sn * v * k.dt;
                    xd += (cs * vd - sn * thd * v) * k.dt;
                    yd += (sn * vd + cs * thd * v) * k.dt;
                }
                acc = fmaf(obar[(size_t)(t * NO + j) * 2], xd, fmaf(obar[(size_t)(t * NO + j) * 2 + 1], yd, acc));
            }
            a.world_bar[(size_t)((j + 1) * 4 + q) * B + b] = acc;
        }
    }
}

// Phase 1 re-runs the winning start with the iteration code k_solve runs for this specialisation (HT, NOT_, LT,
// PRECISE): the register-resident sweep (sgd_iteration), the medium-horizon one (sgd_iteration_q) or the segmented
// adjoint (sgd_iteration_seg), with the same other-car slab; their per-thread buffers live in local memory here.
template <int HT, int NOT_, int LT, bool PRECISE>
__global__ void __launch_bounds__(kVjpThreads) k_solve_vjp(const __grid_constant__ KParams k, const VjpArgs a) {
    constexpr bool SEGK = (HT == 0) || OCD_IS_SEGC(HT, NOT_);
    constexpr bool QK = OCD_IS_Q(HT, NOT_) && !PRECISE;
    const long long b_raw = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = b_raw < a.B;
    const long long b = live ? b_raw : a.B - 1;     // whole warps stay converged: the FAST feature code votes
    const long long B = a.B;
    const bool lin = slab_is_linear(SEGK, PRECISE, k.other_mode, k.H, k.NO, QK);
    float oth[OCD_MAX_H * OCD_MAX_OTHER * 2];
    for (int j = 0; j < k.NO; ++j) {
        const float *st = a.world + (size_t)(j + 1) * 4 * B + b;
        const float *oc = nullptr;
        long long ocs = 0;
        if (k.other_mode == 1) {
            ocs = a.Bo;
            oc = a.other_controls + (size_t)j * k.H * 2 * a.Bo + (a.Bo == 1 ? 0 : b);
        }
        predict_other<PRECISE>(k, st[0], st[B], st[2 * B], st[3 * B], oc, ocs, oth, j, 1, lin);
    }
    const float *w = a.weights + weight_column(a.weight_idx, a.Bw, b);
    const GradW gw = make_gradw<LT>(k, w, (int)a.Bw);
    const float x0 = a.world[b], y0 = a.world[B + b], v0 = a.world[2 * B + b], th0 = a.world[3 * B + b];
    int s = a.best[b];
    s = s < 0 ? 0 : (s >= k.S ? k.S - 1 : s);
    const float speed = a.cur_speed ? a.cur_speed[b] : v0;
    const int H = k.H;
    float *it = a.iters + b;
    if constexpr (SEGK) {
        constexpr int HC = HT;
        constexpr bool FR = HC > 0 && OCD_SEGC_FR && !PRECISE;
        constexpr int SEGL = HC > 0 ? OCD_SEGC_SEG : kSeg;
        float2 ubuf[OCD_MAX_H];
        float4 ckbuf[(OCD_MAX_H + kSeg - 1) / kSeg];
        const SmemTraj us{reinterpret_cast<float *>(ubuf)};
        {
            const float a0 = (s >= 3) ? __fmul_rn(k.mu, __fmul_rn(speed, speed)) : 0.0f;
            const int m = s % 3;
            const float w0 = (m == 0) ? 0.0f : ((m == 1) ? -k.turn : k.turn);
            for (int t = 0; t < H; ++t) us.set(t, a0, w0);
        }
#pragma unroll 1
        for (int n = 0; n < k.n_iter; ++n) {
            if (live)
                for (int t = 0; t < H; ++t) {
                    it[((size_t)(n * H + t) * 2 + 0) * B] = us.acc(t);
                    it[((size_t)(n * H + t) * 2 + 1) * B] = us.ang(t);
                }
            if (!PRECISE && lin)
                sgd_iteration_seg<SEGL, NOT_, LT, PRECISE, !PRECISE, 0, HC, FR>(k, gw, x0, y0, v0, th0, oth, 1, us,
                                                                              reinterpret_cast<float *>(ckbuf));
            else
                sgd_iteration_seg<SEGL, NOT_, LT, PRECISE, false, 0, HC, FR>(k, gw, x0, y0, v0, th0, oth, 1, us,
                                                                           reinterpret_cast<float *>(ckbuf));
        }
    } else {
        Traj<HT> u;
        init_start<HT>(k, s, speed, u);
        float sn0, cs0;
        Mth<PRECISE>::sincos_(th0, sn0, cs0);
        float4 q[QK ? HT : 1];
        float2 q2[QK ? HT : 1];                      // entry t at index t (t = 1 .. HT-1 are used)
#pragma unroll 1
        for (int n = 0; n < k.n_iter; ++n) {
            if (live)
#pragma unroll
                for (int t = 0; t < HT; ++t) {
                    it[((size_t)(n * HT + t) * 2 + 0) * B] = u.ua[t];
                    it[((size_t)(n * HT + t) * 2 + 1) * B] = u.uw[t];
                }
            if constexpr (QK) {
                if (lin) sgd_iteration_q<HT, NOT_, LT, 0, true>(k, gw, x0, y0, v0, th0, sn0, cs0, oth, 1, u, q, q2);
                else sgd_iteration_q<HT, NOT_, LT, 0, false>(k, gw, x0, y0, v0, th0, sn0, cs0, oth, 1, u, q, q2);
            } else {
                sgd_iteration<HT, NOT_, LT, PRECISE, true, 0>(k, gw, x0, y0, v0, th0, sn0, cs0, oth, 1, u, nullptr,
                                                              nullptr);
            }
        }
    }
    if (live) vjp_reverse(k, a, b, s);
}

template <int HT, int NOT_, int LT, bool PRECISE>
int launch_solve_vjp_t(const KParams &k, const VjpArgs &a, cudaStream_t st) {
    k_solve_vjp<HT, NOT_, LT, PRECISE><<<(unsigned)((a.B + kVjpThreads - 1) / kVjpThreads), kVjpThreads, 0, st>>>(k, a);
    return cuda_status();
}

}  // namespace ocd
