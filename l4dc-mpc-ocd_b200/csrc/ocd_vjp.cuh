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
//
// The second half of the file is the reverse pass through whole episodes (ocd_episode_vjp_batch): the same recompute
// phase and reverse sweep per (world, step), seeded on the applied control, then the robot's adjoint along the episode
// (see k_episode_vjp below).  The file ends with the implicit-function derivative of the L-BFGS plan
// (ocd_solve_implicit_vjp_batch: k_solve_implicit_vjp), built from the same forward-over-reverse sweep.
#pragma once

#include <cfloat>

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

// One forward-over-reverse sweep at the controls u ([2H], flat index 2t + c) along the direction d ([2H]): hv gets
// the Hessian-vector product M H M d (zero on the clipped controls), and with GRADS wbar [K], s0bar [4] (robot) and
// obar [H][NO][2] (the other cars' predicted positions) gain scale * the gradients of G(u) . M d with respect to the
// weights, the robot's initial state and the predicted positions.  oth: the predicted positions [H][NO][2] (precise).
template <bool GRADS>
__device__ __forceinline__ void vjp_hvp(const KParams &k, const float *w, int ws, const float (&s0)[4],
                                        const float *oth, const float *u, const float *d, float *hv, float scale,
                                        float *wbar, float *s0bar, float *obar) {
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
        const float acd = in_a ? d[2 * t] : 0.0f, ocd = in_w ? d[2 * t + 1] : 0.0f;
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
        if constexpr (GRADS) {
#pragma unroll
            for (int q = 0; q < kVjpK; ++q)
                if (q < k.K) wbar[q] = fmaf(scale, phid[q], wbar[q]);
            for (int c = 0; c < 2 * k.NO; ++c)
                obar[(size_t)t * k.NO * 2 + c] = fmaf(scale, gd[4 + c], obar[(size_t)t * k.NO * 2 + c]);
        }
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
        hv[2 * t] = ((a >= -8.0f) && (a <= 4.0f)) ? ltd : 0.0f;
        hv[2 * t + 1] = (fabsf(om) <= 4.0f) ? k.dt * mthd : 0.0f;
    }
    if constexpr (GRADS) {
        s0bar[0] = fmaf(scale, lxd, s0bar[0]);
        s0bar[1] = fmaf(scale, lyd, s0bar[1]);
        s0bar[2] = fmaf(scale, lvd, s0bar[2]);
        s0bar[3] = fmaf(scale, lthd, s0bar[3]);
    }
}

// One iteration of the reverse pass at the iterate u = u^n: on entry ubar holds ubar^{n+1}, on exit
// ubar^n = ubar^{n+1} + lr M H M ubar^{n+1}; wbar, s0bar and obar gain lr * grad phi_n.
__device__ __forceinline__ void vjp_iteration(const KParams &k, const float *w, int ws, const float (&s0)[4],
                                              const float *oth, const float *u, float *ubar, float *wbar,
                                              float *s0bar, float *obar) {
    float hv[2 * OCD_MAX_H];
    vjp_hvp<true>(k, w, ws, s0, oth, u, ubar, hv, k.lr, wbar, s0bar, obar);
    for (int t = 0; t < k.H; ++t) {
        const float a = u[2 * t], om = u[2 * t + 1];
        if ((a >= -8.0f) && (a <= 4.0f)) ubar[2 * t] = fmaf(k.lr, hv[2 * t], ubar[2 * t]);
        if (fabsf(om) <= 4.0f) ubar[2 * t + 1] = fmaf(k.lr, hv[2 * t + 1], ubar[2 * t + 1]);
    }
}

// Where the planner's model of the other cars takes its known controls from (other_mode == 1): a solve's
// other_controls [NO][H][2][Bo], or an episode's scenario -- k_episode's model, written out per car into buf [H][2]:
// a fixed-plan car's plan replayed from index 0 and then its control (quirk Q4), zero for every other car.
struct OtherControls {
    const float *table;            // [NO][H][2][Bo] or null
    long long    Bo;
    const ocd_scenario *sc;        // episodes (table null)
    __device__ __forceinline__ const float *car(const KParams &k, int j, long long b, float *buf, long long &ocs) const {
        ocs = 0;
        if (k.other_mode != 1) return nullptr;
        if (sc) {
            for (int t = 0; t < k.H; ++t) {
                float oa = 0.0f, oo = 0.0f;
                if (sc->kind[j] == 1) {
                    const bool in_plan = t < sc->plan_len[j];
                    oa = in_plan ? sc->plan[j][t][0] : sc->control[j][0];
                    oo = in_plan ? sc->plan[j][t][1] : sc->control[j][1];
                }
                buf[2 * t] = oa;
                buf[2 * t + 1] = oo;
            }
            ocs = 1;
            return buf;
        }
        ocs = Bo;
        return table + (size_t)j * k.H * 2 * Bo + (Bo == 1 ? 0 : b);
    }
};

// The other cars' predicted positions [H][NO][2] in precise arithmetic (the reverse pass's own copy of the slab).
__device__ __forceinline__ void vjp_predict_others(const KParams &k, const float *world, long long B, long long b,
                                                   const OtherControls &ocs_src, float *oth) {
    float buf[2 * OCD_MAX_H];
    for (int j = 0; j < k.NO; ++j) {
        const float *st = world + (size_t)(j + 1) * 4 * B + b;
        long long ocs;
        const float *oc = ocs_src.car(k, j, b, buf, ocs);
        predict_other<true>(k, st[0], st[B], st[2 * B], st[3 * B], oc, ocs, oth, j, 1);
    }
}

// The other cars' rows of world_bar [C][4][B]: obar [H][NO][2], the gradient with respect to the predicted positions,
// chained through the prediction model (naive_planner.py:53-66; known controls or constant velocity) in forward
// mode, one seed per component of car j's initial state.
__device__ __forceinline__ void vjp_chain_others(const KParams &k, const float *world, long long B, long long b,
                                                 const OtherControls &ocs_src, const float *obar, float *world_bar) {
    const int H = k.H, NO = k.NO;
    float buf[2 * OCD_MAX_H];
    for (int j = 0; j < NO; ++j) {
        const float *st = world + (size_t)(j + 1) * 4 * B + b;
        long long ocs;
        const float *oc = ocs_src.car(k, j, b, buf, ocs);
        for (int q = 0; q < 4; ++q) {
            float x = st[0], y = st[B], v = st[2 * B], th = st[3 * B];
            float xd = q == 0, yd = q == 1, vd = q == 2, thd = q == 3;
            float acc = 0.0f;
            for (int t = 0; t < H; ++t) {
                const float sn = sinf(th), cs = cosf(th);
                if (oc) {
                    const float oa = oc[(size_t)(t * 2 + 0) * ocs], oo = oc[(size_t)(t * 2 + 1) * ocs];
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
            world_bar[(size_t)((j + 1) * 4 + q) * B + b] = acc;
        }
    }
}

// The reverse pass over the stored iterates of one problem (it: u^0 .. u^{N-1} at element stride B, offset to the
// problem).  On entry ubar holds plan_bar and wbar [K], s0bar [4], obar [H][NO][2] are zero; on exit wbar and s0bar
// hold the VJP with respect to the weights and the robot's initial state -- the extra-init starts' dependence on the
// speed included when the start was built from v0 -- and obar that with respect to the predicted positions.
__device__ __forceinline__ void vjp_sweep(const KParams &k, const float *w, int ws, const float (&s0)[4],
                                          const float *oth, const float *it, long long B, int s, bool speed_is_v0,
                                          float *ubar, float *wbar, float *s0bar, float *obar) {
    const int H = k.H;
    float u[2 * OCD_MAX_H];
    for (int n = k.n_iter - 1; n >= 0; --n) {
        for (int i = 0; i < 2 * H; ++i) u[i] = it[((size_t)n * 2 * H + i) * B];
        vjp_iteration(k, w, ws, s0, oth, u, ubar, wbar, s0bar, obar);
    }
    // the start: a0 = friction * cur_speed^2 for the extra-init starts (naive_planner.py:114-116), cur_speed = v0
    if (s >= 3 && speed_is_v0) {
        float sa = 0.0f;
        for (int t = 0; t < H; ++t) sa += ubar[2 * t];
        s0bar[2] = fmaf(sa, 2.0f * k.mu * s0[2], s0bar[2]);
    }
}

// The reverse pass of problem b (start s, iterates already in the workspace); writes weights_bar and world_bar.
static __device__ __noinline__ void vjp_reverse(const KParams &k, const VjpArgs &a, long long b, int s) {
    const long long B = a.B;
    const int H = k.H, NO = k.NO;
    const OtherControls ocs_src{a.other_controls, a.Bo, nullptr};
    float oth[OCD_MAX_H * OCD_MAX_OTHER * 2], obar[OCD_MAX_H * OCD_MAX_OTHER * 2];
    vjp_predict_others(k, a.world, B, b, ocs_src, oth);
    for (int i = 0; i < H * NO * 2; ++i) obar[i] = 0.0f;
    const float s0[4] = {a.world[b], a.world[B + b], a.world[2 * B + b], a.world[3 * B + b]};
    const float *w = a.weights + weight_column(a.weight_idx, a.Bw, b);
    const int ws = (int)a.Bw;
    float ubar[2 * OCD_MAX_H], wbar[kVjpK], s0bar[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    for (int i = 0; i < 2 * H; ++i) ubar[i] = a.plan_bar[(size_t)i * B + b];
#pragma unroll
    for (int q = 0; q < kVjpK; ++q) wbar[q] = 0.0f;
    vjp_sweep(k, w, ws, s0, oth, a.iters + b, B, s, !a.cur_speed, ubar, wbar, s0bar, obar);
#pragma unroll
    for (int q = 0; q < kVjpK; ++q)
        if (q < k.K) a.weights_bar[(size_t)q * B + b] = wbar[q];
    if (!a.world_bar) return;
    for (int q = 0; q < 4; ++q) a.world_bar[(size_t)q * B + b] = s0bar[q];
    vjp_chain_others(k, a.world, B, b, ocs_src, obar, a.world_bar);
}

// Phase 1 of both reverse kernels: re-run start s of problem b (world [C][4][B], weights w with stride ws, the start
// built from `speed`) with the iteration code k_solve / k_episode run for this specialisation (HT, NOT_, LT, PRECISE):
// the register-resident sweep (sgd_iteration), the medium-horizon one (sgd_iteration_q) or the segmented adjoint
// (sgd_iteration_seg), with the same other-car slab; their per-thread buffers live in local memory here.  Stores
// u^0 .. u^{N-1} (and u^N with store_last) to it [N (+1)][H][2] at element stride B; dead threads (live false) run
// along without storing.
template <int HT, int NOT_, int LT, bool PRECISE>
__device__ __forceinline__ void vjp_recompute(const KParams &k, const float *world, long long B, long long b, bool live,
                                              const OtherControls &ocs_src, const float *w, int ws, int s, float speed,
                                              float *it, bool store_last) {
    constexpr bool SEGK = (HT == 0) || OCD_IS_SEGC(HT, NOT_);
    constexpr bool QK = OCD_IS_Q(HT, NOT_) && !PRECISE;
    const bool lin = slab_is_linear(SEGK, PRECISE, k.other_mode, k.H, k.NO, QK);
    float oth[OCD_MAX_H * OCD_MAX_OTHER * 2];
    {
        float buf[2 * OCD_MAX_H];
        for (int j = 0; j < k.NO; ++j) {
            const float *st = world + (size_t)(j + 1) * 4 * B + b;
            long long ocs;
            const float *oc = ocs_src.car(k, j, b, buf, ocs);
            predict_other<PRECISE>(k, st[0], st[B], st[2 * B], st[3 * B], oc, ocs, oth, j, 1, lin);
        }
    }
    const GradW gw = make_gradw<LT>(k, w, ws);
    const float x0 = world[b], y0 = world[B + b], v0 = world[2 * B + b], th0 = world[3 * B + b];
    const int H = k.H;
    const int n_store = k.n_iter + (store_last ? 1 : 0);
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
        for (int n = 0; n < n_store; ++n) {
            if (live)
                for (int t = 0; t < H; ++t) {
                    it[((size_t)(n * H + t) * 2 + 0) * B] = us.acc(t);
                    it[((size_t)(n * H + t) * 2 + 1) * B] = us.ang(t);
                }
            if (n == k.n_iter) break;
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
        for (int n = 0; n < n_store; ++n) {
            if (live)
#pragma unroll
                for (int t = 0; t < HT; ++t) {
                    it[((size_t)(n * HT + t) * 2 + 0) * B] = u.ua[t];
                    it[((size_t)(n * HT + t) * 2 + 1) * B] = u.uw[t];
                }
            if (n == k.n_iter) break;
            if constexpr (QK) {
                if (lin) sgd_iteration_q<HT, NOT_, LT, 0, true>(k, gw, x0, y0, v0, th0, sn0, cs0, oth, 1, u, q, q2);
                else sgd_iteration_q<HT, NOT_, LT, 0, false>(k, gw, x0, y0, v0, th0, sn0, cs0, oth, 1, u, q, q2);
            } else {
                sgd_iteration<HT, NOT_, LT, PRECISE, true, 0>(k, gw, x0, y0, v0, th0, sn0, cs0, oth, 1, u, nullptr,
                                                              nullptr);
            }
        }
    }
}

template <int HT, int NOT_, int LT, bool PRECISE>
__global__ void __launch_bounds__(kVjpThreads) k_solve_vjp(const __grid_constant__ KParams k, const VjpArgs a) {
    const long long b_raw = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = b_raw < a.B;
    const long long b = live ? b_raw : a.B - 1;     // whole warps stay converged: the FAST feature code votes
    int s = a.best[b];
    s = s < 0 ? 0 : (s >= k.S ? k.S - 1 : s);
    const float speed = a.cur_speed ? a.cur_speed[b] : a.world[2 * a.B + b];
    vjp_recompute<HT, NOT_, LT, PRECISE>(k, a.world, a.B, b, live, OtherControls{a.other_controls, a.Bo, nullptr},
                                         a.weights + weight_column(a.weight_idx, a.Bw, b), (int)a.Bw, s, speed,
                                         a.iters + b, false);
    if (live) vjp_reverse(k, a, b, s);
}

template <int HT, int NOT_, int LT, bool PRECISE>
int launch_solve_vjp_t(const KParams &k, const VjpArgs &a, cudaStream_t st) {
    k_solve_vjp<HT, NOT_, LT, PRECISE><<<(unsigned)((a.B + kVjpThreads - 1) / kVjpThreads), kVjpThreads, 0, st>>>(k, a);
    return cuda_status();
}

// ---------------------------------------------------------------------------------------------
// k_episode_vjp: the reverse pass through whole episodes (ocd_episode_vjp_batch).
//
// For world b, k_episode runs t = 0 .. T-1: world_t (after the replanning teleport; traj_states[t]), the reward
// r_t = w_true . phi(world_t), the applied control u_t = pi(w, world_t) (the first control of the winning start
// traj_best[t], planned from the robot's speed and the planner's model of the scripted cars), and the simulator step
// s_{t+1} = f(s_t, clip(u_t)) of the robot.  The scripted cars depend on neither w nor the robot, so only the robot's
// 4-state adjoint lambda is carried backwards from lambda_T = 0:
//   ubar_t   = M_t (df/du)(s_t, u_t)^T lambda_{t+1}                      (M_t: the simulator's inclusive clip mask)
//   lambda_t = ret_bar grad_s r_t + (df/ds)^T lambda_{t+1} + J_s,t^T ubar_t
//   wbar    += J_w,t^T ubar_t
// with J_t = d u_t / d(w, s_t) the 2 x (K + 4) Jacobian of the applied control: the solve VJP of step t seeded one-hot
// on plan[0][0] and on plan[0][1].  Outputs: plan_weights_bar = wbar, robot_init_bar = lambda_0,
// true_weights_bar = ret_bar sum_t phi(world_t).
//
// The steps' Jacobians are independent, so k_episode_jac runs one thread per (world, step) -- the step on
// blockIdx.y -- and only the 4 x 4 chain is sequential (k_episode_adjoint, one thread per world).  k_episode_jac
// re-runs step t's winning start with k_episode's own iteration code and other-car model (the episode dispatch:
// OCD_DISPATCH, not the solve's compile-time horizons), stores u^0 .. u^N in the workspace -- u^N[0] is the applied
// control, bit for bit traj_controls[t] -- and writes J_t to the workspace rows [T][2][K + 4][B].  The iterate store
// ((N + 1) H 2 floats per world and step) bounds how many steps are in flight: the caller's workspace decides, from
// one step per launch to all T; the results do not depend on it.
// ---------------------------------------------------------------------------------------------
struct EpisodeVjpArgs {
    const float *plan_weights;     // [K][Bw]
    long long    Bw;
    const int32_t *weight_idx;     // [B] or null
    const float *true_weights;     // [K]
    int          T;
    int          t0;               // first step of this k_episode_jac launch
    const float *traj_states;      // [T][C][4][B]
    const int32_t *traj_best;      // [T][B]
    const float *traj_controls;    // [T][2][B]
    const float *returns_bar;      // [B]
    float       *plan_weights_bar; // [K][B]
    float       *robot_init_bar;   // [4][B] or null
    float       *true_weights_bar; // [K][B] or null
    float       *jac;              // [T][2][K + 4][B] workspace
    float       *iters;            // [steps in flight][N + 1][H][2][B] workspace
    long long    B;
};

// The two reverse sweeps of (world b, step t): J_t rows for the seeds plan[0][0] and plan[0][1].
static __device__ __noinline__ void episode_jac_reverse(const KParams &k, const ocd_scenario &sc,
                                                        const EpisodeVjpArgs &a, const float *world, const float *it,
                                                        long long b, int s, int t) {
    const long long B = a.B;
    const int H = k.H, NO = k.NO, KJ = k.K + 4;
    float oth[OCD_MAX_H * OCD_MAX_OTHER * 2], obar[OCD_MAX_H * OCD_MAX_OTHER * 2];
    vjp_predict_others(k, world, B, b, OtherControls{nullptr, 0, &sc}, oth);
    const float s0[4] = {world[b], world[B + b], world[2 * B + b], world[3 * B + b]};
    const float *w = a.plan_weights + weight_column(a.weight_idx, a.Bw, b);
    const int ws = (int)a.Bw;
    float *J = a.jac + (size_t)t * 2 * KJ * B + b;
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
        float ubar[2 * OCD_MAX_H], wbar[kVjpK], s0bar[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        for (int i = 0; i < 2 * H; ++i) ubar[i] = i == c ? 1.0f : 0.0f;
        for (int i = 0; i < H * NO * 2; ++i) obar[i] = 0.0f;
#pragma unroll
        for (int q = 0; q < kVjpK; ++q) wbar[q] = 0.0f;
        vjp_sweep(k, w, ws, s0, oth, it, B, s, true, ubar, wbar, s0bar, obar);
#pragma unroll
        for (int q = 0; q < kVjpK; ++q)
            if (q < k.K) J[(size_t)(c * KJ + q) * B] = wbar[q];
        for (int q = 0; q < 4; ++q) J[(size_t)(c * KJ + k.K + q) * B] = s0bar[q];
    }
}

template <int HT, int NOT_, int LT, bool PRECISE>
__global__ void __launch_bounds__(kVjpThreads)
k_episode_jac(const __grid_constant__ KParams k, const __grid_constant__ ocd_scenario sc, const EpisodeVjpArgs a) {
    const long long b_raw = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = b_raw < a.B;
    const long long b = live ? b_raw : a.B - 1;     // whole warps stay converged: the FAST feature code votes
    const long long B = a.B;
    const int t = a.t0 + (int)blockIdx.y;
    const float *world = a.traj_states + (size_t)t * (k.NO + 1) * 4 * B;
    int s = a.traj_best[(size_t)t * B + b];
    s = s < 0 ? 0 : (s >= k.S ? k.S - 1 : s);
    float *it = a.iters + (size_t)blockIdx.y * (k.n_iter + 1) * k.H * 2 * B + b;
    // k_episode plans from the robot's own speed (cur_speed = v0)
    vjp_recompute<HT, NOT_, LT, PRECISE>(k, world, B, b, live, OtherControls{nullptr, 0, &sc},
                                         a.plan_weights + weight_column(a.weight_idx, a.Bw, b), (int)a.Bw, s,
                                         world[2 * B + b], it, true);
    if (live) episode_jac_reverse(k, sc, a, world, it, b, s, t);
}

// k_episode_jac over the T steps, `group` steps per launch (1 .. T; the iterate store holds `group` steps)
template <int HT, int NOT_, int LT, bool PRECISE>
int launch_episode_jac_t(const KParams &k, const ocd_scenario &sc, const EpisodeVjpArgs &a, int group,
                         cudaStream_t st) {
    EpisodeVjpArgs g = a;
    for (int t0 = 0; t0 < a.T; t0 += group) {
        g.t0 = t0;
        const dim3 grid((unsigned)((a.B + kVjpThreads - 1) / kVjpThreads), (unsigned)(a.T - t0 < group ? a.T - t0 : group));
        k_episode_jac<HT, NOT_, LT, PRECISE><<<grid, kVjpThreads, 0, st>>>(k, sc, g);
        const int rc = cuda_status();
        if (rc) return rc;
    }
    return OCD_OK;
}

#ifndef OCD_HD_ONLY   // built once, by ocd_api.cu
// The sequential part: one thread per world walks t = T-1 .. 0 with lambda and wbar in registers (precise arithmetic).
// T = 0 writes zeros.
__global__ void __launch_bounds__(kVjpThreads) k_episode_adjoint(const __grid_constant__ KParams k, const EpisodeVjpArgs a) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    const long long B = a.B;
    const int C = k.NO + 1, KJ = k.K + 4;
    const float rb = a.T > 0 ? a.returns_bar[b] : 0.0f;
    float lam[4] = {0.0f, 0.0f, 0.0f, 0.0f}, wbar[kVjpK], tbar[kVjpK], wt[kVjpK];
#pragma unroll
    for (int q = 0; q < kVjpK; ++q) {
        wbar[q] = tbar[q] = 0.0f;
        wt[q] = q < k.K ? a.true_weights[q] : 0.0f;
    }
    for (int t = a.T - 1; t >= 0; --t) {
        const float *st = a.traj_states + (size_t)t * C * 4 * B + b;
        const float x = st[0], y = st[B], v = st[2 * B], th = st[3 * B];
        // the simulator step (dynamics_step with the robot's friction; clip masks inclusive, simulation_utils.py:9-21)
        const float ua = a.traj_controls[(size_t)(2 * t) * B + b], uw = a.traj_controls[(size_t)(2 * t + 1) * B + b];
        const float ac = fmaxf(fminf(ua, 4.0f), -8.0f);
        const float sn = sinf(th), cs = cosf(th);
        const float total = ac - k.mu * (v * v);
        const float dist = v * k.dt + k.hdt2 * total;
        const float ld = cs * lam[0] + sn * lam[1];               // adjoint of the step length
        const float lt = k.hdt2 * ld + k.dt * lam[2];             // adjoint of the clipped acceleration
        const float ub0 = (ua >= -8.0f && ua <= 4.0f) ? lt : 0.0f;
        const float ub1 = fabsf(uw) <= 4.0f ? k.dt * lam[3] : 0.0f;
        float nl[4] = {lam[0], lam[1], lam[2] + k.dt * ld - 2.0f * k.mu * v * lt, lam[3] + dist * (cs * lam[1] - sn * lam[0])};
        // through the planner: u_t = pi(w, s_t)
        const float *J = a.jac + (size_t)t * 2 * KJ * B + b;
#pragma unroll
        for (int q = 0; q < kVjpK; ++q)
            if (q < k.K) wbar[q] = fmaf(ub0, J[(size_t)q * B], fmaf(ub1, J[(size_t)(KJ + q) * B], wbar[q]));
        for (int i = 0; i < 4; ++i)
            nl[i] = fmaf(ub0, J[(size_t)(k.K + i) * B], fmaf(ub1, J[(size_t)(KJ + k.K + i) * B], nl[i]));
        // the reward of world_t, the other cars where they are
        HD ox[OCD_MAX_OTHER], oy[OCD_MAX_OTHER];
        for (int c = 0; c < k.NO; ++c) {
            ox[c] = hd_const(st[(size_t)((c + 1) * 4) * B]);
            oy[c] = hd_const(st[(size_t)((c + 1) * 4 + 1) * B]);
        }
        for (int i = 0; i < 4; ++i) {
            HD phi[kVjpK];
            hd_features(k, HD{x, i == 0 ? 1.0f : 0.0f, 0.0f, 0.0f}, HD{y, i == 1 ? 1.0f : 0.0f, 0.0f, 0.0f},
                        HD{v, i == 2 ? 1.0f : 0.0f, 0.0f, 0.0f}, HD{th, i == 3 ? 1.0f : 0.0f, 0.0f, 0.0f}, ox, oy, phi);
            float g = 0.0f;
#pragma unroll
            for (int q = 0; q < kVjpK; ++q)
                if (q < k.K) {
                    g = fmaf(wt[q], phi[q].a, g);
                    if (i == 0) tbar[q] = fmaf(rb, phi[q].v, tbar[q]);
                }
            nl[i] = fmaf(rb, g, nl[i]);
        }
        for (int i = 0; i < 4; ++i) lam[i] = nl[i];
    }
#pragma unroll
    for (int q = 0; q < kVjpK; ++q)
        if (q < k.K) {
            a.plan_weights_bar[(size_t)q * B + b] = wbar[q];
            if (a.true_weights_bar) a.true_weights_bar[(size_t)q * B + b] = tbar[q];
        }
    if (a.robot_init_bar)
        for (int i = 0; i < 4; ++i) a.robot_init_bar[(size_t)i * B + b] = lam[i];
}
// ---------------------------------------------------------------------------------------------
// k_solve_implicit_vjp: the implicit-function derivative of the L-BFGS plan (ocd_solve_implicit_vjp_batch).
//
// k_solve_lbfgs returns a stationary point u* of R: with A the controls inside the inclusive clip box at u* (the
// forward's masks) and G = dR/du (zero on the clipped controls), G_A(u*; theta) = 0 for theta = (w, s0).  The
// implicit function theorem gives du*_A/dtheta = -H_AA^{-1} dG_A/dtheta (H = dG/du) and du*_I/dtheta = 0 for the
// clipped controls I, so with z_A the solution of H_AA z_A = plan_bar_A (z_I = 0)
//   theta_bar = -grad_theta (G(u*; theta) . z).
// The line search, restarts and early breaks of the run that found u* do not enter, and neither do the start it began
// from nor cur_speed.  One thread per problem, precise arithmetic: |A| sweeps of vjp_hvp along the unit vectors of A
// give the columns of H_AA, which is symmetrised and solved in double with partial pivoting; a pivot that vanishes
// relative to the largest entry (below the float rounding of the entries) marks the problem singular and its
// weights_bar and world_bar are NaN.  One more sweep along z with scale -1 gives weights_bar, the robot's world_bar
// and obar, which vjp_chain_others carries to the other cars.  residual (optional) = max_A |G(u*)|, from the
// gradient code k_solve_lbfgs itself runs: the stationarity the derivative assumes.
// ---------------------------------------------------------------------------------------------
struct ImplicitVjpArgs {
    const float *world;            // [C][4][B]
    const float *other_controls;   // [NO][H][2][Bo] or null
    long long    Bo;
    const float *weights;          // [K][Bw]
    long long    Bw;
    const int32_t *weight_idx;     // [B] or null
    const float *plan;             // [H][2][B] (ocd_solve_batch's, optimizer 1)
    const float *plan_bar;         // [H][2][B]
    float       *weights_bar;      // [K][B]
    float       *world_bar;        // [C][4][B] or null
    float       *residual;         // [B] or null
    long long    B;
};

static constexpr int kImplicitN = 2 * OCD_LBFGS_MAX_H;

__global__ void __launch_bounds__(kVjpThreads) k_solve_implicit_vjp(const __grid_constant__ KParams k,
                                                                    const ImplicitVjpArgs a) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    const long long B = a.B;
    const int H = k.H, n = 2 * k.H;
    const OtherControls ocs_src{a.other_controls, a.Bo, nullptr};
    float oth[OCD_LBFGS_MAX_H * OCD_MAX_OTHER * 2], obar[OCD_LBFGS_MAX_H * OCD_MAX_OTHER * 2];
    vjp_predict_others(k, a.world, B, b, ocs_src, oth);
    for (int i = 0; i < H * k.NO * 2; ++i) obar[i] = 0.0f;
    const float s0[4] = {a.world[b], a.world[B + b], a.world[2 * B + b], a.world[3 * B + b]};
    const float *w = a.weights + weight_column(a.weight_idx, a.Bw, b);
    const int ws = (int)a.Bw;
    float u[kImplicitN], d[kImplicitN], hv[kImplicitN];
    int act[kImplicitN];
    int na = 0;
    for (int t = 0; t < H; ++t) {
        const float ua = a.plan[(size_t)(2 * t) * B + b], uw = a.plan[(size_t)(2 * t + 1) * B + b];
        u[2 * t] = ua;
        u[2 * t + 1] = uw;
        if ((ua >= -8.0f) && (ua <= 4.0f)) act[na++] = 2 * t;
        if (fabsf(uw) <= 4.0f) act[na++] = 2 * t + 1;
    }
    if (a.residual) {
        Traj<0> ut;
        float ga[OCD_MAX_H], go[OCD_MAX_H], sn0, cs0;
        for (int t = 0; t < H; ++t) {
            ut.ua[t] = u[2 * t];
            ut.uw[t] = u[2 * t + 1];
        }
        Mth<true>::sincos_(s0[3], sn0, cs0);
        sgd_iteration<0, 0, 0, true, false>(k, make_gradw<0>(k, w, ws), s0[0], s0[1], s0[2], s0[3], sn0, cs0, oth, 1,
                                            ut, ga, go);
        float r = 0.0f;
        for (int t = 0; t < H; ++t) r = fmaxf(r, fmaxf(fabsf(ga[t]), fabsf(go[t])));   // zero on the clipped controls
        a.residual[b] = r;
    }
    // H_AA, column by column, then symmetrised (row-major, n_A x n_A)
    double M[kImplicitN * kImplicitN], z[kImplicitN];
    for (int i = 0; i < n; ++i) d[i] = 0.0f;
    for (int j = 0; j < na; ++j) {
        d[act[j]] = 1.0f;
        vjp_hvp<false>(k, w, ws, s0, oth, u, d, hv, 0.0f, nullptr, nullptr, nullptr);
        d[act[j]] = 0.0f;
        for (int i = 0; i < na; ++i) M[i * na + j] = (double)hv[act[i]];
    }
    double scale = 0.0;
    for (int i = 0; i < na; ++i) {
        for (int j = 0; j < i; ++j) {
            const double m = 0.5 * (M[i * na + j] + M[j * na + i]);
            M[i * na + j] = M[j * na + i] = m;
        }
        for (int j = 0; j < na; ++j) scale = fmax(scale, fabs(M[i * na + j]));
        z[i] = (double)a.plan_bar[(size_t)act[i] * B + b];
    }
    // Gaussian elimination with partial pivoting.  The entries carry float rounding, so a pivot below na float ulps
    // of the largest entry cannot be told apart from zero: the reduced Hessian is singular there.
    const double tiny = (double)na * (double)FLT_EPSILON * scale;
    bool singular = false;
    for (int c = 0; c < na && !singular; ++c) {
        int piv = c;
        for (int r = c + 1; r < na; ++r)
            if (fabs(M[r * na + c]) > fabs(M[piv * na + c])) piv = r;
        if (!(fabs(M[piv * na + c]) > tiny)) {
            singular = true;
            break;
        }
        if (piv != c) {
            for (int j = c; j < na; ++j) {
                const double t = M[c * na + j]; M[c * na + j] = M[piv * na + j]; M[piv * na + j] = t;
            }
            const double t = z[c]; z[c] = z[piv]; z[piv] = t;
        }
        for (int r = c + 1; r < na; ++r) {
            const double f = M[r * na + c] / M[c * na + c];
            for (int j = c + 1; j < na; ++j) M[r * na + j] -= f * M[c * na + j];
            z[r] -= f * z[c];
        }
    }
    if (singular) {
        const float nan = __int_as_float(0x7fffffff);
        for (int q = 0; q < k.K; ++q) a.weights_bar[(size_t)q * B + b] = nan;
        if (a.world_bar)
            for (int q = 0; q < (k.NO + 1) * 4; ++q) a.world_bar[(size_t)q * B + b] = nan;
        return;
    }
    for (int r = na - 1; r >= 0; --r) {
        double acc = z[r];
        for (int j = r + 1; j < na; ++j) acc -= M[r * na + j] * z[j];
        z[r] = acc / M[r * na + r];
    }
    // theta_bar = -grad_theta (G . z): one sweep along z with scale -1
    for (int i = 0; i < na; ++i) d[act[i]] = (float)z[i];
    float wbar[kVjpK], s0bar[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int q = 0; q < kVjpK; ++q) wbar[q] = 0.0f;
    vjp_hvp<true>(k, w, ws, s0, oth, u, d, hv, -1.0f, wbar, s0bar, obar);
#pragma unroll
    for (int q = 0; q < kVjpK; ++q)
        if (q < k.K) a.weights_bar[(size_t)q * B + b] = wbar[q];
    if (!a.world_bar) return;
    for (int q = 0; q < 4; ++q) a.world_bar[(size_t)q * B + b] = s0bar[q];
    vjp_chain_others(k, a.world, B, b, ocs_src, obar, a.world_bar);
}
#endif

}  // namespace ocd
