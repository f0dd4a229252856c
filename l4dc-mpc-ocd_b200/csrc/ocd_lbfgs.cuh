// ocd_lbfgs.cuh -- the opt-in L-BFGS planner (params.optimizer == 1) outside the single solve: one (problem, start)
// of it as a device function (lbfgs_start, which k_solve_lbfgs in ocd_api.cu runs too), the receding-horizon episode
// with that planner (k_episode_lbfgs, ocd_episode_batch) and the implicit-function Jacobians of its applied controls
// (k_episode_jac_implicit, ocd_episode_implicit_vjp_batch).  Built once, by ocd_api.cu.
#pragma once

#include "ocd_kernels.cuh"
#include "ocd_vjp.cuh"

namespace ocd {

static constexpr int kLbfgsM = 4, kLbfgsLS = 6, kLbfgsN = 2 * OCD_LBFGS_MAX_H;

// f(u) = -R(u) and (g non-null) its gradient, precise math; weights w[q * ws], slab oth at element stride P
__device__ __forceinline__ float lbfgs_value_grad(const KParams &k, const GradW &gw, const float *wraw, int ws, float x0,
                                                  float y0, float v0, float th0, const float *oth, int P,
                                                  const float *uf, float *g /* null: value only */) {
    Traj<0> u;
    for (int t = 0; t < k.H; ++t) {
        u.ua[t] = uf[2 * t];
        u.uw[t] = uf[2 * t + 1];
    }
    const float f = -rollout_reward<0, 0, true>(k, wraw, ws, x0, y0, v0, th0, oth, P, u);
    if (g) {
        float ga[OCD_MAX_H], go[OCD_MAX_H], sn0, cs0;
        Mth<true>::sincos_(th0, sn0, cs0);
        sgd_iteration<0, 0, 0, true, false>(k, gw, x0, y0, v0, th0, sn0, cs0, oth, P, u, ga, go);
        for (int t = 0; t < k.H; ++t) {            // gradient of f = -R
            g[2 * t] = -ga[t];
            g[2 * t + 1] = -go[t];
        }
    }
    return f;
}

// One (problem, start) of the L-BFGS planner: start s built from `speed` (naive_planner.py:107-118), then L-BFGS on
// f(u) = -R(u): two-loop recursion over 4 correction pairs held in local memory, Armijo backtracking, gradient from
// the closed-form adjoint.  Leaves the plan in u [2H] (flat index 2t + c) and returns its loss f(u).  The CPU
// restatement used by the parity tests mirrors this loop statement for statement.
__device__ __forceinline__ float lbfgs_start(const KParams &k, const GradW &gw, const float *wraw, int ws, float x0,
                                             float y0, float v0, float th0, const float *oth, int P, int s, float speed,
                                             float (&u)[kLbfgsN]) {
    const int n = 2 * k.H;
    float g[kLbfgsN], gt[kLbfgsN], d[kLbfgsN], ut[kLbfgsN], q[kLbfgsN];
    float Sh[kLbfgsM][kLbfgsN], Yh[kLbfgsM][kLbfgsN], rho[kLbfgsM], al[kLbfgsM];
    {
        const float a0 = (s >= 3) ? __fmul_rn(k.mu, __fmul_rn(speed, speed)) : 0.0f;
        const int mm = s % 3;
        const float w0 = (mm == 0) ? 0.0f : ((mm == 1) ? -k.turn : k.turn);
        for (int t = 0; t < k.H; ++t) {
            u[2 * t] = a0;
            u[2 * t + 1] = w0;
        }
    }
    float f = lbfgs_value_grad(k, gw, wraw, ws, x0, y0, v0, th0, oth, P, u, g);
    float sy_last = 0.0f, yy_last = 1.0f;
    int kk = 0, head = 0;
    for (int it = 0; it < k.n_iter; ++it) {
        for (int j = 0; j < n; ++j) q[j] = g[j];
        for (int i = 0; i < kk; ++i) {                      // newest pair first
            const int idx = (head - 1 - i + 2 * kLbfgsM) % kLbfgsM;
            float dot = 0.0f;
            for (int j = 0; j < n; ++j) dot = __fadd_rn(dot, __fmul_rn(Sh[idx][j], q[j]));
            al[i] = __fmul_rn(rho[idx], dot);
            for (int j = 0; j < n; ++j) q[j] = __fsub_rn(q[j], __fmul_rn(al[i], Yh[idx][j]));
        }
        {
            const float gamma = (kk > 0) ? __fdiv_rn(sy_last, yy_last) : k.lr;
            for (int j = 0; j < n; ++j) q[j] = __fmul_rn(gamma, q[j]);
        }
        for (int i = kk - 1; i >= 0; --i) {                 // oldest pair first
            const int idx = (head - 1 - i + 2 * kLbfgsM) % kLbfgsM;
            float dot = 0.0f;
            for (int j = 0; j < n; ++j) dot = __fadd_rn(dot, __fmul_rn(Yh[idx][j], q[j]));
            const float bb = __fmul_rn(rho[idx], dot);
            for (int j = 0; j < n; ++j) q[j] = __fadd_rn(q[j], __fmul_rn(Sh[idx][j], __fsub_rn(al[i], bb)));
        }
        float gd = 0.0f;
        for (int j = 0; j < n; ++j) {
            d[j] = -q[j];
            gd = __fadd_rn(gd, __fmul_rn(g[j], d[j]));
        }
        if (!(gd < 0.0f)) {                                 // not a descent direction: restart
            kk = 0;
            gd = 0.0f;
            for (int j = 0; j < n; ++j) {
                d[j] = __fmul_rn(-k.lr, g[j]);
                gd = __fadd_rn(gd, __fmul_rn(g[j], d[j]));
            }
        }
        if (!(gd < 0.0f)) break;
        float t = 1.0f, ft = f;
        bool ok = false;
        for (int ls = 0; ls < kLbfgsLS; ++ls) {
            for (int j = 0; j < n; ++j) ut[j] = __fadd_rn(u[j], __fmul_rn(t, d[j]));
            ft = lbfgs_value_grad(k, gw, wraw, ws, x0, y0, v0, th0, oth, P, ut, nullptr);
            if (ft <= __fadd_rn(f, __fmul_rn(__fmul_rn(1e-4f, t), gd))) {
                ok = true;
                break;
            }
            t = __fmul_rn(t, 0.5f);
        }
        if (!ok) break;
        lbfgs_value_grad(k, gw, wraw, ws, x0, y0, v0, th0, oth, P, ut, gt);
        {
            // the candidate pair goes to scratch (d and q are free here): once the ring is full, slot `head` holds the
            // oldest pair the two-loop recursion still reads, and a rejected candidate must not overwrite it
            float sy = 0.0f, yy = 0.0f;
            for (int j = 0; j < n; ++j) {
                const float sj = __fsub_rn(ut[j], u[j]), yj = __fsub_rn(gt[j], g[j]);
                d[j] = sj;
                q[j] = yj;
                sy = __fadd_rn(sy, __fmul_rn(sj, yj));
                yy = __fadd_rn(yy, __fmul_rn(yj, yj));
            }
            if (yy > 0.0f && sy > __fmul_rn(1e-10f, yy)) {
                for (int j = 0; j < n; ++j) {
                    Sh[head][j] = d[j];
                    Yh[head][j] = q[j];
                }
                rho[head] = __fdiv_rn(1.0f, sy);
                head = (head + 1) % kLbfgsM;
                if (kk < kLbfgsM) ++kk;
                sy_last = sy;
                yy_last = yy;
            }
        }
        for (int j = 0; j < n; ++j) {
            u[j] = ut[j];
            g[j] = gt[j];
        }
        f = ft;
    }
    return lbfgs_value_grad(k, gw, wraw, ws, x0, y0, v0, th0, oth, P, u, nullptr);
}

// ---------------------------------------------------------------------------------------------
// k_episode_lbfgs -- MPC_ORD's receding-horizon loop with the L-BFGS planner (ocd_episode_batch, optimizer 1).
// k_episode's block shape (S warps x 32 worlds, one thread per (world, start)) and per-step bookkeeping: the
// replanning teleport, traj_states, the true-weight reward of the past state, the argmin over starts, traj_controls /
// traj_best and the simulator step of every car.  Each step's solve is k_solve_lbfgs's: the same start code
// (lbfgs_start), the other cars predicted by the solve's model fed with the scenario's known controls (OtherControls:
// a fixed-plan car's plan replayed from index 0, zero controls for the others; constant velocity with other_mode 0),
// planned from the robot's own speed.  So step t equals ocd_solve_batch (optimizer 1) on traj_states[t] bit for bit.
// Like k_solve_lbfgs it runs precise math whatever the math mode: the lanes of a warp take different numbers of
// line-search trials.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kMaxThreads)
k_episode_lbfgs(const __grid_constant__ KParams k, const __grid_constant__ ocd_scenario sc, const EpisodeArgs a) {
    extern __shared__ __align__(16) float smem_raw[];
    constexpr int P = kP;
    const Smem m = carve(smem_raw, k, P, true, false, false);
    const int p = threadIdx.x % P, s = threadIdx.x / P;
    const long long b_raw = (long long)blockIdx.x * P + p;
    const bool live = b_raw < a.B;
    const long long b = live ? b_raw : a.B - 1;
    const long long B = a.B;
    const int C = k.NO + 1;
    const OtherControls model{nullptr, 0, &sc};

    if (threadIdx.x < k.K) m.wtrue[threadIdx.x] = a.true_weights[threadIdx.x];
    int unlucky = 0;
    if (s == 0) {
        const long long wc = weight_column(a.weight_idx, a.Bw, b);
        for (int i = 0; i < k.K; ++i) m.wraw[i * P + p] = a.plan_weights[(size_t)i * a.Bw + wc];
        for (int c = 0; c < 4; ++c) m.world[c * P + p] = a.robot_init[(size_t)c * B + b];
        for (int j = 0; j < k.NO; ++j)
            for (int c = 0; c < 4; ++c)
                m.world[((j + 1) * 4 + c) * P + p] =
                    a.other_init ? a.other_init[(size_t)(j * 4 + c) * B + b] : sc.init_state[j][c];
        if (a.unlucky_idx) unlucky = a.unlucky_idx[b];
    }
    __syncthreads();
    const GradW gw = make_gradw<0>(k, m.wraw + p, P);
    float ret = 0.0f;

    for (int i = 0; i < a.T; ++i) {
        const int ti = a.t0 + i;
        if (s == 0) {
            // ReplanningCarWorld.step: teleport before anything else (replanning_world.py:31-34)
            if (sc.critical_t > 0 && ti + 1 == sc.critical_t && unlucky >= 1 && unlucky < C)
                for (int c = 0; c < 4; ++c) m.world[(unlucky * 4 + c) * P + p] = sc.teleport_state[c];
            if (a.traj_states && live)
                for (int c = 0; c < C * 4; ++c)
                    a.traj_states[((size_t)i * C * 4 + c) * B + b] = m.world[c * P + p];
            // true-weight reward of the past state (mpc_ord.py:96-99)
            {
                const float x = m.world[p], y = m.world[P + p], v = m.world[2 * P + p], th = m.world[3 * P + p];
                float sn, cs;
                Mth<true>::sincos_(th, sn, cs);
                ret = __fadd_rn(ret, reward_value<0, true, false>(k, m.wtrue, 1, x, y, v, sn, m.world + 4 * P + p,
                                                                  4 * P, P));
            }
            // what the planner assumes about the other cars: k_solve_lbfgs's slab, fed with the scenario's controls
            float buf[2 * OCD_MAX_H];
            for (int j = 0; j < k.NO; ++j) {
                const float *w = m.world + (size_t)(j + 1) * 4 * P + p;
                long long ocs;
                const float *oc = model.car(k, j, b, buf, ocs);
                predict_other<true>(k, w[0], w[P], w[2 * P], w[3 * P], oc, ocs, m.oth + p, j, P);
            }
        }
        __syncthreads();

        const float x0 = m.world[p], y0 = m.world[P + p], v0 = m.world[2 * P + p], th0 = m.world[3 * P + p];
        float u[kLbfgsN];
        m.loss[s * P + p] = lbfgs_start(k, gw, m.wraw + p, P, x0, y0, v0, th0, m.oth + p, P, s, v0, u);
        m.u0[(s * 2 + 0) * P + p] = u[0];
        m.u0[(s * 2 + 1) * P + p] = u[1];
        __syncthreads();

        if (s == 0) {
            int bi = 0;
            float bl = m.loss[p];
            for (int q = 1; q < k.S; ++q) {
                const float l = m.loss[q * P + p];
                if (l < bl) { bl = l; bi = q; }
            }
            const float ua = m.u0[(bi * 2 + 0) * P + p], uw = m.u0[(bi * 2 + 1) * P + p];
            if (live) {
                if (a.traj_controls) {
                    a.traj_controls[((size_t)i * 2 + 0) * B + b] = ua;
                    a.traj_controls[((size_t)i * 2 + 1) * B + b] = uw;
                }
                if (a.traj_best) a.traj_best[(size_t)i * B + b] = bi;
            }
            // CarWorld.step second phase: every car integrates (world.py:106-107, car.py:87)
            {
                float x = x0, y = y0, v = v0, th = th0;
                dynamics_step<true>(x, y, v, th, ua, uw, k.dt, k.dt2, k.mu);
                m.world[p] = x; m.world[P + p] = y; m.world[2 * P + p] = v; m.world[3 * P + p] = th;
            }
            for (int j = 0; j < k.NO; ++j) {
                float *w = m.world + (size_t)(j + 1) * 4 * P + p;
                float x = w[0], y = w[P], v = w[2 * P], th = w[3 * P];
                const bool in_plan = sc.kind[j] == 1 && ti < sc.plan_len[j];   // fixed_plan_car.py:25-31
                const float oa = in_plan ? sc.plan[j][ti][0] : sc.control[j][0];
                const float oo = in_plan ? sc.plan[j][ti][1] : sc.control[j][1];
                dynamics_step<true>(x, y, v, th, oa, oo, k.dt, k.dt2, sc.friction[j]);
                w[0] = x; w[P] = y; w[2 * P] = v; w[3 * P] = th;
            }
        }
        __syncthreads();
    }
    if (s == 0 && live) {
        a.returns[b] = ret;
        if (a.final_world)
            for (int c = 0; c < C * 4; ++c) a.final_world[(size_t)c * B + b] = m.world[c * P + p];
    }
}

// ---------------------------------------------------------------------------------------------
// k_episode_jac_implicit -- the Jacobians of the applied controls of an L-BFGS episode (ocd_episode_implicit_vjp_batch).
//
// Step t applies u_t = first control of u*(w, s_t), the stationary point L-BFGS found from the winning start at
// world_t = traj_states[t].  As in k_solve_implicit_vjp, with A the controls inside the inclusive clip box and
// H = dG/du (G = dR/du), the implicit function theorem gives du*_A/dtheta = -H_AA^{-1} dG_A/dtheta, theta = (w, s0):
// the row of J_t for seed c (plan[0][c]) is -grad_theta (G . z) with H_AA z = e_c.  k_episode_adjoint then chains the
// rows along the episode exactly as for the SGD planner.  One thread per (world, step), the step on blockIdx.y; it
//   1. re-runs start traj_best[t] with lbfgs_start and k_episode_lbfgs's other-car model and stores the plan (its first
//      control is traj_controls[t] bit for bit),
//   2. builds H_AA from |A| sweeps of vjp_hvp along the unit vectors of A,
//   3. drops the decoupled controls: a control whose row and column of H_AA are exactly zero (the last steering input
//      once the speed feature's `min` has saturated, so that G_j vanishes in a neighbourhood).  Then dG_j/dtheta = 0
//      too and z_j enters nothing, so setting z_j = 0 is exact;
//   4. equilibrates the rest (rows and columns scaled by 1 / sqrt of their largest entry) and eliminates it in double
//      with diagonal pivoting for both seeds.  Controls whose remaining curvature is below the float rounding of
//      H_AA (the rank it resolves) are held at their value: z_j = 0;
//   5. runs one vjp_hvp<true> sweep per seed with scale -1: the weight and robot rows.  The other-car gradient (obar)
//      is dropped: the scripted cars depend on neither w nor the robot.
// Why held controls: at the designer weights of finite_horizon the robot reaches the target speed straight ahead, and
// the last steering input then acts on the reward only through cos(theta_H) and e = v sin(theta_H) - target speed,
// both near zero.  Its curvature (with the accelerations eliminated) is some 1e-13 of the largest entry in f64 and
// below the resolution of the float state itself (an ulp of v near 1 is 1.2e-7), so the float H_AA cannot determine it,
// the float gradient the planner follows does not see it either, and the planner leaves that control where its start
// put it.  Holding it is the derivative of the plan along the directions the planner resolves; the exact optimum's
// derivative along the unresolved one would scale like 1 / (its curvature).
// A clipped seed has a zero row.  A held seed (decoupled or unresolved) is not moved by L-BFGS, so it keeps its start
// value: a0 = friction v0^2 for the acceleration of the extra-init starts, whose row is 2 friction v0 on the robot's
// speed, a constant otherwise.  A matrix the elimination cannot factor (a small pivot beside a large off-diagonal:
// indefinite) makes both rows NaN, which k_episode_adjoint carries into that world's outputs alone.  status [T][B]:
// the number of held controls, or -1 where the step is singular; held [T][B]: their bit mask (bit 2t + c).
// ---------------------------------------------------------------------------------------------
struct EpisodeImplicitArgs {
    const float *plan_weights;     // [K][Bw]
    long long    Bw;
    const int32_t *weight_idx;     // [B] or null
    int          t0;               // first step of this launch
    const float *traj_states;      // [T][C][4][B]
    const int32_t *traj_best;      // [T][B]
    float       *jac;              // [T][2][K + 4][B] workspace
    float       *plans;            // [T][H][2][B] workspace
    float       *status;           // [T][B] workspace
    unsigned    *held;             // [T][B] workspace
    long long    B;
};

__global__ void __launch_bounds__(kVjpThreads)
k_episode_jac_implicit(const __grid_constant__ KParams k, const __grid_constant__ ocd_scenario sc,
                       const EpisodeImplicitArgs a) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    const long long B = a.B;
    const int t = a.t0 + (int)blockIdx.y, H = k.H, n = 2 * k.H, KJ = k.K + 4;
    const float *world = a.traj_states + (size_t)t * (k.NO + 1) * 4 * B;
    int s = a.traj_best[(size_t)t * B + b];
    s = s < 0 ? 0 : (s >= k.S ? k.S - 1 : s);
    float oth[OCD_LBFGS_MAX_H * OCD_MAX_OTHER * 2];
    vjp_predict_others(k, world, B, b, OtherControls{nullptr, 0, &sc}, oth);
    const float s0[4] = {world[b], world[B + b], world[2 * B + b], world[3 * B + b]};
    const float *w = a.plan_weights + weight_column(a.weight_idx, a.Bw, b);
    const int ws = (int)a.Bw;
    float u[kLbfgsN];
    lbfgs_start(k, make_gradw<0>(k, w, ws), w, ws, s0[0], s0[1], s0[2], s0[3], oth, 1, s, s0[2], u);
    for (int i = 0; i < n; ++i) a.plans[((size_t)t * n + i) * B + b] = u[i];

    // H_AA column by column (row-major, n_A x n_A), in double from the float HVPs; a control's row and column are
    // tracked for exact zeros on the way (decoupled controls)
    float d[kLbfgsN], hv[kLbfgsN];
    int act[kLbfgsN];
    int na = 0;
    for (int q = 0; q < H; ++q) {
        if ((u[2 * q] >= -8.0f) && (u[2 * q] <= 4.0f)) act[na++] = 2 * q;
        if (fabsf(u[2 * q + 1]) <= 4.0f) act[na++] = 2 * q + 1;
    }
    double R[kImplicitN * kImplicitN];
    bool zero[kLbfgsN];
    for (int i = 0; i < na; ++i) zero[i] = true;
    for (int i = 0; i < n; ++i) d[i] = 0.0f;
    for (int j = 0; j < na; ++j) {
        d[act[j]] = 1.0f;
        vjp_hvp<false>(k, w, ws, s0, oth, u, d, hv, 0.0f, nullptr, nullptr, nullptr);
        d[act[j]] = 0.0f;
        for (int i = 0; i < na; ++i) {
            const float h = hv[act[i]];
            R[i * na + j] = (double)h;
            if (h != 0.0f) zero[i] = zero[j] = false;        // row i and column j are not zero
        }
    }
    // symmetrised, then compacted in place onto keep[], the positions in A that are not decoupled (the target index
    // i nr + j never passes the source index keep[i] na + keep[j], and both grow in the same order), then equilibrated:
    // row and column i scaled by e_i = 1 / sqrt(max_j |R_ij|)
    for (int i = 0; i < na; ++i)
        for (int j = 0; j < i; ++j) R[i * na + j] = R[j * na + i] = 0.5 * (R[i * na + j] + R[j * na + i]);
    int keep[kLbfgsN], nr = 0;
    for (int i = 0; i < na; ++i)
        if (!zero[i]) keep[nr++] = i;
    for (int i = 0; i < nr; ++i)
        for (int j = 0; j < nr; ++j) R[i * nr + j] = R[keep[i] * na + keep[j]];
    double e[kImplicitN], z[kImplicitN * 2], scale = 0.0;
    int perm[kImplicitN];
    for (int i = 0; i < nr; ++i) {
        double r = 0.0;
        for (int j = 0; j < nr; ++j) r = fmax(r, fabs(R[i * nr + j]));
        e[i] = 1.0 / sqrt(r);                                 // r > 0: the row is not zero
        perm[i] = i;
        z[2 * i] = act[keep[i]] == 0 ? e[i] : 0.0;            // seed plan[0][0]
        z[2 * i + 1] = act[keep[i]] == 1 ? e[i] : 0.0;        // seed plan[0][1]
    }
    for (int i = 0; i < nr; ++i)
        for (int j = 0; j < nr; ++j) {
            R[i * nr + j] *= e[i] * e[j];
            scale = fmax(scale, fabs(R[i * nr + j]));
        }
    // Symmetric elimination with diagonal pivoting (the largest remaining |pivot| first).  The entries carry float
    // rounding, so a remaining diagonal below n_A float ulps of the largest entry cannot be told from zero.  When every
    // remaining diagonal is that small and so is every remaining off-diagonal -- as in a semidefinite matrix, where
    // |R_ij| <= sqrt(|R_ii R_jj|) -- the controls left carry no curvature the float arithmetic resolves: they are held at
    // their value like the decoupled ones (z = 0, bit set in `held`).  A small diagonal beside a large off-diagonal is an
    // indefinite matrix the elimination cannot factor: the step is singular.
    const double tiny = (double)na * (double)FLT_EPSILON * scale;
    bool ok = true;
    int rank = nr;
    for (int c = 0; c < nr; ++c) {
        int pv = c;
        for (int i = c + 1; i < nr; ++i)
            if (fabs(R[i * nr + i]) > fabs(R[pv * nr + pv])) pv = i;
        if (!(fabs(R[pv * nr + pv]) > tiny)) {
            for (int i = c; i < nr; ++i)
                for (int j = c; j < nr; ++j) ok = ok && fabs(R[i * nr + j]) <= tiny;
            rank = c;
            break;
        }
        if (pv != c) {                                        // symmetric swap of c and pv
            for (int j = 0; j < nr; ++j) {
                const double t0 = R[c * nr + j]; R[c * nr + j] = R[pv * nr + j]; R[pv * nr + j] = t0;
            }
            for (int i = 0; i < nr; ++i) {
                const double t0 = R[i * nr + c]; R[i * nr + c] = R[i * nr + pv]; R[i * nr + pv] = t0;
            }
            for (int q = 0; q < 2; ++q) {
                const double t0 = z[2 * c + q]; z[2 * c + q] = z[2 * pv + q]; z[2 * pv + q] = t0;
            }
            const int t1 = perm[c]; perm[c] = perm[pv]; perm[pv] = t1;
        }
        for (int i = c + 1; i < nr; ++i) {
            const double f = R[i * nr + c] / R[c * nr + c];
            for (int j = c + 1; j < nr; ++j) R[i * nr + j] -= f * R[c * nr + j];
            for (int q = 0; q < 2; ++q) z[2 * i + q] -= f * z[2 * c + q];
        }
    }
    double zz[kImplicitN * 2];                                // z in the order of keep[]
    for (int i = 0; i < nr; ++i) zz[2 * i] = zz[2 * i + 1] = 0.0;
    for (int q = 0; q < 2; ++q)
        for (int r = rank - 1; r >= 0; --r) {
            double acc = z[2 * r + q];
            for (int j = r + 1; j < rank; ++j) acc -= R[r * nr + j] * z[2 * j + q];
            z[2 * r + q] = acc / R[r * nr + r];
            zz[2 * perm[r] + q] = z[2 * r + q] * e[perm[r]];
        }
    // held: the decoupled controls and those left after the last resolved pivot (flat index 2t + c)
    unsigned held = 0u;
    for (int i = 0; i < na; ++i)
        if (zero[i]) held |= 1u << act[i];
    for (int r = rank; r < nr; ++r) held |= 1u << act[keep[perm[r]]];
    a.status[(size_t)t * B + b] = ok ? (float)(na - rank) : -1.0f;
    a.held[(size_t)t * B + b] = held;
    float *J = a.jac + (size_t)t * 2 * KJ * B + b;
    if (!ok) {
        const float nan = __int_as_float(0x7fffffff);
        for (int i = 0; i < 2 * KJ; ++i) J[(size_t)i * B] = nan;
        return;
    }
    float obar[OCD_LBFGS_MAX_H * OCD_MAX_OTHER * 2];
    for (int c = 0; c < 2; ++c) {
        float wbar[kVjpK], s0bar[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int q = 0; q < kVjpK; ++q) wbar[q] = 0.0f;
        // seed c is inside the clip box and coupled: the implicit-function row; clipped or decoupled: zero, but for
        // the start value friction v0^2 of a decoupled extra-init acceleration
        const bool in_a = (c == 0) ? ((u[0] >= -8.0f) && (u[0] <= 4.0f)) : (fabsf(u[1]) <= 4.0f);
        if (in_a && !(held & (1u << c))) {
            for (int i = 0; i < n; ++i) d[i] = 0.0f;
            for (int i = 0; i < nr; ++i) d[act[keep[i]]] = (float)zz[2 * i + c];
            vjp_hvp<true>(k, w, ws, s0, oth, u, d, hv, -1.0f, wbar, s0bar, obar);
        } else if (in_a && c == 0 && s >= 3) {
            s0bar[2] = 2.0f * k.mu * s0[2];
        }
#pragma unroll
        for (int q = 0; q < kVjpK; ++q)
            if (q < k.K) J[(size_t)(c * KJ + q) * B] = wbar[q];
        for (int q = 0; q < 4; ++q) J[(size_t)(c * KJ + k.K + q) * B] = s0bar[q];
    }
}

}  // namespace ocd
