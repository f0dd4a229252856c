// ocd_api.cu -- C ABI of the B200-native batched MPC engine (libocd_b200.so): argument
// validation, the (H, other cars, math mode) dispatch onto the kernels of ocd_kernels.cuh, the
// operator kernels (reward + gradient, features, dynamics) and the host-buffer layer.
// Build: make -C l4dc-mpc-ocd_b200/csrc   (nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo)
#include <cuda_runtime.h>
#include <sched.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "ocd_kernels.cuh"
#include "ocd_hessian.cuh"
#include "ocd_vjp.cuh"

namespace ocd {

// specialisations built by ocd_inst.cu
#define OCD_EXTERN(HT, NO, LT)                                                                               \
    extern template int launch_solve_t<HT, NO, LT, false>(const KParams &, const SolveArgs &, cudaStream_t); \
    extern template int launch_solve_t<HT, NO, LT, true>(const KParams &, const SolveArgs &, cudaStream_t);  \
    extern template int launch_episode_t<HT, NO, LT, false>(const KParams &, const ocd_scenario &,           \
                                                            const EpisodeArgs &, cudaStream_t);              \
    extern template int launch_episode_t<HT, NO, LT, true>(const KParams &, const ocd_scenario &,            \
                                                           const EpisodeArgs &, cudaStream_t);               \
    extern template int launch_solve_vjp_t<HT, NO, LT, false>(const KParams &, const VjpArgs &, cudaStream_t); \
    extern template int launch_solve_vjp_t<HT, NO, LT, true>(const KParams &, const VjpArgs &, cudaStream_t);    \
    extern template int launch_episode_jac_t<HT, NO, LT, false>(const KParams &, const ocd_scenario &,         \
                                                                const EpisodeVjpArgs &, int, cudaStream_t);  \
    extern template int launch_episode_jac_t<HT, NO, LT, true>(const KParams &, const ocd_scenario &,          \
                                                               const EpisodeVjpArgs &, int, cudaStream_t);
OCD_EXTERN(5, 1, 3)   // finite_horizon, local_opt, the bench shape
OCD_EXTERN(5, 2, 2)   // replanning
OCD_EXTERN(6, 1, 3)   // finite_horizon validation (H=6, n_iter=200)
OCD_EXTERN(5, 0, 3)   // H=5 on three lanes with any number of other cars (sweep)
OCD_EXTERN(0, 1, 3)   // any horizon, one other car, three lanes: segmented adjoint (sweep H=15, 50)
OCD_EXTERN(0, 0, 3)   // any horizon / cars on three lanes: segmented adjoint
OCD_EXTERN(0, 0, 0)   // any other shape: runtime H, cars, lanes (segmented adjoint)
#undef OCD_EXTERN
// FAST k_solve alone, compile-time car count: the 3..6-car points of the synthetic sweep
#define OCD_EXTERN_SOLVE(HT, NO, LT)                                                                       \
    extern template int launch_solve_t<HT, NO, LT, false>(const KParams &, const SolveArgs &, cudaStream_t); \
    extern template int launch_solve_vjp_t<HT, NO, LT, false>(const KParams &, const VjpArgs &, cudaStream_t);
OCD_EXTERN_SOLVE(5, 2, 3)
OCD_EXTERN_SOLVE(5, 3, 3)
OCD_EXTERN_SOLVE(5, 4, 3)
OCD_EXTERN_SOLVE(5, 5, 3)
OCD_EXTERN_SOLVE(0, 2, 3)
OCD_EXTERN_SOLVE(0, 3, 3)
OCD_EXTERN_SOLVE(0, 4, 3)
OCD_EXTERN_SOLVE(0, 5, 3)
// the sweep's other two horizons at a compile-time H: 15 (medium: the Q kernels) and 50 (long: constant segment count)
OCD_EXTERN_SOLVE(15, 1, 3)
OCD_EXTERN_SOLVE(15, 2, 3)
OCD_EXTERN_SOLVE(15, 3, 3)
OCD_EXTERN_SOLVE(15, 4, 3)
OCD_EXTERN_SOLVE(15, 5, 3)
OCD_EXTERN_SOLVE(50, 1, 3)
OCD_EXTERN_SOLVE(50, 2, 3)
OCD_EXTERN_SOLVE(50, 3, 3)
OCD_EXTERN_SOLVE(50, 4, 3)
OCD_EXTERN_SOLVE(50, 5, 3)
#undef OCD_EXTERN_SOLVE

// ---------------------------------------------------------------------------------------------
// operator kernels: reward + gradient, features, dynamics
// ---------------------------------------------------------------------------------------------
template <bool PRECISE>
__global__ void __launch_bounds__(128)
k_reward_grad(const __grid_constant__ KParams k, const float *world, const float *controls,
              const float *other_controls, long long Bo, const float *weights, long long Bw,
              const int32_t *weight_idx, float *reward, float *grad, long long B, int onehot_stride) {
    // one thread per problem; its slab column lives in local memory (runtime H, runtime NO)
    // onehot_stride > 0 (ocd_feature_jacobian_batch): blockIdx.y = i selects feature i -- the weights are row i of the
    // one-hot table and the outputs row i of phi_sum [K][B] / jac [K][H][2][B]: all K rows in ONE launch
    if (onehot_stride > 0) {
        weights += (size_t)blockIdx.y * onehot_stride;
        reward += (size_t)blockIdx.y * B;
        grad += (size_t)blockIdx.y * k.H * 2 * B;
    }
    const long long b_raw = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = b_raw < B;
    const long long b = live ? b_raw : B - 1;     // whole warps stay converged: feature_grad votes
    float oth[OCD_MAX_H * OCD_MAX_OTHER * 2];
    // weights are read straight from global memory (element stride Bw).  A thread-local copy
    // here was miscompiled by nvcc 12.9: the copy's stack slot was reused for reward_value's
    // phi[] while make_gradw still reloaded it afterwards.
    const float *w = weights + weight_column(weight_idx, Bw, b);
    const int ws = (int)Bw;
    for (int j = 0; j < k.NO; ++j) {
        const float *st = world + (size_t)(j + 1) * 4 * B + b;
        const float *oc = nullptr;
        long long ocs = 0;
        if (k.other_mode == 1) {
            ocs = Bo;
            oc = other_controls + (size_t)j * k.H * 2 * Bo + (Bo == 1 ? 0 : b);
        }
        predict_other<PRECISE>(k, st[0], st[B], st[2 * B], st[3 * B], oc, ocs, oth, j, 1);
    }
    const float x0 = world[b], y0 = world[B + b], v0 = world[2 * B + b], th0 = world[3 * B + b];
    Traj<0> u;
    for (int t = 0; t < k.H; ++t) {
        u.ua[t] = controls[(size_t)(t * 2 + 0) * B + b];
        u.uw[t] = controls[(size_t)(t * 2 + 1) * B + b];
    }
    const float R = rollout_reward<0, 0, PRECISE>(k, w, ws, x0, y0, v0, th0, oth, 1, u);
    if (live) reward[b] = R;
    if (grad) {
        const GradW gw = make_gradw<0>(k, w, ws);
        float ga[OCD_MAX_H], go[OCD_MAX_H];
        float sn0, cs0;
        Mth<PRECISE>::sincos_(th0, sn0, cs0);
        sgd_iteration<0, 0, 0, PRECISE, false>(k, gw, x0, y0, v0, th0, sn0, cs0, oth, 1, u, ga, go);
        for (int t = 0; t < k.H && live; ++t) {
            grad[(size_t)(t * 2 + 0) * B + b] = ga[t];
            grad[(size_t)(t * 2 + 1) * B + b] = go[t];
        }
    }
}

// One-hot weight vectors: row i of an 8x8 identity selects feature i.  ocd_feature_jacobian_batch runs
// k_reward_grad once per feature with these as the (shared) weights.
__device__ float g_onehot[(OCD_MAX_LANES + 4) * (OCD_MAX_LANES + 4)] = {
    1, 0, 0, 0, 0, 0, 0, 0,  0, 1, 0, 0, 0, 0, 0, 0,  0, 0, 1, 0, 0, 0, 0, 0,  0, 0, 0, 1, 0, 0, 0, 0,
    0, 0, 0, 0, 1, 0, 0, 0,  0, 0, 0, 0, 0, 1, 0, 0,  0, 0, 0, 0, 0, 0, 1, 0,  0, 0, 0, 0, 0, 0, 0, 1};

template <bool PRECISE>
__global__ void __launch_bounds__(128)
k_features(const __grid_constant__ KParams k, const float *world, float *phi, long long B) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float sn, cs;
    Mth<PRECISE>::sincos_(world[3 * B + b], sn, cs);
    float f[OCD_MAX_LANES + 4];
    feature_values<0, PRECISE, false>(k, world[b], world[B + b], world[2 * B + b], sn, world + 4 * B + b,
                            (int)(4 * B), (int)B, f);
#pragma unroll
    for (int i = 0; i < OCD_MAX_LANES + 4; ++i)
        if (i < k.K) phi[(size_t)i * B + b] = f[i];
}

template <bool PRECISE>
__global__ void __launch_bounds__(256)
k_dynamics(const float *state, const float *control, float dt, float dt2, float friction,
           const float *friction_b, float *next, long long B) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float x = state[b], y = state[B + b], v = state[2 * B + b], th = state[3 * B + b];
    dynamics_step<PRECISE>(x, y, v, th, control[b], control[B + b], dt, dt2, friction_b ? friction_b[b] : friction);
    next[b] = x; next[B + b] = y; next[2 * B + b] = v; next[3 * B + b] = th;
}

// ---------------------------------------------------------------------------------------------
// k_solve_lbfgs -- the opt-in L-BFGS optimiser (params.optimizer == 1; include/ocd_b200.h).
// Same block shape, slab and argmin as k_solve; per (problem, start) the thread runs L-BFGS on
// f(u) = -R(u): two-loop recursion over 4 correction pairs held in local memory, Armijo backtracking,
// gradient from the same closed-form adjoint.  Lanes of a warp take different numbers of line-search
// trials, so the warp-voting FAST feature code cannot be used here: the kernel always runs the precise
// math path.  The CPU restatement used by the parity tests mirrors this loop statement for statement.
// ---------------------------------------------------------------------------------------------
static constexpr int kLbfgsM = 4, kLbfgsLS = 6, kLbfgsN = 2 * OCD_LBFGS_MAX_H;

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

__global__ void __launch_bounds__(kMaxThreads) k_solve_lbfgs(const __grid_constant__ KParams k, const SolveArgs a) {
    extern __shared__ __align__(16) float smem_raw[];
    constexpr int P = kP;
    const Smem m = carve(smem_raw, k, P, false, false, false);
    const int p = threadIdx.x % P, s = threadIdx.x / P;
    const long long b_raw = (long long)blockIdx.x * P + p;
    const bool live = b_raw < a.B;
    const long long b = live ? b_raw : a.B - 1;
    const long long B = a.B;
    if (s == 0) {
        const long long wc = weight_column(a.weight_idx, a.Bw, b);
        for (int i = 0; i < k.K; ++i) m.wraw[i * P + p] = a.weights[(size_t)i * a.Bw + wc];
        for (int j = 0; j < k.NO; ++j) {
            const float *st = a.world + (size_t)(j + 1) * 4 * B + b;
            const float *oc = nullptr;
            long long ocs = 0;
            if (k.other_mode == 1) {
                ocs = a.Bo;
                oc = a.other_controls + (size_t)j * k.H * 2 * a.Bo + (a.Bo == 1 ? 0 : b);
            }
            predict_other<true>(k, st[0], st[B], st[2 * B], st[3 * B], oc, ocs, m.oth + p, j, P);
        }
    }
    __syncthreads();
    const float x0 = a.world[b], y0 = a.world[B + b], v0 = a.world[2 * B + b], th0 = a.world[3 * B + b];
    const GradW gw = make_gradw<0>(k, m.wraw + p, P);
    const float *wraw = m.wraw + p, *oth = m.oth + p;
    const int n = 2 * k.H;
    float u[kLbfgsN], g[kLbfgsN], gt[kLbfgsN], d[kLbfgsN], ut[kLbfgsN], q[kLbfgsN];
    float Sh[kLbfgsM][kLbfgsN], Yh[kLbfgsM][kLbfgsN], rho[kLbfgsM], al[kLbfgsM];
    {
        const float speed = a.cur_speed ? a.cur_speed[b] : v0;
        const float a0 = (s >= 3) ? __fmul_rn(k.mu, __fmul_rn(speed, speed)) : 0.0f;
        const int mm = s % 3;
        const float w0 = (mm == 0) ? 0.0f : ((mm == 1) ? -k.turn : k.turn);
        for (int t = 0; t < k.H; ++t) {
            u[2 * t] = a0;
            u[2 * t + 1] = w0;
        }
    }
    float f = lbfgs_value_grad(k, gw, wraw, P, x0, y0, v0, th0, oth, P, u, g);
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
            ft = lbfgs_value_grad(k, gw, wraw, P, x0, y0, v0, th0, oth, P, ut, nullptr);
            if (ft <= __fadd_rn(f, __fmul_rn(__fmul_rn(1e-4f, t), gd))) {
                ok = true;
                break;
            }
            t = __fmul_rn(t, 0.5f);
        }
        if (!ok) break;
        lbfgs_value_grad(k, gw, wraw, P, x0, y0, v0, th0, oth, P, ut, gt);
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
    const float loss = lbfgs_value_grad(k, gw, wraw, P, x0, y0, v0, th0, oth, P, u, nullptr);
    m.loss[s * P + p] = loss;
    if (live) {
        a.losses[(size_t)s * B + b] = loss;
        if (a.all_plans)
            for (int j = 0; j < n; ++j) a.all_plans[((size_t)s * n + j) * B + b] = u[j];
    }
    __syncthreads();
    int bi = 0;
    float bl = m.loss[p];
    for (int qs = 1; qs < k.S; ++qs) {
        const float l = m.loss[qs * P + p];
        if (l < bl) { bl = l; bi = qs; }
    }
    if (live && s == bi) {
        a.best[b] = bi;
        for (int j = 0; j < n; ++j) a.plan[(size_t)j * B + b] = u[j];
    }
}

// math_utils.py helpers as operators (precise math, reference op order)
__global__ void __launch_bounds__(256)
k_smooth(int kind, const float *z, float a, float b, float c, float *out, long long B) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const float x = z[i];
    float r = 0.0f;
    if (kind == OCD_SMOOTH_F) {                    // a = shape
        if (x > 0.0f) r = expf(__fdiv_rn(-1.0f, __fmul_rn(a, x)));
    } else if (kind == OCD_SMOOTH_THRESHOLD) {     // a = threshold - width, b = width, c = shape
        const float q = __fsub_rn(x, a), u2 = __fsub_rn(b, q);
        const float F1 = q > 0.0f ? expf(__fdiv_rn(-1.0f, __fmul_rn(c, q))) : 0.0f;
        const float F2 = u2 > 0.0f ? expf(__fdiv_rn(-1.0f, __fmul_rn(c, u2))) : 0.0f;
        r = __fdiv_rn(F1, __fadd_rn(F1, F2));
    } else {                                       // a = start, b = end
        const float width = __fmul_rn(__fsub_rn(b, a), 0.5f), center = __fmul_rn(__fadd_rn(a, b), 0.5f);
        const float n = __fdiv_rn(__fsub_rn(x, center), width);
        if (__fmul_rn(n, n) < 1.0f) r = expf(__fadd_rn(__fdiv_rn(-1.0f, __fsub_rn(1.0f, __fmul_rn(n, n))), 1.0f));
    }
    out[i] = r;
}

// dependent-free FMA loop: 8 independent chains per thread, 512 FFMA per loop trip (so the loop's own counter,
// compare and branch are 0.6 % of the issue slots; with 64 per trip the probe read 92 % of nominal), 2 FLOP per FMA
static constexpr int kPeakFmaPerTrip = 512;
__global__ void __launch_bounds__(256) k_fp32_peak(int iters, float *sink) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f;
    float a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float m = 0.999f, c = 1e-3f;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < kPeakFmaPerTrip / 8; ++r) {
            a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
            a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
        }
    }
    const float r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == 123.456f) sink[0] = r;
}

// ---------------------------------------------------------------------------------------------
// host side: parameter digest, validation, dispatch
// ---------------------------------------------------------------------------------------------
static int digest(const ocd_params *p, KParams &k) {
    if (!p) return OCD_EINVAL;
    if (p->H < 1 || p->C < 2 || p->L < 1 || p->n_iter < 0) return OCD_EINVAL;
    if (p->H > OCD_MAX_H || p->C > OCD_MAX_OTHER + 1 || p->L > OCD_MAX_LANES) return OCD_EUNSUP;
    if (p->other_mode != 0 && p->other_mode != 1) return OCD_EINVAL;
    if (p->math_mode != 0 && p->math_mode != 1) return OCD_EINVAL;
    std::memset(&k, 0, sizeof(k));
    k.H = p->H;
    k.NO = p->C - 1;
    k.L = p->L;
    k.K = p->L + 4;
    k.n_iter = p->n_iter;
    k.S = p->extra_inits ? 6 : 3;
    k.other_mode = p->other_mode;
    k.extra_inits = p->extra_inits ? 1 : 0;
    if (p->optimizer != 0 && p->optimizer != 1) return OCD_EINVAL;
    if (p->reserved != 0) return OCD_EINVAL;
    if (p->optimizer == 1 && p->H > OCD_LBFGS_MAX_H) return OCD_EUNSUP;
    k.optimizer = p->optimizer;
    k.lr = (float)p->lr;
    k.dt = (float)p->dt;
    k.dt2 = (float)(p->dt * p->dt);              // dt**2 in double, cast once (simulation_utils.py:16)
    k.hdt2 = 0.5f * k.dt2;
    k.mu = (float)p->friction;
    k.ts = (float)p->target_speed;               // np.float32(target_speed), merging.py:49
    k.bound = (float)(4.0 * (double)k.ts * (double)k.ts);
    {   // float squaring is monotone, so the mask e*e <= bound (TF's Minimum gradient) is |e| <= ebound exactly
        float e = sqrtf(k.bound);
        while (e > 0.0f && e * e > k.bound) e = nextafterf(e, 0.0f);
        while (nextafterf(e, INFINITY) * nextafterf(e, INFINITY) <= k.bound) e = nextafterf(e, INFINITY);
        k.ebound = e;
    }
    k.thr_lo = (float)(0.05 * (double)p->num_lanes - 0.05);   // threshold - width, math_utils.py:92
    k.thr_w = 0.05f;
    k.fshape = (float)(5.0 / 0.05);
    k.turn = (float)(5 * 0.13);                  // naive_planner.py:109-110
    for (int i = 0; i < p->L; ++i) k.lane_x[i] = (float)p->lane_x[i];
    {   // midpoints between lanes adjacent in sorted order (the only places where the lane-min can tie)
        float sorted[OCD_MAX_LANES];
        for (int i = 0; i < p->L; ++i) sorted[i] = k.lane_x[i];
        for (int i = 1; i < p->L; ++i)
            for (int j = i; j > 0 && sorted[j] < sorted[j - 1]; --j) {
                const float t = sorted[j]; sorted[j] = sorted[j - 1]; sorted[j - 1] = t;
            }
        for (int i = 0; i + 1 < p->L; ++i) k.lane_mid[i] = (float)(((double)sorted[i] + (double)sorted[i + 1]) * 0.5);
        for (int i = 0; i < OCD_MAX_LANES; ++i) k.lane_sorted[i] = i < p->L ? sorted[i] : 0.0f;
    }
    k.fs_lo = k.fshape * k.thr_lo;
    k.fs_w = k.fshape * k.thr_w;
    {
        const double ln2 = 0.69314718055994530942;
        k.fl_shape = (float)(ln2 * (double)k.fshape);
        k.fl_lo = (float)(ln2 * (double)k.fshape * (double)k.thr_lo);
        k.fl_w = (float)(ln2 * (double)k.fshape * (double)k.thr_w);
        k.fl_c = (float)(ln2 * ln2 * (double)k.fshape);
        k.mid_c = p->L == 3 ? 0.5f * (k.lane_mid[0] + k.lane_mid[1]) : 0.0f;
        k.mid_h = p->L == 3 ? 0.5f * (k.lane_mid[1] - k.lane_mid[0]) : 0.0f;
    }
    return OCD_OK;
}

static int check_weights(const float *weights, long long Bw, const int32_t *idx, long long B) {
    if (!weights || Bw < 1) return OCD_EINVAL;
    if (Bw > (1LL << 27)) return OCD_EUNSUP;   // (K-1)*Bw is indexed in 32 bits
    if (!idx && Bw != 1 && Bw != B) return OCD_EINVAL;
    return OCD_OK;
}

// host-resident weight_idx (the *_host entry points): every entry must select a column of the table
static int check_host_idx(const int32_t *idx, long long Bw, long long B) {
    if (!idx) return OCD_OK;
    for (long long b = 0; b < B; ++b)
        if (idx[b] < 0 || idx[b] >= Bw) return OCD_EINVAL;
    return OCD_OK;
}

static int pick_P(long long) { return kP; }

// (H, other cars, lanes) specialisations: the shipped scenarios; everything else takes the
// runtime-shape kernels.
#define OCD_DISPATCH(FN, PRECISE, ...)                                                      \
    do {                                                                                    \
        if (k.H == 5 && k.NO == 1 && k.L == 3) return FN<5, 1, 3, PRECISE>(__VA_ARGS__);    \
        if (k.H == 5 && k.NO == 2 && k.L == 2) return FN<5, 2, 2, PRECISE>(__VA_ARGS__);    \
        if (k.H == 6 && k.NO == 1 && k.L == 3) return FN<6, 1, 3, PRECISE>(__VA_ARGS__);    \
        if (k.H == 5 && k.L == 3) return FN<5, 0, 3, PRECISE>(__VA_ARGS__);                 \
        if (k.NO == 1 && k.L == 3) return FN<0, 1, 3, PRECISE>(__VA_ARGS__);                \
        if (k.L == 3) return FN<0, 0, 3, PRECISE>(__VA_ARGS__);                             \
        return FN<0, 0, 0, PRECISE>(__VA_ARGS__);                                           \
    } while (0)

// FAST k_solve on three lanes with 1..5 other cars: compile-time car count, and a compile-time horizon for the
// three horizons of the synthetic sweep (5: register-resident, 15: Q kernels, 50: constant segment count).
#define OCD_SOLVE_SWITCH(FN, NO_, ...)                                          \
    do {                                                                        \
        if (k.H == 15) return FN<15, NO_, 3, false>(__VA_ARGS__);               \
        if (k.H == 50) return FN<50, NO_, 3, false>(__VA_ARGS__);               \
        if (NO_ > 1) {                                                          \
            if (k.H == 5) return FN<5, (NO_ > 1 ? NO_ : 2), 3, false>(__VA_ARGS__); \
            return FN<0, (NO_ > 1 ? NO_ : 2), 3, false>(__VA_ARGS__);           \
        }                                                                       \
    } while (0)

// OCD_RUNTIME_H=1 (tests and tuning, read at every launch): skip the compile-time H = 15 / 50 specialisations, i.e.
// run those horizons on the runtime-horizon segmented kernels every other horizon uses.
static bool runtime_h_forced() {
    const char *e = std::getenv("OCD_RUNTIME_H");
    return e && e[0] == '1';
}

static int launch_solve(const KParams &k, bool precise, const SolveArgs &a, cudaStream_t st) {
    if (precise) OCD_DISPATCH(launch_solve_t, true, k, a, st);
    if (k.L == 3 && k.NO >= 1 && k.NO <= 5 && !((k.H == 15 || k.H == 50) && runtime_h_forced())) {
        switch (k.NO) {
            case 1: OCD_SOLVE_SWITCH(launch_solve_t, 1, k, a, st); break;
            case 2: OCD_SOLVE_SWITCH(launch_solve_t, 2, k, a, st); break;
            case 3: OCD_SOLVE_SWITCH(launch_solve_t, 3, k, a, st); break;
            case 4: OCD_SOLVE_SWITCH(launch_solve_t, 4, k, a, st); break;
            default: OCD_SOLVE_SWITCH(launch_solve_t, 5, k, a, st); break;
        }
    }
    OCD_DISPATCH(launch_solve_t, false, k, a, st);
}

// the solve's own dispatch: the reverse pass re-runs the iterations of the specialisation the forward ran
static int launch_solve_vjp(const KParams &k, bool precise, const VjpArgs &a, cudaStream_t st) {
    if (precise) OCD_DISPATCH(launch_solve_vjp_t, true, k, a, st);
    if (k.L == 3 && k.NO >= 1 && k.NO <= 5 && !((k.H == 15 || k.H == 50) && runtime_h_forced())) {
        switch (k.NO) {
            case 1: OCD_SOLVE_SWITCH(launch_solve_vjp_t, 1, k, a, st); break;
            case 2: OCD_SOLVE_SWITCH(launch_solve_vjp_t, 2, k, a, st); break;
            case 3: OCD_SOLVE_SWITCH(launch_solve_vjp_t, 3, k, a, st); break;
            case 4: OCD_SOLVE_SWITCH(launch_solve_vjp_t, 4, k, a, st); break;
            default: OCD_SOLVE_SWITCH(launch_solve_vjp_t, 5, k, a, st); break;
        }
    }
    OCD_DISPATCH(launch_solve_vjp_t, false, k, a, st);
}

static int launch_episode(const KParams &k, bool precise, const ocd_scenario &sc, const EpisodeArgs &a,
                          cudaStream_t st) {
    if (precise) OCD_DISPATCH(launch_episode_t, true, k, sc, a, st);
    OCD_DISPATCH(launch_episode_t, false, k, sc, a, st);
}

// the episode's own dispatch: the reverse pass re-runs the iterations of the specialisation k_episode ran
static int launch_episode_jac(const KParams &k, bool precise, const ocd_scenario &sc, const EpisodeVjpArgs &a,
                              int group, cudaStream_t st) {
    if (precise) OCD_DISPATCH(launch_episode_jac_t, true, k, sc, a, group, st);
    OCD_DISPATCH(launch_episode_jac_t, false, k, sc, a, group, st);
}

// the same two dispatches, asking which kernel form would run (ocd_kernel_form)
static int form_of(const KParams &k, bool precise, long long B, bool episode) {
    if (precise) OCD_DISPATCH(form_t, true, k, B, episode);
    if (!episode && k.L == 3 && k.NO >= 1 && k.NO <= 5 && !((k.H == 15 || k.H == 50) && runtime_h_forced())) {
        switch (k.NO) {
            case 1: OCD_SOLVE_SWITCH(form_t, 1, k, B, false); break;
            case 2: OCD_SOLVE_SWITCH(form_t, 2, k, B, false); break;
            case 3: OCD_SOLVE_SWITCH(form_t, 3, k, B, false); break;
            case 4: OCD_SOLVE_SWITCH(form_t, 4, k, B, false); break;
            default: OCD_SOLVE_SWITCH(form_t, 5, k, B, false); break;
        }
    }
    OCD_DISPATCH(form_t, false, k, B, episode);
}

}  // namespace ocd

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
using namespace ocd;

extern "C" {

int ocd_abi_version(void) { return OCD_ABI_VERSION; }

const char *ocd_strerror(int code) {
    switch (code) {
        case OCD_OK: return "ok";
        case OCD_EINVAL: return "invalid argument";
        case OCD_EUNSUP: return "unsupported problem shape (H, C or L out of range)";
        case OCD_ECUDA: return "CUDA error (no device, or launch/copy failure)";
        case OCD_ENOMEM: return "out of memory";
        default: return "unknown error";
    }
}

int ocd_num_starts(const ocd_params *p) { return (p && p->extra_inits) ? 6 : 3; }

int ocd_kernel_form(const ocd_params *p, int64_t B, int episode) {
    KParams k;
    const int rc = digest(p, k);
    if (rc) return rc;
    if (B < 0) return OCD_EINVAL;
    if (k.optimizer == 1) return episode ? (int)OCD_EUNSUP : (int)OCD_FORM_THROUGHPUT;     // k_solve_lbfgs has one form
    return form_of(k, p->math_mode == 1, B, episode != 0);
}

int ocd_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int ocd_dynamics_step_batch(const float *state, const float *control, float dt, float friction,
                            const float *friction_b, float *next_state, int64_t B, void *stream) {
    if (B == 0) return OCD_OK;
    if (!state || !control || !next_state || B < 0) return OCD_EINVAL;
    const float dt2 = (float)((double)dt * (double)dt);
    k_dynamics<true><<<(unsigned)((B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        state, control, dt, dt2, friction, friction_b, next_state, B);
    return cuda_status();
}

int ocd_smooth_batch(int kind, const float *z, double p0, double p1, float *out, int64_t B, void *stream) {
    if (B == 0) return OCD_OK;
    if (!z || !out || B < 0) return OCD_EINVAL;
    float a, b = 0.0f, c = 0.0f;
    if (kind == OCD_SMOOTH_F) {
        a = (float)p0;
    } else if (kind == OCD_SMOOTH_THRESHOLD) {
        if (!(p1 > 0.0)) return OCD_EINVAL;
        a = (float)(p0 - p1);          // Python-double difference, cast once (math_utils.py:92)
        b = (float)p1;
        c = (float)(5.0 / p1);
    } else if (kind == OCD_SMOOTH_BUMP) {
        a = (float)p0;
        b = (float)p1;
    } else {
        return OCD_EINVAL;
    }
    k_smooth<<<(unsigned)((B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(kind, z, a, b, c, out, B);
    return cuda_status();
}

int ocd_features_batch(const ocd_params *p, const float *world, float *phi, int64_t B, void *stream) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (B == 0) return OCD_OK;
    if (!world || !phi || B < 0) return OCD_EINVAL;
    if (4 * B > 0x7fffffffLL) return OCD_EUNSUP;
    const unsigned grid = (unsigned)((B + 127) / 128);
    if (p->math_mode == 1) k_features<true><<<grid, 128, 0, (cudaStream_t)stream>>>(k, world, phi, B);
    else k_features<false><<<grid, 128, 0, (cudaStream_t)stream>>>(k, world, phi, B);
    return cuda_status();
}

int ocd_reward_grad_batch(const ocd_params *p, const float *world, const float *controls,
                          const float *other_controls, int64_t Bo, const float *weights, int64_t Bw,
                          const int32_t *weight_idx, float *reward, float *grad, int64_t B, void *stream) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (B == 0) return OCD_OK;
    if (!world || !controls || !reward || B < 0) return OCD_EINVAL;
    if ((rc = check_weights(weights, Bw, weight_idx, B))) return rc;
    if (k.other_mode == 1 && (!other_controls || (Bo != 1 && Bo != B))) return OCD_EINVAL;
    if (B == 0) return OCD_OK;
    const unsigned grid = (unsigned)((B + 127) / 128);
    if (p->math_mode == 1)
        k_reward_grad<true><<<grid, 128, 0, (cudaStream_t)stream>>>(k, world, controls, other_controls, Bo, weights,
                                                                    Bw, weight_idx, reward, grad, B, 0);
    else
        k_reward_grad<false><<<grid, 128, 0, (cudaStream_t)stream>>>(k, world, controls, other_controls, Bo, weights,
                                                                     Bw, weight_idx, reward, grad, B, 0);
    return cuda_status();
}

int ocd_feature_jacobian_batch(const ocd_params *p, const float *world, const float *controls,
                               const float *other_controls, int64_t Bo, float *phi_sum, float *jac, int64_t B,
                               void *stream) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (B == 0) return OCD_OK;
    if (!world || !controls || !phi_sum || !jac || B < 0) return OCD_EINVAL;
    if (k.other_mode == 1 && (!other_controls || (Bo != 1 && Bo != B))) return OCD_EINVAL;
    float *eye = nullptr;
    if (cudaGetSymbolAddress((void **)&eye, g_onehot) != cudaSuccess) {
        cudaGetLastError();
        return OCD_ECUDA;
    }
    constexpr int KM = OCD_MAX_LANES + 4;
    // row i: the reward with weights e_i is the summed feature i; the K rows are the K slices of ONE 2-D grid
    const dim3 grid((unsigned)((B + 127) / 128), (unsigned)k.K);
    if (p->math_mode == 1)
        k_reward_grad<true><<<grid, 128, 0, (cudaStream_t)stream>>>(k, world, controls, other_controls, Bo, eye, 1,
                                                                    nullptr, phi_sum, jac, B, KM);
    else
        k_reward_grad<false><<<grid, 128, 0, (cudaStream_t)stream>>>(k, world, controls, other_controls, Bo, eye, 1,
                                                                     nullptr, phi_sum, jac, B, KM);
    return cuda_status();
}

int ocd_feature_hessian_batch(const ocd_params *p, const float *world, const float *controls,
                              const float *other_controls, int64_t Bo, float *hess, int64_t B, void *stream) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (B == 0) return OCD_OK;
    if (!world || !controls || !hess || B < 0) return OCD_EINVAL;
    if (k.other_mode == 1 && (!other_controls || (Bo != 1 && Bo != B))) return OCD_EINVAL;
    const int n = 2 * k.H;
    if (n * (n + 1) / 2 > 65535) return OCD_EUNSUP;
    const dim3 grid((unsigned)((B + 127) / 128), (unsigned)(n * (n + 1) / 2));     // one slice per control pair i <= j
    k_feature_hessian<<<grid, 128, 0, (cudaStream_t)stream>>>(k, world, controls, other_controls, Bo, hess, B);
    return cuda_status();
}

int ocd_solve_batch(const ocd_params *p, const float *world, const float *other_controls, int64_t Bo,
                    const float *weights, int64_t Bw, const int32_t *weight_idx, const float *cur_speed,
                    float *plan, float *losses, int32_t *best, float *all_plans, int64_t B, void *stream) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (B == 0) return OCD_OK;
    if (!world || !plan || !losses || !best || B < 0) return OCD_EINVAL;
    if ((rc = check_weights(weights, Bw, weight_idx, B))) return rc;
    if (k.other_mode == 1 && (!other_controls || (Bo != 1 && Bo != B))) return OCD_EINVAL;
    SolveArgs a{world, other_controls, Bo, weights, Bw, weight_idx, cur_speed, plan, losses, best, all_plans,
                B, pick_P(B)};
    if (k.optimizer == 1) {
        const size_t bytes = smem_floats(k.H, k.NO, k.K, k.S, kP, false, false, false) * sizeof(float);
        if ((rc = prepare_smem(k_solve_lbfgs, bytes))) return rc;
        k_solve_lbfgs<<<(unsigned)((B + kP - 1) / kP), k.S * kP, bytes, (cudaStream_t)stream>>>(k, a);
        return cuda_status();
    }
    return launch_solve(k, p->math_mode == 1, a, (cudaStream_t)stream);
}

static size_t vjp_workspace_bytes(const KParams &k, int64_t B) {
    return (size_t)k.n_iter * (size_t)k.H * 2 * (size_t)B * sizeof(float);
}

int ocd_solve_vjp_workspace_bytes(const ocd_params *p, int64_t B, size_t *bytes) {
    KParams k;
    const int rc = digest(p, k);
    if (rc) return rc;
    if (!bytes || B < 0) return OCD_EINVAL;
    if (k.optimizer != 0) return OCD_EUNSUP;      // L-BFGS: its line search is not differentiable
    *bytes = vjp_workspace_bytes(k, B);
    return OCD_OK;
}

int ocd_solve_vjp_batch(const ocd_params *p, const float *world, const float *other_controls, int64_t Bo,
                        const float *weights, int64_t Bw, const int32_t *weight_idx, const float *cur_speed,
                        const int32_t *best, const float *plan_bar, float *weights_bar, float *world_bar,
                        void *workspace, size_t workspace_bytes, int64_t B, void *stream) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (k.optimizer != 0) return OCD_EUNSUP;
    if (B == 0) return OCD_OK;
    if (!world || !best || !plan_bar || !weights_bar || B < 0) return OCD_EINVAL;
    if ((rc = check_weights(weights, Bw, weight_idx, B))) return rc;
    if (k.other_mode == 1 && (!other_controls || (Bo != 1 && Bo != B))) return OCD_EINVAL;
    const size_t need = vjp_workspace_bytes(k, B);
    if (workspace_bytes < need || (need > 0 && !workspace)) return OCD_EINVAL;
    VjpArgs a{world, other_controls, Bo, weights, Bw, weight_idx, cur_speed, best, plan_bar, weights_bar, world_bar,
              static_cast<float *>(workspace), B};
    return launch_solve_vjp(k, p->math_mode == 1, a, (cudaStream_t)stream);
}

int ocd_episode_batch(const ocd_params *p, const ocd_scenario *sc, const float *robot_init,
                      const float *other_init, const float *plan_weights, int64_t Bw,
                      const int32_t *weight_idx, const float *true_weights, const int32_t *unlucky_idx,
                      int32_t t0, int32_t T, float *returns, float *traj_controls, int32_t *traj_best,
                      float *traj_states, float *final_world, int64_t B, void *stream) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (B == 0) return OCD_OK;
    if (!sc || !robot_init || !true_weights || !returns || B < 0 || T < 0 || t0 < 0) return OCD_EINVAL;
    if (sc->n_other != k.NO) return OCD_EINVAL;
    if (k.optimizer != 0) return OCD_EUNSUP;      // the episode loop runs the reference's SGD planner only
    for (int j = 0; j < k.NO; ++j)
        if (sc->plan_len[j] < 0 || sc->plan_len[j] > OCD_MAX_PLAN || (sc->kind[j] != 0 && sc->kind[j] != 1))
            return OCD_EINVAL;
    if ((rc = check_weights(plan_weights, Bw, weight_idx, B))) return rc;
    if (B == 0) return OCD_OK;
    EpisodeArgs a{robot_init, other_init, plan_weights, Bw, weight_idx, true_weights, unlucky_idx, t0, T,
                  returns, traj_controls, traj_best, traj_states, final_world, B, pick_P(B)};
    return launch_episode(k, p->math_mode == 1, *sc, a, (cudaStream_t)stream);
}

// workspace of ocd_episode_vjp_batch: the Jacobian rows [T][2][K + 4][B], then the iterates of the steps in flight,
// [N + 1][H][2][B] per step
static size_t episode_jac_bytes(const KParams &k, int32_t T, int64_t B) {
    return (size_t)T * 2 * (size_t)(k.K + 4) * (size_t)B * sizeof(float);
}
static size_t episode_step_bytes(const KParams &k, int64_t B) {
    return (size_t)(k.n_iter + 1) * (size_t)k.H * 2 * (size_t)B * sizeof(float);
}

int ocd_episode_vjp_workspace_bytes(const ocd_params *p, int32_t T, int64_t B, size_t *min_bytes, size_t *full_bytes) {
    KParams k;
    const int rc = digest(p, k);
    if (rc) return rc;
    if (!min_bytes || !full_bytes || B < 0 || T < 0) return OCD_EINVAL;
    if (k.optimizer != 0) return OCD_EUNSUP;      // L-BFGS: its line search is not differentiable
    const size_t jac = episode_jac_bytes(k, T, B), step = episode_step_bytes(k, B);
    *min_bytes = jac + (T > 0 ? step : 0);
    *full_bytes = jac + (size_t)T * step;
    return OCD_OK;
}

int ocd_episode_vjp_batch(const ocd_params *p, const ocd_scenario *sc, const float *plan_weights, int64_t Bw,
                          const int32_t *weight_idx, const float *true_weights, int32_t T, const float *traj_states,
                          const int32_t *traj_best, const float *traj_controls, const float *returns_bar,
                          float *plan_weights_bar, float *robot_init_bar, float *true_weights_bar, void *workspace,
                          size_t workspace_bytes, int64_t B, void *stream) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (k.optimizer != 0) return OCD_EUNSUP;
    if (B == 0) return OCD_OK;
    if (!sc || !true_weights || !returns_bar || !plan_weights_bar || B < 0 || T < 0) return OCD_EINVAL;
    if (T > 0 && (!traj_states || !traj_best || !traj_controls)) return OCD_EINVAL;
    if (sc->n_other != k.NO) return OCD_EINVAL;
    for (int j = 0; j < k.NO; ++j)
        if (sc->plan_len[j] < 0 || sc->plan_len[j] > OCD_MAX_PLAN || (sc->kind[j] != 0 && sc->kind[j] != 1))
            return OCD_EINVAL;
    if ((rc = check_weights(plan_weights, Bw, weight_idx, B))) return rc;
    const size_t jac = episode_jac_bytes(k, T, B), step = episode_step_bytes(k, B);
    const size_t need = jac + (T > 0 ? step : 0);
    if (workspace_bytes < need || (need > 0 && !workspace)) return OCD_EINVAL;
    EpisodeVjpArgs a{plan_weights, Bw, weight_idx, true_weights, T, 0, traj_states, traj_best, traj_controls,
                     returns_bar, plan_weights_bar, robot_init_bar, true_weights_bar, static_cast<float *>(workspace),
                     reinterpret_cast<float *>(static_cast<char *>(workspace) + jac), B};
    const cudaStream_t st = (cudaStream_t)stream;
    if (T > 0) {
        // as many steps in flight as the workspace holds (at most 65 535: gridDim.y)
        size_t group = (workspace_bytes - jac) / step;
        if (group > (size_t)T) group = (size_t)T;
        if (group > 65535) group = 65535;
        if ((rc = launch_episode_jac(k, p->math_mode == 1, *sc, a, (int)group, st))) return rc;
    }
    k_episode_adjoint<<<(unsigned)((B + kVjpThreads - 1) / kVjpThreads), kVjpThreads, 0, st>>>(k, a);
    return cuda_status();
}

// ---- host-buffer layer ------------------------------------------------------------------------
static constexpr int kCtxStreams = 4;     // H2D, two compute lanes, D2H
static constexpr int kMaxChunks = 16;

struct CopyPool;
static CopyPool *copy_pool_new();
static void copy_pool_free(CopyPool *);

struct ocd_ctx {
    int device;
    cudaStream_t stream;                 // small calls (episodes)
    cudaStream_t lanes[kCtxStreams];     // the chunk pipeline of ocd_solve_batch_host
    cudaEvent_t loaded[kMaxChunks];      // chunk c's inputs are on the device
    cudaEvent_t solved[kMaxChunks];      // chunk c's kernel has finished
    cudaEvent_t done[kMaxChunks];        // chunk c's outputs are in host memory
    char *dev;      size_t dev_cap;
    char *pin;      size_t pin_cap;
    CopyPool *pool;                      // staging-copy workers (created on the first large copy)
    // ocd_episode_batch_host: the copy-in / episode kernel / copy-out sequence of the last call, captured as a CUDA graph
    // and replayed while the call's signature (every argument but the array contents) and the buffers stay the same --
    // a CMA-ES run makes the same call once per generation
    cudaGraphExec_t ep_graph;
    std::vector<unsigned char> ep_sig;
    char *ep_dev, *ep_pin;               // buffers the captured graph points into
};

static int ctx_reserve(ocd_ctx *c, size_t dev_bytes, size_t pin_bytes) {
    if (dev_bytes > c->dev_cap) {
        if (c->dev) cudaFree(c->dev);
        c->dev = nullptr; c->dev_cap = 0;
        if (cudaMalloc((void **)&c->dev, dev_bytes) != cudaSuccess) { cudaGetLastError(); return OCD_ENOMEM; }
        c->dev_cap = dev_bytes;
    }
    if (pin_bytes > c->pin_cap) {
        if (c->pin) cudaFreeHost(c->pin);
        c->pin = nullptr; c->pin_cap = 0;
        if (cudaMallocHost((void **)&c->pin, pin_bytes) != cudaSuccess) { cudaGetLastError(); return OCD_ENOMEM; }
        c->pin_cap = pin_bytes;
    }
    return OCD_OK;
}

int ocd_ctx_create(int device, ocd_ctx **out) {
    if (!out) return OCD_EINVAL;
    *out = nullptr;
    if (device < 0 || device >= ocd_device_count()) return OCD_ECUDA;
    if (cudaSetDevice(device) != cudaSuccess) return OCD_ECUDA;
    ocd_ctx *c = new (std::nothrow) ocd_ctx();
    if (!c) return OCD_ENOMEM;
    c->device = device;
    c->pool = copy_pool_new();
    c->ep_graph = nullptr;
    c->ep_dev = c->ep_pin = nullptr;
    bool ok = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < kCtxStreams; ++i)
        ok = ok && cudaStreamCreateWithFlags(&c->lanes[i], cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < kMaxChunks; ++i)
        ok = ok && cudaEventCreateWithFlags(&c->done[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c->loaded[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&c->solved[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        cudaGetLastError();
        copy_pool_free(c->pool);
        delete c;
        return OCD_ECUDA;
    }
    *out = c;
    return OCD_OK;
}

void ocd_ctx_destroy(ocd_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    copy_pool_free(c->pool);
    if (c->ep_graph) cudaGraphExecDestroy(c->ep_graph);
    if (c->dev) cudaFree(c->dev);
    if (c->pin) cudaFreeHost(c->pin);
    cudaStreamDestroy(c->stream);
    for (int i = 0; i < kCtxStreams; ++i) cudaStreamDestroy(c->lanes[i]);
    for (int i = 0; i < kMaxChunks; ++i) {
        cudaEventDestroy(c->done[i]);
        cudaEventDestroy(c->loaded[i]);
        cudaEventDestroy(c->solved[i]);
    }
    delete c;
}

// a tiny bump allocator over the ctx buffers
struct Arena {
    size_t off = 0;
    size_t take(size_t bytes) {
        const size_t at = off;
        off += (bytes + 255) & ~(size_t)255;
        return at;
    }
};

// true when `ptr` is page-locked host memory the copy engines can read or write directly
int ocd_host_register(void *ptr, size_t bytes) {
    if (!ptr || bytes == 0) return OCD_EINVAL;
    if (cudaHostRegister(ptr, bytes, cudaHostRegisterPortable) != cudaSuccess) {
        cudaGetLastError();
        return OCD_ECUDA;
    }
    return OCD_OK;
}

int ocd_host_unregister(void *ptr) {
    if (!ptr) return OCD_EINVAL;
    if (cudaHostUnregister(ptr) != cudaSuccess) {
        cudaGetLastError();
        return OCD_ECUDA;
    }
    return OCD_OK;
}

static bool is_pinned(const void *ptr) {
    if (!ptr) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// Column chunks of the host-buffer solve: start[0..n] with start[n] = B, every boundary a multiple of 64
// problems (256-byte aligned rows).  Small batches are one chunk.  Large ones ramp up and down -- weights
// 1,2,4,6,...,6,4,2,1 -- so that the first kernel starts after a short copy and only a short copy is left
// when the last kernel ends, while the middle chunks are several full waves each.
// OCD_HOST_CHUNKS="w0,w1,..." overrides the weights (tuning knob, read at every call).
static int chunk_schedule(int64_t B, int64_t *start) {
    int w[kMaxChunks], n = 0;
    if (const char *e = std::getenv("OCD_HOST_CHUNKS")) {
        for (const char *q = e; *q && n < kMaxChunks;) {
            char *end;
            const long v = std::strtol(q, &end, 10);
            if (end == q) break;
            if (v > 0) w[n++] = (int)v;
            q = (*end == ',') ? end + 1 : end;
        }
    }
    if (n == 0) {
        if (B <= 65536) {
            w[n++] = 1;
        } else if (B <= 262144) {
            for (int i = 0; i < 4; ++i) w[n++] = 1;
        } else {
            const int ramp[] = {1, 2, 4, 6, 6, 6, 4, 2, 1};
            for (int v : ramp) w[n++] = v;
        }
    }
    int64_t tot = 0;
    for (int i = 0; i < n; ++i) tot += w[i];
    int64_t acc = 0;
    int m = 0;
    start[0] = 0;
    for (int i = 0; i < n; ++i) {
        acc += w[i];
        int64_t e = (i == n - 1) ? B : ((B * acc / tot) + 63) / 64 * 64;
        if (e > B) e = B;
        if (e > start[m]) start[++m] = e;
    }
    if (start[m] != B) start[++m] = B;
    return m;
}

// Staging copies between pageable user arrays and the context's pinned area: `rows` row segments of `bytes`
// bytes each.  One core moves ~10 GB/s, far less than the PCIe link, so copies above 1 MiB are cut into slices
// (by bytes, not by rows: a chunk has as few as one row) that the context's worker threads and the caller take
// from a shared counter.  The workers are created once per context, on the first large copy: a thread per copy
// cost more than the copy (a 2^20-problem call makes ~40 such copies).
struct CopyJob {
    char *dst; const char *src;
    size_t dst_stride, src_stride, bytes, total, slice, nslices;
    std::atomic<size_t> next{0}, done{0};
    void span(size_t lo, size_t hi) const {                   // bytes [lo, hi) of the rows laid end to end
        while (lo < hi) {
            const size_t r = lo / bytes, off = lo % bytes;
            const size_t len = (bytes - off < hi - lo) ? bytes - off : hi - lo;
            std::memcpy(dst + r * dst_stride + off, src + r * src_stride + off, len);
            lo += len;
        }
    }
    void work() {                                             // take slices until none is left
        for (;;) {
            const size_t i = next.fetch_add(1);
            if (i >= nslices) return;
            const size_t lo = i * slice, hi = lo + slice < total ? lo + slice : total;
            span(lo, hi);
            done.fetch_add(1);
        }
    }
};

struct CopyPool {
    std::vector<std::thread> workers;
    std::mutex m;
    std::condition_variable cv;
    std::shared_ptr<CopyJob> job;       // the current job; a late worker keeps its (exhausted) job alive on its own
    uint64_t gen = 0;
    bool stop = false;

    void run() {
        uint64_t seen = 0;
        for (;;) {
            std::shared_ptr<CopyJob> j;
            {
                std::unique_lock<std::mutex> lk(m);
                cv.wait(lk, [&] { return stop || gen != seen; });
                if (stop) return;
                seen = gen;
                j = job;
            }
            if (j) j->work();
        }
    }
    bool start(unsigned n) {            // false: no workers (the caller copies alone)
        if (!workers.empty()) return true;
        try {
            workers.reserve(n);
            for (unsigned i = 0; i < n; ++i) workers.emplace_back([this] { run(); });
        } catch (...) {
        }
        return !workers.empty();
    }
    void shutdown() {
        {
            std::lock_guard<std::mutex> lk(m);
            stop = true;
        }
        cv.notify_all();
        for (std::thread &t : workers) t.join();
        workers.clear();
    }
};

static CopyPool *copy_pool_new() { return new (std::nothrow) CopyPool(); }
static void copy_pool_free(CopyPool *p) {
    if (!p) return;
    p->shutdown();
    delete p;
}

// Staging-copy workers beside the caller: from the cores THIS process may run on (its affinity mask -- with one
// process per GPU each rank owns a slice of the host, and eight ranks sizing their pools from the whole machine
// oversubscribed it: 7 workers x 8 ranks on 32 cores), at most 7.  OCD_HOST_THREADS=<n> (copy threads, caller
// included) overrides it.
static unsigned copy_workers() {
    if (const char *e = std::getenv("OCD_HOST_THREADS")) {
        const long v = std::strtol(e, nullptr, 10);
        if (v >= 1) return (unsigned)(v - 1 > 15 ? 15 : v - 1);
    }
    unsigned cores = 0;
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof(set), &set) == 0) cores = (unsigned)CPU_COUNT(&set);
    if (!cores) cores = std::thread::hardware_concurrency();
    if (cores < 2) return 0;
    return cores - 1 > 7 ? 7 : cores - 1;
}

static void copy_rows(CopyPool *pool, char *dst, size_t dst_stride, const char *src, size_t src_stride, int rows,
                      size_t bytes) {
    const size_t total = (size_t)rows * bytes;
    CopyJob local{dst, src, dst_stride, src_stride, bytes, total, total, 1};
    if (!pool || total < (1u << 20)) {
        local.span(0, total);
        return;
    }
    const unsigned nw = copy_workers();                                       // workers beside the caller
    std::shared_ptr<CopyJob> j;
    try {                                                                     // nothing may throw across the C ABI
        if (nw && pool->start(nw)) j = std::make_shared<CopyJob>();
    } catch (...) {
    }
    if (!j) {
        local.span(0, total);
        return;
    }
    j->dst = dst; j->src = src; j->dst_stride = dst_stride; j->src_stride = src_stride; j->bytes = bytes; j->total = total;
    j->slice = (size_t)512 << 10;                                             // 512 KiB slices
    j->nslices = (total + j->slice - 1) / j->slice;
    {
        std::lock_guard<std::mutex> lk(pool->m);
        pool->job = j;
        ++pool->gen;
    }
    pool->cv.notify_all();
    j->work();
    while (j->done.load() < j->nslices) std::this_thread::yield();           // the last slices are in flight
}

// One [rows][B] host array moved in column chunks.  Pinned user memory is copied in place (a
// strided 2-D copy); pageable memory goes through the context's pinned staging area.
struct HostArray {
    char  *user;        // host array [rows][B] of `elem`-byte items (null: absent)
    int    rows;        // rows of the device buffer
    size_t elem;
    bool   pinned;
    size_t dev_off, pin_off;    // per-chunk compact [rows][n] buffers in the device / pinned arena
    int    rows_out = -1;       // outputs: rows copied back to `user` ([rows_out][B]; -1: all of them)
    bool   dev_only = false;    // output the caller did not ask for: the kernel writes it, nothing comes back
    int    out_rows() const { return rows_out < 0 ? rows : rows_out; }
};

static int h2d_chunk(ocd_ctx *c, const HostArray &a, int64_t B, int64_t b0, int64_t n, cudaStream_t st) {
    if (!a.user) return OCD_OK;
    char *dst = c->dev + a.dev_off + (size_t)a.rows * b0 * a.elem;     // chunks are packed back to back
    cudaError_t e;
    if (a.pinned) {
        e = cudaMemcpy2DAsync(dst, n * a.elem, a.user + b0 * a.elem, B * a.elem, n * a.elem, a.rows,
                              cudaMemcpyHostToDevice, st);
    } else {
        char *stage = c->pin + a.pin_off + (size_t)a.rows * b0 * a.elem;
        copy_rows(c->pool, stage, n * a.elem, a.user + b0 * a.elem, B * a.elem, a.rows, n * a.elem);
        e = cudaMemcpyAsync(dst, stage, (size_t)a.rows * n * a.elem, cudaMemcpyHostToDevice, st);
    }
    return e == cudaSuccess ? OCD_OK : OCD_ECUDA;
}

static int d2h_chunk(ocd_ctx *c, const HostArray &a, int64_t B, int64_t b0, int64_t n, cudaStream_t st) {
    if (a.dev_only) return OCD_OK;
    const char *src = c->dev + a.dev_off + (size_t)a.rows * b0 * a.elem;     // the first out_rows() rows of the chunk
    cudaError_t e;
    if (a.pinned)
        e = cudaMemcpy2DAsync(a.user + b0 * a.elem, B * a.elem, src, n * a.elem, n * a.elem, a.out_rows(),
                              cudaMemcpyDeviceToHost, st);
    else
        e = cudaMemcpyAsync(c->pin + a.pin_off + (size_t)a.rows * b0 * a.elem, src,
                            (size_t)a.out_rows() * n * a.elem, cudaMemcpyDeviceToHost, st);
    return e == cudaSuccess ? OCD_OK : OCD_ECUDA;
}

static void unstage_chunk(ocd_ctx *c, const HostArray &a, int64_t B, int64_t b0, int64_t n) {
    if (a.pinned || a.dev_only) return;
    const char *stage = c->pin + a.pin_off + (size_t)a.rows * b0 * a.elem;
    copy_rows(c->pool, a.user + b0 * a.elem, B * a.elem, stage, n * a.elem, a.out_rows(), n * a.elem);
}

// The batch is cut into column chunks that flow through four streams linked by per-chunk events: one
// stream feeds the H2D copy engine (running ahead as far as it can -- every chunk has its own device
// buffers), two compute lanes take the chunks alternately (so that one kernel's tail wave is filled by the
// next kernel's blocks), one stream drains results through the D2H copy engine.  The SMs never wait for
// a copy after the first chunk and the call costs about max(copy, solve) instead of their sum.
// plan_rows: rows of the plan [H][2][B] that travel back (2 H: the whole plan; 2: the first control only);
// losses / best may be null when plan_rows == 2 (the kernel still writes them on the device, nothing comes back).
static int solve_host(ocd_ctx *c, const ocd_params *p, const float *world, const float *other_controls,
                      int64_t Bo, const float *weights, int64_t Bw, const int32_t *weight_idx,
                      const float *cur_speed, float *plan, int plan_rows, float *losses, int32_t *best, int64_t B) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (B == 0) return OCD_OK;
    if (!c || !world || !plan || B < 0) return OCD_EINVAL;
    if (plan_rows != 2 && (!losses || !best)) return OCD_EINVAL;
    if ((rc = check_weights(weights, Bw, weight_idx, B))) return rc;
    if (k.other_mode == 1 && (!other_controls || (Bo != 1 && Bo != B))) return OCD_EINVAL;
    if (cudaSetDevice(c->device) != cudaSuccess) return OCD_ECUDA;
    const int C = k.NO + 1;
    const bool per_problem_w = !weight_idx && Bw == B && B > 1;     // weights travel with the chunks
    const bool per_problem_oc = k.other_mode == 1 && Bo == B && B > 1;

    int64_t start[kMaxChunks + 1];
    const int nchunks = chunk_schedule(B, start);

    HostArray a_world{(char *)world, C * 4, 4, is_pinned(world), 0, 0};
    HostArray a_idx{(char *)weight_idx, 1, 4, is_pinned(weight_idx), 0, 0};
    HostArray a_w{per_problem_w ? (char *)weights : nullptr, k.K, 4, is_pinned(weights), 0, 0};
    HostArray a_oc{per_problem_oc ? (char *)other_controls : nullptr, k.NO * k.H * 2, 4, is_pinned(other_controls), 0, 0};
    HostArray a_cs{(char *)cur_speed, 1, 4, is_pinned(cur_speed), 0, 0};
    HostArray a_plan{(char *)plan, k.H * 2, 4, is_pinned(plan), 0, 0, plan_rows};
    HostArray a_loss{(char *)losses, k.S, 4, is_pinned(losses), 0, 0, -1, losses == nullptr};
    HostArray a_best{(char *)best, 1, 4, is_pinned(best), 0, 0, -1, best == nullptr};
    HostArray *arrays[] = {&a_world, &a_idx, &a_w, &a_oc, &a_cs, &a_plan, &a_loss, &a_best};
    Arena dev, pin;
    for (HostArray *a : arrays)
        if (a->user || a->dev_only) {
            a->dev_off = dev.take((size_t)a->rows * B * a->elem);
            if (!a->pinned && !a->dev_only) a->pin_off = pin.take((size_t)a->rows * B * a->elem);
        }
    // shared (not per-problem) inputs: copied once, in full -- straight from the user's array when it is
    // page-locked, through the staging area otherwise
    const size_t n_w = per_problem_w ? 0 : sizeof(float) * k.K * Bw;
    const size_t n_oc = (k.other_mode == 1 && !per_problem_oc) ? sizeof(float) * k.NO * k.H * 2 * Bo : 0;
    const bool pin_w = n_w && is_pinned(weights), pin_oc = n_oc && is_pinned(other_controls);
    const size_t o_w = dev.take(n_w), s_w = pin.take(pin_w ? 0 : n_w);
    const size_t o_oc = dev.take(n_oc), s_oc = pin.take(pin_oc ? 0 : n_oc);
    if ((rc = ctx_reserve(c, dev.off, pin.off))) return rc;
    if (n_w && !pin_w) copy_rows(c->pool, c->pin + s_w, n_w, (const char *)weights, n_w, 1, n_w);
    if (n_oc && !pin_oc) std::memcpy(c->pin + s_oc, other_controls, n_oc);
    cudaStream_t s0 = c->lanes[0];        // the H2D stream: chunk copies are ordered behind the shared inputs
    if (n_w && cudaMemcpyAsync(c->dev + o_w, pin_w ? (const char *)weights : c->pin + s_w, n_w, cudaMemcpyHostToDevice,
                               s0) != cudaSuccess)
        return OCD_ECUDA;
    if (n_oc && cudaMemcpyAsync(c->dev + o_oc, pin_oc ? (const char *)other_controls : c->pin + s_oc, n_oc,
                                cudaMemcpyHostToDevice, s0) != cudaSuccess)
        return OCD_ECUDA;

    auto chunk_ptr = [&](const HostArray &a, int ch) -> char * {
        return (a.user || a.dev_only) ? c->dev + a.dev_off + (size_t)a.rows * start[ch] * a.elem : nullptr;
    };
    cudaStream_t s_in = c->lanes[0], s_out = c->lanes[3];
    for (int ch = 0; ch < nchunks && rc == OCD_OK; ++ch) {
        const int64_t b0 = start[ch], n = start[ch + 1] - b0;
        cudaStream_t st = c->lanes[1 + (ch & 1)];
        // the chunk's indices are validated right before they go up: the scan of a later chunk overlaps the kernels of
        // the earlier ones (one pass over 2^20 indices ahead of the first copy cost 0.4 ms of a 4.9 ms call)
        if ((rc = check_host_idx(weight_idx ? weight_idx + b0 : nullptr, Bw, n))) break;
        for (HostArray *a : {&a_world, &a_idx, &a_w, &a_oc, &a_cs})
            if (rc == OCD_OK) rc = h2d_chunk(c, *a, B, b0, n, s_in);
        if (rc) break;
        if (cudaEventRecord(c->loaded[ch], s_in) != cudaSuccess ||
            cudaStreamWaitEvent(st, c->loaded[ch], 0) != cudaSuccess) { rc = OCD_ECUDA; break; }
        rc = ocd_solve_batch(p, (const float *)chunk_ptr(a_world, ch),
                             per_problem_oc ? (const float *)chunk_ptr(a_oc, ch) : (n_oc ? (const float *)(c->dev + o_oc) : nullptr),
                             per_problem_oc ? n : Bo,
                             per_problem_w ? (const float *)chunk_ptr(a_w, ch) : (const float *)(c->dev + o_w),
                             per_problem_w ? n : Bw, (const int32_t *)chunk_ptr(a_idx, ch),
                             (const float *)chunk_ptr(a_cs, ch), (float *)chunk_ptr(a_plan, ch),
                             (float *)chunk_ptr(a_loss, ch), (int32_t *)chunk_ptr(a_best, ch), nullptr, n, st);
        if (rc) break;
        if (cudaEventRecord(c->solved[ch], st) != cudaSuccess ||
            cudaStreamWaitEvent(s_out, c->solved[ch], 0) != cudaSuccess) { rc = OCD_ECUDA; break; }
        for (HostArray *a : {&a_plan, &a_loss, &a_best})
            if (rc == OCD_OK) rc = d2h_chunk(c, *a, B, b0, n, s_out);
        if (rc == OCD_OK && cudaEventRecord(c->done[ch], s_out) != cudaSuccess) rc = OCD_ECUDA;
    }
    if (rc) {
        cudaDeviceSynchronize();
        cudaGetLastError();
        return rc;
    }
    for (int ch = 0; ch < nchunks; ++ch) {
        if (cudaEventSynchronize(c->done[ch]) != cudaSuccess) { cudaGetLastError(); return OCD_ECUDA; }
        for (HostArray *a : {&a_plan, &a_loss, &a_best}) unstage_chunk(c, *a, B, start[ch], start[ch + 1] - start[ch]);
    }
    return OCD_OK;
}

int ocd_solve_batch_host(ocd_ctx *c, const ocd_params *p, const float *world, const float *other_controls,
                         int64_t Bo, const float *weights, int64_t Bw, const int32_t *weight_idx,
                         const float *cur_speed, float *plan, float *losses, int32_t *best, int64_t B) {
    if (!losses || !best) return OCD_EINVAL;
    return solve_host(c, p, world, other_controls, Bo, weights, Bw, weight_idx, cur_speed, plan, p ? 2 * p->H : 0, losses,
                      best, B);
}

int ocd_solve_first_host(ocd_ctx *c, const ocd_params *p, const float *world, const float *other_controls,
                         int64_t Bo, const float *weights, int64_t Bw, const int32_t *weight_idx,
                         const float *cur_speed, float *first_control, float *losses, int32_t *best, int64_t B) {
    return solve_host(c, p, world, other_controls, Bo, weights, Bw, weight_idx, cur_speed, first_control, 2, losses,
                      best, B);
}

int ocd_episode_batch_host(ocd_ctx *c, const ocd_params *p, const ocd_scenario *sc, const float *robot_init,
                           const float *other_init, const float *plan_weights, int64_t Bw,
                           const int32_t *weight_idx, const float *true_weights, const int32_t *unlucky_idx,
                           int32_t t0, int32_t T, float *returns, float *final_world, int64_t B) {
    KParams k;
    int rc = digest(p, k);
    if (rc) return rc;
    if (!c || !sc || !robot_init || !true_weights || !returns || B < 0) return OCD_EINVAL;
    if ((rc = check_weights(plan_weights, Bw, weight_idx, B))) return rc;
    if ((rc = check_host_idx(weight_idx, Bw, B))) return rc;
    if (B == 0) return OCD_OK;
    if (cudaSetDevice(c->device) != cudaSuccess) return OCD_ECUDA;
    const int C = k.NO + 1;
    Arena ar;
    const size_t n_ri = sizeof(float) * 4 * B, o_ri = ar.take(n_ri);
    const size_t n_oi = other_init ? sizeof(float) * k.NO * 4 * B : 0, o_oi = ar.take(n_oi);
    const size_t n_w = sizeof(float) * k.K * Bw, o_w = ar.take(n_w);
    const size_t n_idx = weight_idx ? sizeof(int32_t) * B : 0, o_idx = ar.take(n_idx);
    const size_t n_tw = sizeof(float) * k.K, o_tw = ar.take(n_tw);
    const size_t n_ul = unlucky_idx ? sizeof(int32_t) * B : 0, o_ul = ar.take(n_ul);
    const size_t in_end = ar.off;
    // outputs: returns, then the final worlds -- contiguous, one copy back
    const size_t n_ret = sizeof(float) * B, o_ret = ar.take(n_ret);
    const size_t n_fw = final_world ? sizeof(float) * C * 4 * B : 0, o_fw = ar.take(n_fw);
    const size_t out_bytes = ar.off - o_ret;
    if ((rc = ctx_reserve(c, ar.off, ar.off))) return rc;
    std::memcpy(c->pin + o_ri, robot_init, n_ri);
    if (n_oi) std::memcpy(c->pin + o_oi, other_init, n_oi);
    std::memcpy(c->pin + o_w, plan_weights, n_w);
    if (n_idx) std::memcpy(c->pin + o_idx, weight_idx, n_idx);
    std::memcpy(c->pin + o_tw, true_weights, n_tw);
    if (n_ul) std::memcpy(c->pin + o_ul, unlucky_idx, n_ul);

    // the call's signature: everything that shapes the launch sequence (not the array contents, which travel through
    // the pinned buffer the graph reads)
    std::vector<unsigned char> sig;
    auto put = [&](const void *q, size_t n) { sig.insert(sig.end(), (const unsigned char *)q, (const unsigned char *)q + n); };
    const int64_t dims[] = {B, Bw, t0, T, other_init != nullptr, weight_idx != nullptr, unlucky_idx != nullptr,
                            final_world != nullptr, forced_form()};
    put(p, sizeof(*p)); put(sc, sizeof(*sc)); put(dims, sizeof(dims));
    auto enqueue = [&](cudaStream_t st) -> int {
        if (cudaMemcpyAsync(c->dev, c->pin, in_end, cudaMemcpyHostToDevice, st) != cudaSuccess) return OCD_ECUDA;
        int r = ocd_episode_batch(p, sc, (const float *)(c->dev + o_ri), n_oi ? (const float *)(c->dev + o_oi) : nullptr,
                                  (const float *)(c->dev + o_w), Bw, n_idx ? (const int32_t *)(c->dev + o_idx) : nullptr,
                                  (const float *)(c->dev + o_tw), n_ul ? (const int32_t *)(c->dev + o_ul) : nullptr, t0, T,
                                  (float *)(c->dev + o_ret), nullptr, nullptr, nullptr,
                                  n_fw ? (float *)(c->dev + o_fw) : nullptr, B, st);
        if (r) return r;
        if (cudaMemcpyAsync(c->pin + o_ret, c->dev + o_ret, out_bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess)
            return OCD_ECUDA;
        return OCD_OK;
    };
    const bool replay = c->ep_graph && c->ep_dev == c->dev && c->ep_pin == c->pin && sig == c->ep_sig;
    if (replay) {
        if (cudaGraphLaunch(c->ep_graph, c->stream) != cudaSuccess) { cudaGetLastError(); return OCD_ECUDA; }
    } else {
        if (c->ep_graph) { cudaGraphExecDestroy(c->ep_graph); c->ep_graph = nullptr; }
        // first call with this signature: run it directly (a kernel whose shared-memory attribute is not yet set cannot
        // be configured inside a capture), then capture the same sequence for the calls to come
        if ((rc = enqueue(c->stream))) return rc;
        if (cudaStreamSynchronize(c->stream) != cudaSuccess) { cudaGetLastError(); return OCD_ECUDA; }
        cudaGraph_t g = nullptr;
        if (cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            const int r2 = enqueue(c->stream);
            const cudaError_t e = cudaStreamEndCapture(c->stream, &g);
            if (r2 == OCD_OK && e == cudaSuccess && g &&
                cudaGraphInstantiate(&c->ep_graph, g, nullptr, nullptr, 0) == cudaSuccess) {
                c->ep_sig = sig; c->ep_dev = c->dev; c->ep_pin = c->pin;
            } else {
                c->ep_graph = nullptr;
            }
            if (g) cudaGraphDestroy(g);
            cudaGetLastError();
        } else {
            cudaGetLastError();
        }
        std::memcpy(returns, c->pin + o_ret, n_ret);
        if (n_fw) std::memcpy(final_world, c->pin + o_fw, n_fw);
        return OCD_OK;
    }
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) { cudaGetLastError(); return OCD_ECUDA; }
    std::memcpy(returns, c->pin + o_ret, n_ret);
    if (n_fw) std::memcpy(final_world, c->pin + o_fw, n_fw);
    return OCD_OK;
}

int ocd_fp32_peak(int iters, double *flops, void *stream) {
    if (!flops || iters < 1) return OCD_EINVAL;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return OCD_ECUDA; }
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return OCD_ECUDA;
    float *sink = nullptr;
    if (cudaMalloc((void **)&sink, sizeof(float)) != cudaSuccess) { cudaGetLastError(); return OCD_ENOMEM; }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = sms * 16, threads = 256;
    const int trips = (iters + 7) / 8;                              // `iters` keeps its meaning: rounds of 64 FMAs
    k_fp32_peak<<<blocks, threads, 0, st>>>(trips / 4 + 1, sink);   // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 3; ++rep) {
        cudaEventRecord(e0, st);
        k_fp32_peak<<<blocks, threads, 0, st>>>(trips, sink);
        cudaEventRecord(e1, st);
        if (cudaEventSynchronize(e1) != cudaSuccess) break;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double fl = 2.0 * kPeakFmaPerTrip * (double)trips * (double)blocks * threads / (ms * 1e-3);
        if (fl > best) best = fl;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    *flops = best;
    return cuda_status() == OCD_OK && best > 0.0 ? OCD_OK : OCD_ECUDA;
}

}  // extern "C"
