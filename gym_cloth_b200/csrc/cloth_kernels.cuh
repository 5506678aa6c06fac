// cloth_kernels.cuh - __global__ entry points and host launchers, templated on the scalar type.
// Included by cloth_f32.cu (production, FMA contraction on) and cloth_f64.cu (parity build, -fmad=false).
#pragma once
#include <atomic>
#include <cstdio>

#include "cloth_device.cuh"

namespace clothb200 {

extern std::atomic<long long> g_launch_count;   // defined in cloth_abi.cu
extern int g_debug_flags;
extern int g_force_slots, g_force_slice;         // tests: clothb200_debug_set_slicing
extern long long *g_prof_ptr;
// clothb200_step_kernel_info: when set, launch_step_inst reports the kernel it would launch instead of launching it
struct KernelInfo { int ctas_per_sm, registers, local_bytes, smem_bytes; };
extern thread_local KernelInfo *g_kernel_query;
// cloth_abi.cu: the calling thread's buffer for per-environment material rows on the current device (see there)
void *material_rows(size_t bytes, cudaStream_t st, int *rc);
int material_rows_release(cudaStream_t st);
#define CLOTHB200_MAX_DEVICES 64                    // debug: per-env phase counters (clothb200_debug_set_profile)
void set_cuda_error(cudaError_t e, const char *where);

// ------------------------------------------------------------------------------------------------
// The action kernel: one CTA = one cloth = one whole ClothEnv.step (or n bare updates).
// ------------------------------------------------------------------------------------------------
// f32, 128 threads: eight cloths per SM need <= 64 registers per thread (the shared-memory footprint allows exactly eight)
// (f64: four per SM by shared memory -> 128 registers)
template <typename T, int NT> struct MinBlocks { static constexpr int v = NT == 128 ? (sizeof(T) == 4 ? 8 : 4) : 1; };
// PHYS: every cloth takes its material constants from its own row A.mat[env] (per-environment physics) instead of P
template <typename T, int NT, int WC, bool REST_TABLE, bool COLOURED, bool PHYS>
__global__ void __launch_bounds__(NT, MinBlocks<T, NT>::v) cloth_step_kernel(const __grid_constant__ DevParams<T> P, const __grid_constant__ StepArgs<T> A) {
    typedef ClothCTA<T, NT, WC, REST_TABLE, COLOURED, PHYS> CTA;
    typedef typename CTA::P4 P4;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x;
    const bool sliced = A.slice > 0;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + CTA::smem_bytes(P.N, P.table_size, P.ev_words) - 16);
    int *s_item = reinterpret_cast<int *>(bar + 1);     // the 8 bytes behind the mbarrier: item, progress << 16 | grip count
    if (tid == 0) mbar_init(bar, 1);
    uint32_t bar_phase = 0;
  for (;;) {
    int item = (int)blockIdx.x, i_begin = 0, ngrab_in = -1;
    if (sliced) {
        __syncthreads();
        if (tid == 0) {
            const int it = queue_pop(A);
            s_item[0] = it;
            if (it >= 0) { s_item[1] = (A.progress[it] << 16) | (A.ngrab_s[it] & 0xffff); fence_async_all(); }
        }
        __syncthreads();
        item = s_item[0];
        if (item < 0) return;
        i_begin = s_item[1] >> 16; ngrab_in = s_item[1] & 0xffff;
    }
    const int env = A.env_order ? A.env_order[item] : item;
    const T *rest_env = REST_TABLE ? A.rest + (long long)env * A.rest_env_stride : nullptr;
    // (a resumed cloth of the time-sliced launch comes through here again: it takes its row again)
    const DevMaterial<T> *mat = PHYS ? A.mat + item : nullptr;
    CTA c(P, smem, rest_env, mat);
    c.prof_on = A.prof != nullptr;
    unsigned long long gt0 = 0;
    if (A.prof && threadIdx.x == 0) { asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt0)); }
    if (A.debug_flags & 1) c.rot = 0;
    const int N = c.N;
    const uint32_t bytes = (uint32_t)(sizeof(P4) * (size_t)N);
    T *gpos = A.pos + (size_t)env * N * 4, *gprev = A.prev + (size_t)env * N * 4;

    // ---- stage the cloth into shared memory: two TMA bulk copies completing on one mbarrier ----
    c.sync();
    if (tid == 0) {
        mbar_expect_tx(bar, 2 * bytes);
        bulk_g2s(c.pos, gpos, bytes, bar);
        bulk_g2s(c.prev, gprev, bytes, bar);
    }
    for (int j = tid; j < P.table_size; j += NT) { c.tkey[j] = CLOTH_KEY_EMPTY; c.tinfo[j] = 0u; }
    for (int j = tid; j < P.ev_words; j += NT) c.ev[j] = 0u;
    // misc[8..11]: a pinned point at the origin that nobody writes - the idle lanes of the f32 sweep read it
    if (tid < 16) { c.misc[tid] = (tid == 11 && sizeof(T) == 4) ? 0x3f800000 : 0; c.pacc[tid] = 0; }
    if (tid < 8) {
        const float r = (float)P.rest_k[tid < 6 ? tid : 0], ct = r * (float)c.tear_thresh();
        c.kc[tid] = make_float2(r * 1.1f, ct * ct);
    }
    int flags_in = A.flags ? A.flags[env] : 0;
    // a material row that derive_material() rejected: the cloth is not stepped (as a CLOTHB200_PLAN_BAD_ACTION plan)
    const bool bad_mat = PHYS ? __ldg(&mat->valid) == 0 : false;
    mbar_wait(bar, bar_phase);
    bar_phase ^= 1u;
    c.sync();
    if (tid == 0) c.misc[2] = (flags_in & CLOTHB200_FLAG_TEAR) ? 1 : 0;
    if (tid == 0 && (flags_in & CLOTHB200_FLAG_BADSTATE)) c.misc[3] = 1;
    c.sync();

    int nupd = 0, ngrab = -1;
    // one loop (one inlined copy of Cloth.update) serves both the action and the bare-update mode
    int iterations = 0, e0 = 0, e1 = 0, e2 = 0, e3 = 0;
    T dxr = T(0), dyr = T(0);
    const bool stepping = A.mode == KMODE_STEP;
    if (stepping) {
        const ClothB200Plan plan = A.plans[env];
        const bool bad_action = (plan.reserved & CLOTHB200_PLAN_BAD_ACTION) != 0 || bad_mat;   // NaN action: nothing is gripped, BADSTATE
        if (bad_action) { ngrab = 0; if (tid == 0) c.misc[3] = 1; }
        else if (i_begin > 0) ngrab = ngrab_in;       // resumed slice: the grip is part of the stored state
        else ngrab = c.grab_top(plan.gx, plan.gy, P.grip_radius);
        if (P.force_grab && i_begin == 0 && !bad_action) {
            // cloth_env.py:434-444: `while len(grabbed_pts) == 0: grip_radius += 0.02; grab_top(...)` (radius restored afterwards).
            // A cloth with no point under z = height + 2*thickness can never be gripped; the reference would spin forever,
            // we stop once the cylinder covers any reachable (x, y) and report NOGRAB.
            double rad = P.grip_radius;
            for (int tries = 0; ngrab == 0 && tries < 4096; tries++) { rad += 0.02; ngrab = c.grab_top(plan.gx, plan.gy, rad); }
        }
        if (A.grab_mask && i_begin == 0) { c.write_grab_mask(A.grab_mask + (size_t)env * ((N + 31) >> 5)); c.sync(); }
        // _pull thresholds (cloth_env.py:352-367, 472-475): `i < t` for integer i <=> i < ceil(t)
        const double iu = A.iters_up_env ? A.iters_up_env[env] : P.iu;
        const double t1 = iu + P.iur, t2 = t1 + (double)plan.iters_pull, t3 = t2 + P.igr, t4 = t3 + P.ir;
        e0 = (int)ceil(iu); e1 = (int)ceil(t1); e2 = (int)ceil(t2); e3 = (int)ceil(t3);
        iterations = ngrab == 0 ? 0 : (int)ceil(t4);   // cloth_env.py:490-493
        dxr = (T)plan.dxr; dyr = (T)plan.dyr;
    } else if (A.mode == KMODE_UPDATE) {
        iterations = bad_mat ? 0 : A.n_updates;
        if (bad_mat && tid == 0) c.misc[3] = 1;
    } else if (A.mode == KMODE_GRAB) {
        ngrab = c.grab_top(A.grab_xy[2 * env], A.grab_xy[2 * env + 1], A.grab_radius);
        if (A.grab_mask) c.write_grab_mask(A.grab_mask + (size_t)env * ((N + 31) >> 5));
    }
    bool released = stepping && i_begin > e3;
    // slices and the swap hysteresis shrink to a quarter for the last six slices of an action: the launch ends when its last
    // cloth does, and near the end the grain of the hand-over is what the slots differ by
    const int endgame = A.endgame_slices * A.slice;
    auto slice_len = [&](int left) { return left <= endgame ? max(A.slice >> A.endgame_shift, 1) : A.slice; };
    int i_end = sliced ? min(iterations, i_begin + slice_len(iterations - i_begin)) : iterations;
    const long long t_loop0 = clock64();
    int i = i_begin;
    bool broke = false, parked = false;
    for (;;) {
        for (; i < i_end; i++) {
            if (stepping) {
                if (i < e0) { c.gripper_adjust(T(0.0), T(0.0), T(0.0025)); c.sync(); }
                else if (i < e1) { }
                else if (i < e2) { c.gripper_adjust(dxr, dyr, T(0.0)); c.sync(); }
                else if (i < e3) { }
                else if (!released) { c.gripper_release(); released = true; c.sync(); }
            }
            c.update();
            if (stepping && c.misc[2]) { broke = true; i++; break; }   // tear: cloth_env.py:511-514 (gripper is not released)
        }
        if (!sliced || broke || i >= iterations) break;
        // ---- end of a slice: longest-remaining-first.  Keep the cloth unless a waiting one has more substeps left
        // (then the launch ends at max(longest action, total work / slots) instead of with the last whole action) ----
        // (ordering by measured time left instead - substeps left x this action's cycles per substep - was tried and is
        // worse: the FIFO of waiting cloths stays sorted by substeps left, not by such estimates, and long cloths starve)
        if (tid == 0) {
            const int left = iterations - i, slack = left <= endgame ? A.yield_slack >> A.endgame_shift : A.yield_slack;
            s_item[0] = left; s_item[1] = queue_head_remaining(A) > left + slack ? 1 : 0;
        }
        c.sync();
        const bool yield = s_item[1] != 0;
        const int left_units = s_item[0];
        c.sync();
        if (!yield) { i_end = min(iterations, i + slice_len(left_units)); continue; }
        const int bad_now = c.misc[3];
        fence_async_smem();
        c.sync();
        if (tid == 0) {
            bulk_s2g(gpos, c.pos, bytes);
            bulk_s2g(gprev, c.prev, bytes);
            A.progress[item] = i; A.ngrab_s[item] = ngrab;
            A.cycles_s[item] = (float)(clock64() - t_loop0) + (i_begin > 0 ? A.cycles_s[item] : 0.f);
            if (bad_now && A.flags) A.flags[env] = flags_in | CLOTHB200_FLAG_BADSTATE;
            if (A.prof) for (int k = 0; k < 16; k++) if (k != 10) A.prof[(size_t)env * 16 + k] += c.pacc[k];
            bulk_commit_wait_all();
            fence_async_all();
            queue_push(A, item, left_units);
        }
        parked = true;
        break;
    }
    if (parked) continue;
    nupd = i;
    const long long t_loop1 = clock64();
    float cycles_total = (float)(t_loop1 - t_loop0);
    if (sliced && i_begin > 0) cycles_total += A.cycles_s[item];

    // ---- reward terms ----
    const bool want_measure = (A.coverage || A.variance_inv || A.reward) && A.mode != KMODE_GRAB;
    double cov = 0.0, vinv = 0.0;
    const bool oob = c.out_of_bounds();
    if (want_measure) {
        vinv = c.variance_inv();
        cov = c.hull_area();
    }
    const int tear = c.misc[2], bad = c.misc[3];
    c.sync();

    // ---- write back: state via TMA bulk store, scalars by thread 0 ----
    if (A.mode != KMODE_MEASURE) {
        fence_async_smem();
        c.sync();
        if (tid == 0) {
            bulk_s2g(gpos, c.pos, bytes);
            bulk_s2g(gprev, c.prev, bytes);
            bulk_commit_wait();
        }
    }
    if (A.obs) {
        const T *flat = reinterpret_cast<const T *>(c.pos);
        T *o = A.obs + (size_t)env * 3 * N;
        for (int i = tid; i < 3 * N; i += NT) { const int p = i / 3; o[i] = flat[p * 4 + (i - p * 3)]; }
    }
    if (tid == 0 && A.cost && stepping && nupd > 0) A.cost[env] = cycles_total / (float)nupd;
    if (tid == 0) {
        int f = (tear ? CLOTHB200_FLAG_TEAR : 0) | (oob ? CLOTHB200_FLAG_OOB : 0) | (bad ? CLOTHB200_FLAG_BADSTATE : 0);
        if (A.mode == KMODE_STEP && ngrab == 0) f |= CLOTHB200_FLAG_NOGRAB;
        if (A.flags) A.flags[env] = f;
        if (A.sim_steps) A.sim_steps[env] = nupd;
        if (A.n_grabbed && ngrab >= 0) A.n_grabbed[env] = ngrab;
        if (want_measure) {
            if (A.coverage) A.coverage[env] = cov;
            if (A.variance_inv) A.variance_inv[env] = vinv;
        }
        if (A.mode == KMODE_STEP && A.reward && !A.initialize) {
            // ClothEnv.step bookkeeping + _reward + _terminal (cloth_env.py:519-521, 536-715), reward_type coverage-delta
            const int steps = A.num_steps[env] + 1;
            A.num_steps[env] = steps;
            A.num_sim_steps[env] += nupd;
            double rew = 0;
            if (tear) rew += 0.0; else if (oob) rew += 0.0;
            if (ngrab == 0) rew += -0.01;
            if (cov > 0.92) rew += 5.;
            rew += 0.0;
            if (P.reward_abs) rew += cov;                         // 'coverage' (cloth_env.py:657-659): _prev_reward is left alone
            else {                                                // 'coverage-delta' (cloth_env.py:660-662, compute_delta :640-643)
                const double prevc = A.prev_coverage[env];
                rew += cov - prevc;
                A.prev_coverage[env] = cov;
            }
            A.reward[env] = rew;
            A.done[env] = (steps >= P.max_actions) || tear || oob || (cov > 0.92);
        }
    }
    if (A.prof && tid == 0) {
        unsigned long long gt1; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt1));
        unsigned smid; asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
        if (A.debug_flags & 2) { c.pacc[14] = (long long)gt0; c.pacc[15] = (long long)gt1; c.pacc[11] = (long long)smid * 1000000 + c.pacc[11] % 1000000; }
        if (sliced) {
            for (int k = 0; k < 16; k++) if (k != 10) A.prof[(size_t)env * 16 + k] += c.pacc[k];
            A.prof[(size_t)env * 16 + 10] = nupd;
        } else {
            c.pacc[10] = nupd;
            for (int k = 0; k < 16; k++) A.prof[(size_t)env * 16 + k] = c.pacc[k];
        }
    }
    if (!sliced) return;
    if (tid == 0) { __threadfence(); atomicAdd(&A.qctl[2], 1); }
  }
}

// queue of the time-sliced mode: every item once, in launch order, with the substeps its plan will run
static __global__ void queue_init_kernel(int n, const unsigned long long *keys, unsigned long long *queue, int *qctl, int *progress,
                                         int *ngrab_s, float *cycles_s) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) {
        const float work = __uint_as_float(~(unsigned)(keys[j] >> 32));      // plan_work_kernel's key, after the sort: planned substeps
        const unsigned rem = (unsigned)fminf(fmaxf(work, 0.f), 65535.f);
        queue[j] = ((unsigned long long)(unsigned)(j + 1) << 32) | (rem << 16) | (unsigned)j;
        progress[j] = 0; ngrab_s[j] = -1; cycles_s[j] = 0.f;
    }
    if (j == 0) { qctl[0] = 0; qctl[1] = n; qctl[2] = 0; qctl[3] = 0; }
}

// ------------------------------------------------------------------------------------------------
// longest-first scheduling: work estimate per environment, then a single-CTA bitonic sort of (work, env)
// ------------------------------------------------------------------------------------------------
// One warp per environment.  work = number of substeps the plan will run (0 if the grip catches nothing).
// This only orders the launch: it is a heuristic (the z-band test is simplified), results never depend on it.
template <typename T>
__global__ void plan_work_kernel(int n_env, int n_pow2, int N, const T *__restrict__ pos, const T *__restrict__ prev,
                                 const ClothB200Plan *__restrict__ plans, const float *__restrict__ cost, double grip_radius,
                                 double thickness, double height, double iu, double iur, double igr, double ir,
                                 const double *__restrict__ iters_up_env, unsigned long long *__restrict__ keys) {
    const int env = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (env >= n_pow2) return;
    if (env >= n_env) { if (lane == 0) keys[env] = ~0ull; return; }   // padding sorts last
    const ClothB200Plan pl = plans[env];
    const T *pp = pos + (size_t)env * N * 4, *qq = prev + (size_t)env * N * 4;
    bool any = false;
    for (int p = lane; p < N; p += 32) {
        const double x = (double)pp[4 * p], y = (double)pp[4 * p + 1], z = (double)pp[4 * p + 2];
        const bool in_r = (x - pl.gx) * (x - pl.gx) + (y - pl.gy) * (y - pl.gy) < grip_radius;
        any |= (in_r && z > -2 * thickness && z < height + 2 * thickness) || (qq[4 * p + 3] > T(0));
    }
    any = __any_sync(0xffffffffu, any);
    if (lane == 0) {
        const double i0 = iters_up_env ? iters_up_env[env] : iu;
        const float iters = any ? (float)(i0 + iur + (double)pl.iters_pull + igr + ir) : 0.f;
        // Measured (scripts/quick_bench.py sched, scripts/cost_model.py): an environment's cycles per substep in its
        // last step says almost nothing about the coming one (correlation 0.08-0.25) and ordering by it is no better
        // than not ordering, while the planned substep count alone orders as well as the exact cost would.
        (void)cost;
        const float work = iters;
        // descending by work: invert the (non-negative) float bits; ties by env id
        keys[env] = ((unsigned long long)(~__float_as_uint(work)) << 32) | (unsigned)env;
    }
}

// bitonic sort of n_pow2 64-bit keys by one CTA (n_pow2 <= 65536), then env_order[i] = low word
static __global__ void __launch_bounds__(1024) sort_keys_kernel(int n_env, int n_pow2, unsigned long long *__restrict__ keys,
                                                         int32_t *__restrict__ env_order) {
    for (int k = 2; k <= n_pow2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
                const int l = i ^ j;
                if (l > i) {
                    const unsigned long long a = keys[i], b = keys[l];
                    const bool up = (i & k) == 0;
                    if (up ? (a > b) : (a < b)) { keys[i] = b; keys[l] = a; }
                }
            }
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < n_env; i += blockDim.x) env_order[i] = (int32_t)(keys[i] & 0xffffffffull);
}

// ------------------------------------------------------------------------------------------------
// small utility kernels
// ------------------------------------------------------------------------------------------------
// ClothEnv.step action decode (cloth_env.py:401-470) with x*x for `**2`
template <typename T>
__global__ void decode_actions_kernel(int n, const T *__restrict__ actions, ClothB200Plan *__restrict__ plans, int clip_act_space,
                                      int delta_actions, double reduce_factor, int iters_pull_max) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    double lo[4], hi[4];
    const double pi_f32 = 3.1415927410125732;
    if (clip_act_space) { for (int i = 0; i < 4; i++) { lo[i] = -1.0; hi[i] = 1.0; } }
    else if (delta_actions) { lo[0] = 0; lo[1] = 0; lo[2] = -1; lo[3] = -1; hi[0] = hi[1] = hi[2] = hi[3] = 1; }
    else { lo[0] = -0.25; lo[1] = -0.25; lo[2] = 0.0; lo[3] = -pi_f32; hi[0] = 1.25; hi[1] = 1.25; hi[2] = 1.0; hi[3] = pi_f32; }
    double a[4];
    bool nan_action = false;
    for (int i = 0; i < 4; i++) {
        double v = (double)actions[4 * e + i];
        if (v != v) { nan_action = true; v = 0.0; }   // see clothb200_decode_actions_host
        double m = (hi[i] < v) ? hi[i] : v;
        a[i] = (lo[i] > m) ? lo[i] : m;
    }
    double x = a[0], y = a[1], length = a[2], radians = a[3];
    if (clip_act_space) {
        x = (x / 2.0) + 0.5; y = (y / 2.0) + 0.5;
        if (!delta_actions) { length = (length / 2.0) + 0.5; radians = radians * 3.141592653589793; }
    }
    double xd, yd, total = 0.0;
    if (delta_actions) {
        total = sqrt(a[2] * a[2] + a[3] * a[3]);
        xd = a[2] / (total + 1e-5); yd = a[3] / (total + 1e-5);
    } else { xd = cos(radians); yd = sin(radians); }
    const double xr = xd * reduce_factor, yr = yd * reduce_factor;
    int ip;
    if (delta_actions) {
        const double stepl = sqrt(xr * xr + yr * yr);
        int ii = 0;
        if (stepl > 0.0) { double cur = 0; for (;;) { cur += stepl; if (cur >= total || ii >= CLOTHB200_MAX_ITERS_PULL) break; ii += 1; } }
        ip = ii;
    } else ip = (int)(iters_pull_max * length);
    ClothB200Plan pl; pl.gx = x; pl.gy = y; pl.dxr = xr; pl.dyr = yr; pl.iters_pull = ip; pl.reserved = 0;
    if (nan_action) { pl.gx = 0.5; pl.gy = 0.5; pl.dxr = 0.0; pl.dyr = 0.0; pl.iters_pull = 0; pl.reserved = CLOTHB200_PLAN_BAD_ACTION; }
    plans[e] = pl;
}

template <typename T>
__global__ void broadcast_state_kernel(int n4, int n_env, const T *__restrict__ pos4, const T *__restrict__ prev4, T *__restrict__ pos,
                                       T *__restrict__ prev) {
    const size_t total = (size_t)n4 * n_env;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int j = (int)(i % n4);
        pos[i] = pos4[j];
        prev[i] = prev4[j];
    }
}

// Gripper.adjust / release over a batch (facade-level calls; the step kernel has its own in-smem versions)
template <typename T>
__global__ void gripper_adjust_kernel(size_t total_pts, T dx, T dy, T dz, T *__restrict__ pos, T *__restrict__ prev) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= total_pts) return;
    T *p = pos + 4 * i, *q = prev + 4 * i;
    const int m = (int)q[3];
    for (int r = 0; r < m; r++) {
        q[0] = p[0]; q[1] = p[1]; q[2] = p[2];
        p[0] = dx + p[0]; p[1] = dy + p[1]; p[2] = dz + p[2];
    }
}
template <typename T> __global__ void gripper_release_kernel(size_t total_pts, T *__restrict__ pos, T *__restrict__ prev) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= total_pts) return;
    if (prev[4 * i + 3] > T(0)) { pos[4 * i + 3] = T(0); prev[4 * i + 3] = T(0); }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
const uint32_t *get_sweep_table(int W, int *levels, int *lw);   // cloth_abi.cu (cached per device and grid width)
int sweep_threshold();

template <typename T> int make_dev_params(const ClothB200Params &hp, DevParams<T> &P) {
    const int W = hp.num_width_points, H = hp.num_height_points;
    P.W = W; P.H = H; P.N = W * H;
    // hash table slots: 3x the cells a flat cloth occupies (cell = 3 grid spacings; oracle runs never exceeded 1.15x)
    const int cells = (W + 2) / 3 + 1;
    int ts = 64; while (ts < 3 * cells * cells) ts <<= 1;
    { int np2 = 1; while (np2 < P.N) np2 <<= 1; while (4 * ts < np2) ts <<= 1; }   // the coverage sort borrows the table area
    P.table_size = ts;
    int sh = 0; while ((1 << sh) < ts) sh++;
    P.table_shift = 32 - sh;
    P.ev_words = (6 * P.N + 31) / 32;
    P.max_actions = hp.max_actions;
    const double dx = hp.width * 1.0 / (W - 1), dy = hp.height * 1.0 / (H - 1);
    const double cw = 3 * dx, ch = 3 * dy;
    P.cell_w = (T)cw; P.cell_h = (T)ch; P.cell_t = (T)(cw > ch ? cw : ch);
    P.thresh = (T)(2.0 * hp.thickness);
    P.thresh2 = P.thresh * P.thresh;
    P.inv_cell_w = (T)(1.0 / cw); P.inv_cell_h = (T)(1.0 / ch); P.inv_cell_t = (T)(1.0 / (cw > ch ? cw : ch));
    {
        int e1, e2;
        const bool p2w = frexp(cw, &e1) == 0.5, p2h = frexp(ch, &e2) == 0.5;
        P.cell_pow2 = (p2w && p2h) ? 1 : 0;
    }
    P.sim_steps = (T)hp.simulation_steps;
    P.min_z = (T)hp.minimum_z;
    P.surf_off = (T)0.0001;
    const double diag = sqrt(dx * dx + dy * dy);
    const double rk[6] = {dx, dy, diag, diag, 2 * dx, 2 * dy};
    for (int k = 0; k < 6; k++) P.rest_k[k] = (T)rk[k];
    // the material constants (mass*gravity, ks terms, damping, friction, tear threshold)
    DevMaterial<T> m;
    derive_material<T>(hp.density, hp.ks, hp.damping, hp.plane_friction, hp.tear_thresh, hp.gravity, W, H, hp.frames_per_sec,
                       hp.simulation_steps, P.rest_k, m);
    P.mg = m.mg; P.kk_struct = m.kk_struct; P.kk_bend = m.kk_bend; P.dsdm = m.dsdm; P.damp = m.damp;
    P.fric1 = m.fric1; P.tear_thresh = m.tear_thresh;
    for (int k = 0; k < 6; k++) { P.kkrest_k[k] = m.kkrest_k[k]; P.limit_c2_k[k] = m.limit_c2_k[k]; }
    P.grip_radius = hp.grip_radius; P.thickness = hp.thickness; P.gripper_height = hp.gripper_height;
    int nlev = 0;
    for (double z = hp.gripper_height; z > 0; z -= hp.thickness) { nlev++; if (nlev > 8 * ts / 8) break; }
    P.n_levels = nlev;
    P.iu = hp.iters_up; P.iur = hp.iters_up_rest; P.igr = hp.iters_grip_rest; P.ir = hp.iters_rest;
    P.sweep_tbl = get_sweep_table(W, &P.sweep_levels, &P.sweep_lw);
    P.sweep_thresh = sweep_threshold();
    P.relax_iters = hp.reserved0 > 1 ? hp.reserved0 : 1;
    P.force_grab = hp.force_grab ? 1 : 0;
    P.reward_abs = hp.reward_type == CLOTHB200_REWARD_COVERAGE ? 1 : 0;
    return 0;
}

template <typename T, int NT, int WC, bool RT, bool COL, bool PHYS> int launch_step_inst(const DevParams<T> &P, const StepArgs<T> &A, cudaStream_t st) {
    typedef ClothCTA<T, NT, WC, RT, COL, PHYS> CTA;
    const size_t smem = CTA::smem_bytes(P.N, P.table_size, P.ev_words);
    auto kern = cloth_step_kernel<T, NT, WC, RT, COL, PHYS>;
    // cudaFuncSetAttribute and occupancy are per device: one process may drive several GPUs (SURVEY.md 8(e) allows one
    // process with a stream per device), so both caches are keyed by the current device
    static std::atomic<size_t> configured[CLOTHB200_MAX_DEVICES];
    static std::atomic<int> slots_of[CLOTHB200_MAX_DEVICES];
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= CLOTHB200_MAX_DEVICES) return CLOTHB200_ERR_UNSUPPORTED;
    if (smem > configured[dev].load()) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            // too large for one CTA: refused before anything runs.  The runtime also keeps the error as this thread's
            // last error, where the next launch check (ours or the caller's) would find it: clear it
            set_cuda_error(e, "cudaFuncSetAttribute(smem)");
            cudaGetLastError();
            return CLOTHB200_ERR_UNSUPPORTED;
        }
        configured[dev].store(smem);
    }
    if (g_kernel_query) {
        cudaFuncAttributes fa;
        int occ = 0;
        if (cudaFuncGetAttributes(&fa, kern) != cudaSuccess || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem) != cudaSuccess) {
            set_cuda_error(cudaGetLastError(), "step kernel attributes");
            return CLOTHB200_ERR_CUDA;
        }
        *g_kernel_query = KernelInfo{occ, fa.numRegs, (int)fa.localSizeBytes, (int)smem};
        return CLOTHB200_OK;
    }
    if (A.slice > 0) {
        // time-sliced mode: a persistent grid, one CTA per resident slot; pointless when every cloth has its own slot
        int slots = slots_of[dev].load();
        if (!slots) {
            int occ = 0, sms = 0;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem) != cudaSuccess || occ < 1) occ = 1;
            slots = occ * sms;
            slots_of[dev].store(slots);
        }
        const int use_slots = g_force_slots > 0 ? g_force_slots : slots;
        if (A.n_env > use_slots) {
            queue_init_kernel<<<(A.n_env + 255) / 256, 256, 0, st>>>(A.n_env, A.sorted_keys, A.queue, A.qctl, A.progress, A.ngrab_s, A.cycles_s);
            StepArgs<T> B = A;
            if (g_force_slice > 0) { B.slice = g_force_slice; B.yield_slack = 0; B.endgame_slices = 0; }
            kern<<<use_slots, NT, smem, st>>>(P, B);
            g_launch_count += 2;
            cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) { set_cuda_error(e, "cloth_step_kernel (sliced) launch"); return CLOTHB200_ERR_CUDA; }
            return CLOTHB200_OK;
        }
    }
    StepArgs<T> B = A;
    B.slice = 0;
    kern<<<A.n_env, NT, smem, st>>>(P, B);
    g_launch_count++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_cuda_error(e, "cloth_step_kernel launch"); return CLOTHB200_ERR_CUDA; }
    return CLOTHB200_OK;
}

int slice_substeps();           // cloth_abi.cu: CLOTHB200_SLICE env var; default 64, 0 = whole actions
int yield_slack_substeps();     // cloth_abi.cu: CLOTHB200_YIELD_SLACK env var (substeps)
int endgame_slices();           // cloth_abi.cu: CLOTHB200_ENDGAME env var (slices), CLOTHB200_ENDGAME_SHIFT
int endgame_shift();
int threads_per_cloth(int W);   // cloth_abi.cu: CLOTHB200_NT env var; default 128 (512 for 64x64)

template <typename T, int WC, bool RT, bool COL, bool PHYS> int launch_step_nt(const DevParams<T> &P, const StepArgs<T> &A, cudaStream_t st) {
    const int nt = threads_per_cloth(P.W);
    if (WC == 64) {   // one resident cloth per SM: wide CTAs
        if (nt == 256) return launch_step_inst<T, 256, WC, RT, COL, PHYS>(P, A, st);
        return launch_step_inst<T, 512, WC, RT, COL, PHYS>(P, A, st);
    }
    if (nt == 256) return launch_step_inst<T, 256, WC, RT, COL, PHYS>(P, A, st);
    return launch_step_inst<T, 128, WC, RT, COL, PHYS>(P, A, st);
}

// One (scalar type, compile-time grid width, per-environment material or not) triple per translation unit
// (cloth_inst.cu, built twelve times in parallel): the kernel is one large force-inlined function and a single TU
// holding every variant compiles for a quarter of an hour.
template <typename T, int WC, bool PHYS> int launch_step_wc(const DevParams<T> &P, const StepArgs<T> &A, cudaStream_t st, bool rt, bool coloured) {
    if (coloured) {
        if constexpr (WC != 0) return rt ? launch_step_nt<T, WC, true, true, PHYS>(P, A, st) : launch_step_nt<T, WC, false, true, PHYS>(P, A, st);
        else return CLOTHB200_ERR_UNSUPPORTED;   // coloured mode is built for the 25x25 and 64x64 grids
    }
    return rt ? launch_step_nt<T, WC, true, false, PHYS>(P, A, st) : launch_step_nt<T, WC, false, false, PHYS>(P, A, st);
}
#ifdef CLOTH_INSTANTIATE_WC
#ifndef CLOTH_INSTANTIATE_PHYS
#define CLOTH_INSTANTIATE_PHYS 0
#endif
template int launch_step_wc<CLOTH_T, CLOTH_INSTANTIATE_WC, CLOTH_INSTANTIATE_PHYS != 0>(const DevParams<CLOTH_T> &, const StepArgs<CLOTH_T> &, cudaStream_t, bool, bool);
#else
#define CLOTH_EXTERN_WC(T, WC, PH) extern template int launch_step_wc<T, WC, PH>(const DevParams<T> &, const StepArgs<T> &, cudaStream_t, bool, bool);
CLOTH_EXTERN_WC(float, 0, false) CLOTH_EXTERN_WC(float, 25, false) CLOTH_EXTERN_WC(float, 64, false)
CLOTH_EXTERN_WC(double, 0, false) CLOTH_EXTERN_WC(double, 25, false) CLOTH_EXTERN_WC(double, 64, false)
CLOTH_EXTERN_WC(float, 0, true) CLOTH_EXTERN_WC(float, 25, true) CLOTH_EXTERN_WC(float, 64, true)
CLOTH_EXTERN_WC(double, 0, true) CLOTH_EXTERN_WC(double, 25, true) CLOTH_EXTERN_WC(double, 64, true)
#undef CLOTH_EXTERN_WC
#endif

// per-environment material rows, by launch position i (the step kernel's `item`): row i holds the constants of
// environment env_order[i] (or i), derived by the same derive_material() make_dev_params calls
template <typename T>
__global__ void derive_material_kernel(int n, const ClothB200Physics *__restrict__ phys, const int32_t *__restrict__ env_order,
                                       const __grid_constant__ DevParams<T> P, double frames_per_sec, int simulation_steps,
                                       DevMaterial<T> *__restrict__ mat) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ClothB200Physics ph = phys[env_order ? env_order[i] : i];
    DevMaterial<T> m;
    derive_material<T>(ph.density, ph.ks, ph.damping, ph.plane_friction, ph.tear_thresh, ph.gravity, P.W, P.H, frames_per_sec,
                       simulation_steps, P.rest_k, m);
    mat[i] = m;
}

template <typename T>
int launch_step(const ClothB200Params &hp, const StepArgs<T> &A, cudaStream_t st, int rmode = 0, const ClothB200Physics *phys = nullptr) {
    if (A.n_env == 0) return CLOTHB200_OK;
    DevParams<T> P;
    make_dev_params(hp, P);
    if (P.N >= 32768) return CLOTHB200_ERR_UNSUPPORTED;   // 15-bit slots / 16-bit indices
    const bool rt = A.rest != nullptr;
    if (!rt && sizeof(T) == 8 && rmode == 0) return CLOTHB200_ERR_ARG;  // the parity build always takes the exact rest table
    const bool coloured = rmode == CLOTHB200_MODE_COLOURED;
    if (phys) {
        StepArgs<T> B = A;
        int rc = CLOTHB200_OK;
        if (!g_kernel_query) {
            // the rows go to the calling thread's cached buffer (no allocation per call); it is released to the next call
            // behind this call's step kernel
            DevMaterial<T> *mat = (DevMaterial<T> *)material_rows(sizeof(DevMaterial<T>) * (size_t)A.n_env, st, &rc);
            if (rc) return rc;
            derive_material_kernel<T><<<(A.n_env + 127) / 128, 128, 0, st>>>(A.n_env, phys, A.env_order, P, (double)hp.frames_per_sec,
                                                                             hp.simulation_steps, mat);
            g_launch_count++;
            const cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) { set_cuda_error(e, "derive_material_kernel"); rc = CLOTHB200_ERR_CUDA; }
            B.mat = mat;
        }
        if (rc == CLOTHB200_OK) {
            if (P.W == 25 && P.H == 25) rc = launch_step_wc<T, 25, true>(P, B, st, rt, coloured);
            else if (P.W == 64 && P.H == 64) rc = launch_step_wc<T, 64, true>(P, B, st, rt, coloured);
            else rc = launch_step_wc<T, 0, true>(P, B, st, rt, coloured);
        }
        if (!g_kernel_query) {
            const int rc2 = material_rows_release(st);
            if (rc == CLOTHB200_OK) rc = rc2;
        }
        return rc;
    }
    if (P.W == 25 && P.H == 25) return launch_step_wc<T, 25, false>(P, A, st, rt, coloured);
    if (P.W == 64 && P.H == 64) return launch_step_wc<T, 64, false>(P, A, st, rt, coloured);
    return launch_step_wc<T, 0, false>(P, A, st, rt, coloured);
}

template <typename T> size_t step_smem_bytes(const ClothB200Params &hp) {
    DevParams<T> P;
    make_dev_params(hp, P);
    // what the reference-order step kernel launched for this grid takes (the ordered scatter needs no counter block)
    if (P.W == 25 && threads_per_cloth(25) == 128) return ClothCTA<T, 128, 25, true, false>::smem_bytes(P.N, P.table_size, P.ev_words);
    return ClothCTA<T, 128, 0, true, false>::smem_bytes(P.N, P.table_size, P.ev_words);
}

}  // namespace clothb200
