// cloth_typed.cuh - typed C++ entry points shared by cloth_f32.cu / cloth_f64.cu and used by cloth_abi.cu.
// CLOTH_T and CLOTH_SUFFIX select the scalar type of the including translation unit.
#pragma once
#include "cloth_kernels.cuh"

namespace clothb200 {

template <typename T> StepArgs<T> make_args(int n_env, const ClothB200Step *io) {
    StepArgs<T> A;
    memset(&A, 0, sizeof(A));
    A.n_env = n_env;
    if (io) {
        A.pos = (T *)io->pos; A.prev = (T *)io->prev;
        A.rest = (const T *)io->rest; A.rest_env_stride = io->rest_env_stride;
        A.flags = io->flags; A.sim_steps = io->sim_steps; A.n_grabbed = io->n_grabbed; A.grab_mask = io->grab_mask;
        A.coverage = io->coverage; A.variance_inv = io->variance_inv; A.obs = (T *)io->obs;
        if (io->prev_coverage && io->num_steps && io->num_sim_steps && io->reward && io->done) {
            A.prev_coverage = io->prev_coverage; A.num_steps = io->num_steps; A.num_sim_steps = io->num_sim_steps;
            A.reward = io->reward; A.done = io->done;
        }
        A.iters_up_env = io->iters_up_env; A.env_order = io->env_order;
        A.cost = io->cost;
    }
    A.prof = g_prof_ptr;
    A.debug_flags = g_debug_flags;
    return A;
}

template <typename T> int check_io(int n_env, const ClothB200Step *io) {
    if (n_env < 0 || !io) return CLOTHB200_ERR_ARG;
    if (n_env == 0) return CLOTHB200_OK;
    if (!io->pos || !io->prev) return CLOTHB200_ERR_ARG;
    if (((uintptr_t)io->pos & 15) || ((uintptr_t)io->prev & 15)) return CLOTHB200_ERR_ARG;   // TMA bulk copies
    return CLOTHB200_OK;
}

template <typename T>
int step_plans_t(const ClothB200Params *hp, int mode, int n_env, const ClothB200Plan *plans, const ClothB200Step *io, int initialize,
                 const ClothB200Physics *phys, cudaStream_t st) {
    int rc = check_io<T>(n_env, io);
    if (rc || n_env == 0) return rc;
    if (!hp || !plans) return CLOTHB200_ERR_ARG;
    if (mode != CLOTHB200_MODE_REFERENCE_ORDER && mode != CLOTHB200_MODE_COLOURED) return CLOTHB200_ERR_UNSUPPORTED;
    StepArgs<T> A = make_args<T>(n_env, io);
    A.plans = plans; A.mode = KMODE_STEP; A.initialize = initialize;
    if (!io->env_order && io->sched_scratch && n_env > 1 && n_env <= 65536) {
        // longest-first schedule (heuristic ordering only; results do not depend on it)
        int n_pow2 = 1; while (n_pow2 < n_env) n_pow2 <<= 1;
        unsigned long long *keys = (unsigned long long *)io->sched_scratch;
        int32_t *order = (int32_t *)(keys + n_pow2);
        const int N = hp->num_width_points * hp->num_height_points;
        const int warps_per_block = 8;
        plan_work_kernel<T><<<(n_pow2 + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, st>>>(
            n_env, n_pow2, N, (const T *)io->pos, (const T *)io->prev, plans, io->cost, hp->grip_radius, hp->thickness,
            hp->gripper_height, hp->iters_up, hp->iters_up_rest, hp->iters_grip_rest, hp->iters_rest, io->iters_up_env, keys);
        sort_keys_kernel<<<1, 1024, 0, st>>>(n_env, n_pow2, keys, order);
        g_launch_count += 2;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { set_cuda_error(e, "schedule kernels"); return CLOTHB200_ERR_CUDA; }
        A.env_order = order;
        // time slicing (see StepArgs): needs the larger scratch; a debug timeline wants one CTA per cloth
        const size_t need = clothb200_sched_scratch_bytes(n_env);
        const int slice = slice_substeps();
        if (slice > 0 && io->sched_scratch_bytes >= (int64_t)need && !(g_debug_flags & 2)) {
            unsigned char *base = (unsigned char *)io->sched_scratch + (size_t)8 * n_pow2 + (size_t)8 * ((n_env + 1) / 2);
            A.queue = (unsigned long long *)base;
            A.progress = (int *)(base + (size_t)8 * n_env);
            A.ngrab_s = A.progress + n_env;
            A.cycles_s = (float *)(A.ngrab_s + n_env);
            A.qctl = (int *)(A.cycles_s + n_env);
            A.slice = slice; A.yield_slack = yield_slack_substeps(); A.endgame_slices = endgame_slices(); A.endgame_shift = endgame_shift(); A.qcap = n_env; A.sorted_keys = keys;
        }
    }
    return launch_step<T>(*hp, A, st, mode, phys);
}

template <typename T>
int update_n_t(const ClothB200Params *hp, int mode, int n_env, int n_updates, const ClothB200Step *io, const ClothB200Physics *phys,
               cudaStream_t st) {
    int rc = check_io<T>(n_env, io);
    if (rc || n_env == 0) return rc;
    if (!hp || n_updates < 0) return CLOTHB200_ERR_ARG;
    if (mode != CLOTHB200_MODE_REFERENCE_ORDER && mode != CLOTHB200_MODE_COLOURED) return CLOTHB200_ERR_UNSUPPORTED;
    StepArgs<T> A = make_args<T>(n_env, io);
    A.mode = KMODE_UPDATE; A.n_updates = n_updates;
    return launch_step<T>(*hp, A, st, mode, phys);
}

template <typename T>
int grab_top_t(const ClothB200Params *hp, int n_env, const double *xy, double radius, const ClothB200Step *io, cudaStream_t st) {
    int rc = check_io<T>(n_env, io);
    if (rc || n_env == 0) return rc;
    if (!hp || !xy) return CLOTHB200_ERR_ARG;
    StepArgs<T> A = make_args<T>(n_env, io);
    A.mode = KMODE_GRAB; A.grab_xy = xy; A.grab_radius = radius;
    return launch_step<T>(*hp, A, st);
}

// the step kernel that step_plans would launch for this configuration, queried instead of launched
template <typename T> int kernel_info_t(const ClothB200Params *hp, int mode, int rest_table, int per_env_physics, int *out) {
    StepArgs<T> A = make_args<T>(1, nullptr);
    A.mode = KMODE_STEP;
    static const T dummy_rest[1] = {T(0)};
    A.rest = rest_table ? dummy_rest : nullptr;              // only tested for NULL: nothing is read
    static const ClothB200Physics dummy_phys = {};
    KernelInfo info = {0, 0, 0, 0};
    g_kernel_query = &info;
    const int rc = launch_step<T>(*hp, A, 0, mode, per_env_physics ? &dummy_phys : nullptr);
    g_kernel_query = nullptr;
    out[0] = info.ctas_per_sm; out[1] = info.registers; out[2] = info.local_bytes; out[3] = info.smem_bytes;
    return rc;
}

template <typename T> int measure_t(const ClothB200Params *hp, int n_env, const ClothB200Step *io, cudaStream_t st) {
    int rc = check_io<T>(n_env, io);
    if (rc || n_env == 0) return rc;
    if (!hp) return CLOTHB200_ERR_ARG;
    StepArgs<T> A = make_args<T>(n_env, io);
    A.mode = KMODE_MEASURE;
    A.reward = nullptr;   // no bookkeeping
    return launch_step<T>(*hp, A, st);
}

template <typename T>
int decode_actions_t(const ClothB200Params *hp, int n_env, const T *actions, ClothB200Plan *plans, cudaStream_t st) {
    if (!hp || n_env < 0 || (n_env > 0 && (!actions || !plans))) return CLOTHB200_ERR_ARG;
    if (n_env == 0) return CLOTHB200_OK;
    decode_actions_kernel<T><<<(n_env + 127) / 128, 128, 0, st>>>(n_env, actions, plans, hp->clip_act_space, hp->delta_actions,
                                                                 hp->reduce_factor, hp->iters_pull_max);
    g_launch_count++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_cuda_error(e, "decode_actions_kernel"); return CLOTHB200_ERR_CUDA; }
    return CLOTHB200_OK;
}

template <typename T>
int broadcast_state_t(int n_points, int n_env, const T *pos4, const T *prev4, T *pos, T *prev, cudaStream_t st) {
    if (n_points <= 0 || n_env < 0 || !pos4 || !prev4 || !pos || !prev) return CLOTHB200_ERR_ARG;
    if (n_env == 0) return CLOTHB200_OK;
    const size_t total = (size_t)n_points * 4 * n_env;
    int blocks = (int)((total + 255) / 256); if (blocks > 148 * 16) blocks = 148 * 16;
    broadcast_state_kernel<T><<<blocks, 256, 0, st>>>(n_points * 4, n_env, pos4, prev4, pos, prev);
    g_launch_count++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_cuda_error(e, "broadcast_state_kernel"); return CLOTHB200_ERR_CUDA; }
    return CLOTHB200_OK;
}

template <typename T> int gripper_adjust_t(int n_points, int n_env, double x, double y, double z, T *pos, T *prev, cudaStream_t st) {
    if (n_points <= 0 || n_env < 0 || !pos || !prev) return CLOTHB200_ERR_ARG;
    const size_t total = (size_t)n_points * n_env;
    if (!total) return CLOTHB200_OK;
    gripper_adjust_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(total, (T)x, (T)y, (T)z, pos, prev);
    g_launch_count++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_cuda_error(e, "gripper_adjust_kernel"); return CLOTHB200_ERR_CUDA; }
    return CLOTHB200_OK;
}
template <typename T> int gripper_release_t(int n_points, int n_env, T *pos, T *prev, cudaStream_t st) {
    if (n_points <= 0 || n_env < 0 || !pos || !prev) return CLOTHB200_ERR_ARG;
    const size_t total = (size_t)n_points * n_env;
    if (!total) return CLOTHB200_OK;
    gripper_release_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(total, pos, prev);
    g_launch_count++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_cuda_error(e, "gripper_release_kernel"); return CLOTHB200_ERR_CUDA; }
    return CLOTHB200_OK;
}

}  // namespace clothb200
