// cloth_f32.cu - production instantiation (float state, FMA contraction allowed).
#include <cstring>
#include "cloth_typed.cuh"
#include "cloth_render.cuh"
namespace clothb200 {
int step_plans_f32(const ClothB200Params *p, int mode, int n, const ClothB200Plan *plans, const ClothB200Step *io, int init, const ClothB200Physics *ph, cudaStream_t st) { return step_plans_t<float>(p, mode, n, plans, io, init, ph, st); }
int update_n_f32(const ClothB200Params *p, int mode, int n, int k, const ClothB200Step *io, const ClothB200Physics *ph, cudaStream_t st) { return update_n_t<float>(p, mode, n, k, io, ph, st); }
int grab_top_f32(const ClothB200Params *p, int n, const double *xy, double r, const ClothB200Step *io, cudaStream_t st) { return grab_top_t<float>(p, n, xy, r, io, st); }
int measure_f32(const ClothB200Params *p, int n, const ClothB200Step *io, cudaStream_t st) { return measure_t<float>(p, n, io, st); }
int decode_actions_f32(const ClothB200Params *p, int n, const float *a, ClothB200Plan *plans, cudaStream_t st) { return decode_actions_t<float>(p, n, a, plans, st); }
int broadcast_state_f32(int np, int n, const float *a, const float *b, float *c, float *d, cudaStream_t st) { return broadcast_state_t<float>(np, n, a, b, c, d, st); }
int gripper_adjust_f32(int np, int n, double x, double y, double z, float *pos, float *prev, cudaStream_t st) { return gripper_adjust_t<float>(np, n, x, y, z, pos, prev, st); }
int gripper_release_f32(int np, int n, float *pos, float *prev, cudaStream_t st) { return gripper_release_t<float>(np, n, pos, prev, st); }
thread_local KernelInfo *g_kernel_query = nullptr;   // declared in cloth_kernels.cuh
size_t step_smem_f32(const ClothB200Params *p) { return step_smem_bytes<float>(*p); }
int kernel_info_f32(const ClothB200Params *p, int mode, int rt, int phys, int *out) { return kernel_info_t<float>(p, mode, rt, phys, out); }
int render_f32(const ClothB200Params *p, const ClothB200Scene *sc, const ClothB200SceneEnv *env, int n, const float *pos, int depth, uint8_t *out, float *zbuf, unsigned *minmax, cudaStream_t st) { return render_t<float>(p, sc, env, n, pos, depth != 0, out, zbuf, minmax, st); }
}  // namespace clothb200
