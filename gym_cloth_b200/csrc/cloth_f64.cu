// cloth_f64.cu - parity instantiation (double state).  Compiled with -fmad=false so that every operator is one
// rounded IEEE operation, like the reference's Python-float arithmetic: results are bit-identical to the oracle.
#include <cstring>
#include "cloth_typed.cuh"
#include "cloth_render.cuh"
namespace clothb200 {
int step_plans_f64(const ClothB200Params *p, int mode, int n, const ClothB200Plan *plans, const ClothB200Step *io, int init, const ClothB200Physics *ph, cudaStream_t st) { return step_plans_t<double>(p, mode, n, plans, io, init, ph, st); }
int update_n_f64(const ClothB200Params *p, int mode, int n, int k, const ClothB200Step *io, const ClothB200Physics *ph, cudaStream_t st) { return update_n_t<double>(p, mode, n, k, io, ph, st); }
int grab_top_f64(const ClothB200Params *p, int n, const double *xy, double r, const ClothB200Step *io, cudaStream_t st) { return grab_top_t<double>(p, n, xy, r, io, st); }
int measure_f64(const ClothB200Params *p, int n, const ClothB200Step *io, cudaStream_t st) { return measure_t<double>(p, n, io, st); }
int decode_actions_f64(const ClothB200Params *p, int n, const double *a, ClothB200Plan *plans, cudaStream_t st) { return decode_actions_t<double>(p, n, a, plans, st); }
int broadcast_state_f64(int np, int n, const double *a, const double *b, double *c, double *d, cudaStream_t st) { return broadcast_state_t<double>(np, n, a, b, c, d, st); }
int gripper_adjust_f64(int np, int n, double x, double y, double z, double *pos, double *prev, cudaStream_t st) { return gripper_adjust_t<double>(np, n, x, y, z, pos, prev, st); }
int gripper_release_f64(int np, int n, double *pos, double *prev, cudaStream_t st) { return gripper_release_t<double>(np, n, pos, prev, st); }
size_t step_smem_f64(const ClothB200Params *p) { return step_smem_bytes<double>(*p); }
int kernel_info_f64(const ClothB200Params *p, int mode, int rt, int phys, int *out) { return kernel_info_t<double>(p, mode, rt, phys, out); }
int render_f64(const ClothB200Params *p, const ClothB200Scene *sc, const ClothB200SceneEnv *env, int n, const double *pos, int depth, uint8_t *out, float *zbuf, unsigned *minmax, cudaStream_t st) { return render_t<double>(p, sc, env, n, pos, depth != 0, out, zbuf, minmax, st); }
}  // namespace clothb200
