// cloth_abi.cu - the extern "C" surface declared in include/clothb200.h, plus the host-side pieces
// (config-derived constants, initial grid, exact action decode) and two peak microbenchmarks.
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/clothb200.h"

namespace clothb200 {
std::atomic<long long> g_launch_count{0};
long long *g_prof_ptr = nullptr;
int g_force_slots = 0, g_force_slice = 0;
// Longest-remaining-first swapping with hysteresis: with equal-length actions every slice would otherwise end in a swap
// (the waiting cloth is always one slice behind the running one); two slices of slack cut the swaps - 40 KB of L2/HBM
// traffic each - to a third at the same throughput (measured 0 / 64 / 192 / 448 substeps: 18.73 / 18.82 / 18.65 / 18.59 M
// substeps/s).
int yield_slack_substeps() {
    static int v = [] { const char *s = getenv("CLOTHB200_YIELD_SLACK"); int x = s ? atoi(s) : 128; return x < 0 ? 0 : x; }();
    return v;
}
// The last CLOTHB200_ENDGAME slices of an action run in slices (and with a swap hysteresis) of 1 / 2^CLOTHB200_ENDGAME_SHIFT
// of the normal length: a launch ends with its last cloth, and what the slots differ by at the end is the grain of the
// hand-over.  Measured (4096 cloths, seeds 1337-1340): launch 402 / 398 / 390 / 405 ms without, 387-389 / 386 / 384 / 391 ms
// with the defaults 12 and 2, against 379 ms of work per slot.
int endgame_slices() {
    static int v = [] { const char *s = getenv("CLOTHB200_ENDGAME"); int x = s ? atoi(s) : 12; return x < 0 ? 0 : x; }();
    return v;
}
int endgame_shift() {
    static int v = [] { const char *s = getenv("CLOTHB200_ENDGAME_SHIFT"); int x = s ? atoi(s) : 2; return x < 0 ? 0 : (x > 6 ? 6 : x); }();
    return v;
}
int slice_substeps() {
    static int v = [] { const char *s = getenv("CLOTHB200_SLICE"); int x = s ? atoi(s) : 64; return x < 0 ? 0 : x; }();
    return v;
}
int g_debug_flags = [] { const char *s = getenv("CLOTHB200_DEBUG"); return s ? atoi(s) : 0; }();
static thread_local std::string g_cuda_err;
void set_cuda_error(cudaError_t e, const char *where) {
    g_cuda_err = std::string(where) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
}
int threads_per_cloth(int W) {
    static int nt = [] {
        const char *s = getenv("CLOTHB200_NT");
        int v = s ? atoi(s) : 0;
        return (v == 128 || v == 256 || v == 512) ? v : 0;
    }();
    if (nt) return nt;
    return W >= 64 ? 512 : 128;
}
int sweep_threshold() {
    static int v = [] { const char *s = getenv("CLOTHB200_SWEEP_THRESH"); return s ? atoi(s) : 128; }();
    return v;
}
// Static dependency-level schedule of the spring list (cloth.pyx:135-146 order).  A few KB of device memory per
// (device, grid width), built once and kept for the life of the process: the one exception to "the library owns no
// persistent device memory".
const uint32_t *get_sweep_table(int W, int *levels, int *lw) {
    struct Entry { uint32_t *dev; int levels, lw; };
    static std::map<std::pair<int, int>, Entry> cache;
    static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { *levels = 0; *lw = 0; return nullptr; }
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find({dev, W});
    if (it == cache.end()) {
        const int N = W * W;
        if (N > 4096 || sweep_threshold() <= 0) { cache[{dev, W}] = {nullptr, 0, 0}; it = cache.find({dev, W}); }
        else {
            std::vector<int> last(N, 0);
            std::vector<std::vector<uint32_t>> per_level;
            const int offs[6] = {W, 1, W + 1, W - 1, 2 * W, 2};
            for (int q = 0; q < N; q++) {
                const int r = q / W, c = q % W;
                const bool ok[6] = {r > 0, c > 0, r > 0 && c > 0, r > 0 && c + 1 < W, r > 1, c > 1};
                for (int k = 0; k < 6; k++) if (ok[k]) {
                    const int a = q - offs[k];
                    const int l = 1 + (last[a] > last[q] ? last[a] : last[q]);
                    last[a] = l; last[q] = l;
                    if ((int)per_level.size() < l) per_level.resize(l);
                    per_level[l - 1].push_back((uint32_t)a | ((uint32_t)q << 12) | ((uint32_t)k << 24));
                }
            }
            size_t width = 0;
            for (auto &v : per_level) width = v.size() > width ? v.size() : width;
            // rows of 32 entries (one per lane), padded with empty rows to a multiple of eight levels plus eight more:
            // limit_sweep() reads eight levels ahead without bounds or lane checks
            Entry en{nullptr, (int)per_level.size(), 32};
            if (width <= 32) {
                const size_t rows = (((size_t)en.levels + 7) / 8) * 8 + 8;
                std::vector<uint32_t> flat(rows * 32, 0xffffffffu);
                for (int l = 0; l < en.levels; l++) for (size_t i = 0; i < per_level[l].size(); i++) flat[(size_t)l * 32 + i] = per_level[l][i];
                if (cudaMalloc((void **)&en.dev, flat.size() * 4) == cudaSuccess)
                    cudaMemcpy(en.dev, flat.data(), flat.size() * 4, cudaMemcpyHostToDevice);
                else en.dev = nullptr;
            }
            cache[{dev, W}] = en;
            it = cache.find({dev, W});
        }
    }
    *levels = it->second.levels; *lw = it->second.lw;
    return it->second.dev;
}
// typed entry points (cloth_f32.cu / cloth_f64.cu)
#define DECL_TYPED(SFX, T)                                                                                                               \
    int step_plans_##SFX(const ClothB200Params *, int, int, const ClothB200Plan *, const ClothB200Step *, int, const ClothB200Physics *, cudaStream_t); \
    int update_n_##SFX(const ClothB200Params *, int, int, int, const ClothB200Step *, const ClothB200Physics *, cudaStream_t);          \
    int grab_top_##SFX(const ClothB200Params *, int, const double *, double, const ClothB200Step *, cudaStream_t);                       \
    int measure_##SFX(const ClothB200Params *, int, const ClothB200Step *, cudaStream_t);                                                \
    int decode_actions_##SFX(const ClothB200Params *, int, const T *, ClothB200Plan *, cudaStream_t);                                    \
    int broadcast_state_##SFX(int, int, const T *, const T *, T *, T *, cudaStream_t);                                                   \
    int gripper_adjust_##SFX(int, int, double, double, double, T *, T *, cudaStream_t);                                                  \
    int gripper_release_##SFX(int, int, T *, T *, cudaStream_t);                                                                         \
    int render_##SFX(const ClothB200Params *, const ClothB200Scene *, const ClothB200SceneEnv *, int, const T *, int, uint8_t *, float *, unsigned *, cudaStream_t); \
    size_t step_smem_##SFX(const ClothB200Params *);                                                                                    \
    int kernel_info_##SFX(const ClothB200Params *, int, int, int, int *);
DECL_TYPED(f32, float)
DECL_TYPED(f64, double)

static int check_cuda(cudaError_t e, const char *where) {
    if (e == cudaSuccess) return CLOTHB200_OK;
    set_cuda_error(e, where);
    return CLOTHB200_ERR_CUDA;
}

// Cloth.__init__ grid + Spring.rest_length in IEEE double (cloth.pyx:92-146, 411-417)
template <typename T>
static int init_grid(const ClothB200Params *hp, int init_type, const double *noise, int init_side, T *pos4, T *prev4, T *rest6) {
    if (!hp) return CLOTHB200_ERR_ARG;
    const int W = hp->num_width_points, H = hp->num_height_points;
    if (W != H || W < 2) return CLOTHB200_ERR_CONFIG;                 // cloth.pyx:91
    if (init_type < 1 || init_type > 3) return CLOTHB200_ERR_CONFIG;  // cloth.pyx:131-132
    if (init_type == 2 && !noise) return CLOTHB200_ERR_ARG;
    const int N = W * H;
    const double dx = hp->width * 1.0 / (W - 1), dy = hp->height * 1.0 / (H - 1);
    double *xyz = (double *)malloc(sizeof(double) * 3 * N);
    if (rest6) for (int i = 0; i < 6 * N; i++) rest6[i] = (T)0;
    for (int r = 0; r < H; r++)
        for (int c = 0; c < W; c++) {
            const int p = r * W + c;
            double x, y, z;
            if (init_type == 2) {
                double nz = noise[p];
                if (r == 0) nz = 0.0;
                x = init_side ? 0.0 + fabs(nz) : 1.0 - fabs(nz);
                y = dx * c; z = dy * r;
            } else { x = dx * r; y = dy * c; z = 0.0; }
            xyz[3 * p] = x; xyz[3 * p + 1] = y; xyz[3 * p + 2] = z;
            if (pos4) { pos4[4 * p] = (T)x; pos4[4 * p + 1] = (T)y; pos4[4 * p + 2] = (T)z; pos4[4 * p + 3] = (T)0; }
            if (prev4) { prev4[4 * p] = (T)x; prev4[4 * p + 1] = (T)y; prev4[4 * p + 2] = (T)z; prev4[4 * p + 3] = (T)0; }
            if (rest6) {
                const int offs[6] = {W, 1, W + 1, W - 1, 2 * W, 2};
                const bool ok[6] = {r > 0, c > 0, r > 0 && c > 0, r > 0 && c + 1 < W, r > 1, c > 1};
                for (int k = 0; k < 6; k++)
                    if (ok[k]) {
                        const double *a = xyz + 3 * (p - offs[k]);
                        const double d0 = a[0] - x, d1 = a[1] - y, d2 = a[2] - z;   // ptA - ptB
                        rest6[6 * p + k] = (T)sqrt(d0 * d0 + d1 * d1 + d2 * d2);
                    }
            }
        }
    free(xyz);
    return CLOTHB200_OK;
}

static double clampd(double v, double lo, double hi) {
    const double m = (hi < v) ? hi : v;   // Python min(v, hi)
    return (lo > m) ? lo : m;             // Python max(m, lo)
}

// per-thread scratch of the *_host entry points
struct HostScratch {
    ClothB200Plan *pinned = nullptr, *dev = nullptr;
    int cap = 0, device = -1;
    int ensure(int n) {
        int cur = 0;
        cudaGetDevice(&cur);
        if (n <= cap && cur == device) return CLOTHB200_OK;      // the device buffer belongs to the device it was made on
        device = cur;
        if (pinned) cudaFreeHost(pinned);
        if (dev) cudaFree(dev);
        pinned = nullptr; dev = nullptr; cap = 0;
        int rc = check_cuda(cudaMallocHost((void **)&pinned, sizeof(ClothB200Plan) * (size_t)n), "cudaMallocHost(plans)");
        if (rc) return rc;
        rc = check_cuda(cudaMalloc((void **)&dev, sizeof(ClothB200Plan) * (size_t)n), "cudaMalloc(plans)");
        if (rc) return rc;
        cap = n;
        return CLOTHB200_OK;
    }
};
static thread_local HostScratch g_scratch;

// Per-environment material rows of the *_phys_* entry points (launch_step): one device buffer per thread, grown when a
// call needs more and reused by the next call, so that the many small update_n calls of a reset allocate nothing.  An
// event recorded behind each call's step kernel orders reuse: a call on another stream waits for it before its derive
// kernel overwrites the rows (on the same stream the wait is already implied).
struct MaterialRows {
    void *dev = nullptr;
    size_t cap = 0;
    int device = -1;
    cudaEvent_t done = nullptr;
};
static thread_local MaterialRows g_rows;

void *material_rows(size_t bytes, cudaStream_t st, int *rc) {
    int cur = 0;
    cudaGetDevice(&cur);
    MaterialRows &m = g_rows;
    if (m.device != cur || bytes > m.cap) {
        if (m.done) { cudaEventSynchronize(m.done); cudaEventDestroy(m.done); }   // the old rows may still be read
        if (m.dev) cudaFree(m.dev);
        m = MaterialRows();
        size_t cap = 8192;
        while (cap < bytes) cap <<= 1;
        *rc = check_cuda(cudaMalloc(&m.dev, cap), "cudaMalloc(material rows)");
        if (*rc == CLOTHB200_OK) *rc = check_cuda(cudaEventCreateWithFlags(&m.done, cudaEventDisableTiming), "cudaEventCreate(material rows)");
        if (*rc) {
            if (m.dev) cudaFree(m.dev);
            m = MaterialRows();
            cudaGetLastError();
            return nullptr;
        }
        m.cap = cap; m.device = cur;
        return m.dev;
    }
    *rc = check_cuda(cudaStreamWaitEvent(st, m.done, 0), "cudaStreamWaitEvent(material rows)");
    return *rc ? nullptr : m.dev;
}
int material_rows_release(cudaStream_t st) { return check_cuda(cudaEventRecord(g_rows.done, st), "cudaEventRecord(material rows)"); }

// ---- microbenchmarks: this GPU's shared-memory bandwidth and FP32 FMA rate (roofline denominators) ----
__global__ void __launch_bounds__(1024) smem_bw_kernel(int iters, float *sink) {
    __shared__ float4 buf[2048];   // 32 KB
    for (int i = threadIdx.x; i < 2048; i += blockDim.x) buf[i] = make_float4(i, 1.f, 2.f, 3.f);
    __syncthreads();
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int idx = threadIdx.x;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const float4 v = buf[(idx + u * 256) & 2047];
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        idx = (idx + 32) & 2047;
    }
    if (acc.x + acc.y + acc.z + acc.w == 123.456f) sink[0] = acc.x;
}
__global__ void __launch_bounds__(1024) fp32_fma_kernel(int iters, float *sink) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float b = 1.000001f, c = 1e-7f;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
            a0 = fmaf(a0, b, c); a1 = fmaf(a1, b, c); a2 = fmaf(a2, b, c); a3 = fmaf(a3, b, c);
            a4 = fmaf(a4, b, c); a5 = fmaf(a5, b, c); a6 = fmaf(a6, b, c); a7 = fmaf(a7, b, c);
        }
    }
    const float s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123.456f) sink[0] = s;
}

// ---- what cloth_env.py does to the PNG Blender wrote (cloth_env.py:296-315) ----
// cv2.bilateralFilter(img, 7, 50, 50) on a three-channel image whose channels are equal: radius 3, circular support,
// BORDER_REFLECT_101, colour distance = sum of the three channel differences; then max(0, img - sub) and the noise
__global__ void post_depth_kernel(int n, int H, int W, const uint8_t *__restrict__ gray, const float *__restrict__ sub,
                                  const float *__restrict__ noise, uint8_t *__restrict__ out) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= (size_t)n * H * W) return;
    const int e = (int)(i / ((size_t)H * W));
    const int r = (int)((i / W) % H), c = (int)(i % W);
    const uint8_t *img = gray + (size_t)e * H * W;
    const int v0 = img[r * W + c];
    const float gc = -0.5f / (50.f * 50.f), gs = -0.5f / (50.f * 50.f);
    float sum = 0.f, wsum = 0.f;
    for (int di = -3; di <= 3; di++)
        for (int dj = -3; dj <= 3; dj++) {
            const int rr2 = di * di + dj * dj;
            if (rr2 > 9) continue;
            int y = r + di, x = c + dj;
            y = y < 0 ? -y : (y >= H ? 2 * H - 2 - y : y);
            x = x < 0 ? -x : (x >= W ? 2 * W - 2 - x : x);
            const int v = img[y * W + x];
            const int dc = 3 * abs(v - v0);
            const float w = expf((float)rr2 * gs) * expf((float)(dc * dc) * gc);
            sum += (float)v * w; wsum += w;
        }
    const int f = __float2int_rn(sum * (1.f / wsum));
    const double g = sub ? (double)sub[e] : 50.0;
    double d = (double)f - g;
    const uint8_t v1 = (uint8_t)(d > 0.0 ? d : 0.0);                      // np.uint8(np.maximum(0, np.double(img) - gval))
    for (int ch = 0; ch < 3; ch++) {
        uint8_t o = v1;
        if (noise) { double t = (double)v1 + (double)noise[3 * i + ch]; t = t < 0.0 ? 0.0 : (t > 255.0 ? 255.0 : t); o = (uint8_t)t; }
        out[3 * i + ch] = o;
    }
}
__global__ void post_rgb_kernel(int n, int H, int W, uint8_t *__restrict__ bgr, const uint8_t *__restrict__ lut, const float *__restrict__ noise) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= (size_t)n * H * W * 3) return;
    const int e = (int)(i / ((size_t)H * W * 3));
    uint8_t v = bgr[i];
    if (lut) v = lut[256 * e + v];                                         // cv2.LUT(image, table), cloth_env.py:1217-1228
    if (noise) { double t = (double)v + (double)noise[i]; t = t < 0.0 ? 0.0 : (t > 255.0 ? 255.0 : t); v = (uint8_t)t; }
    bgr[i] = v;
}
}  // namespace clothb200

using namespace clothb200;

extern "C" {

int clothb200_version(void) { return CLOTHB200_VERSION; }

const char *clothb200_error_string(int code) {
    switch (code) {
        case CLOTHB200_OK: return "ok";
        case CLOTHB200_ERR_ARG: return "bad argument (NULL / negative size / tensor not 16-byte aligned)";
        case CLOTHB200_ERR_CONFIG: return "configuration rejected (non-square grid, unknown init type or pin_cond)";
        case CLOTHB200_ERR_CUDA: return "CUDA runtime error (see clothb200_last_cuda_error)";
        case CLOTHB200_ERR_UNSUPPORTED: return "unsupported (mode not built, or cloth too large for one CTA's shared memory)";
        case CLOTHB200_ERR_NO_DEVICE: return "no usable CUDA device";
        default: return "unknown error";
    }
}
const char *clothb200_last_cuda_error(void) { return g_cuda_err.c_str(); }
size_t clothb200_sizeof_params(void) { return sizeof(ClothB200Params); }
size_t clothb200_sizeof_plan(void) { return sizeof(ClothB200Plan); }
size_t clothb200_sizeof_step(void) { return sizeof(ClothB200Step); }
size_t clothb200_sizeof_physics(void) { return sizeof(ClothB200Physics); }
int clothb200_debug_set_slicing(int resident_ctas, int slice_substeps) {
    g_force_slots = resident_ctas > 0 ? resident_ctas : 0;
    g_force_slice = slice_substeps > 0 ? slice_substeps : 0;
    return CLOTHB200_OK;
}
size_t clothb200_sched_scratch_bytes(int n_env) {
    if (n_env < 1) return 0;
    size_t np2 = 1; while (np2 < (size_t)n_env) np2 <<= 1;
    // sort keys | launch order (padded to 8 bytes) | queue | progress, grip count, cycles | queue counters
    return 8 * np2 + 8 * (((size_t)n_env + 1) / 2) + 8 * (size_t)n_env + 12 * (size_t)n_env + 16;
}
int64_t clothb200_launch_count(void) { return (int64_t)g_launch_count.load(); }
int clothb200_debug_set_profile(void *dev_int64_nenv_x16) { g_prof_ptr = (long long *)dev_int64_nenv_x16; return CLOTHB200_OK; }

int clothb200_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, int *smem_per_sm) {
    int dev = device;
    if (dev < 0 && cudaGetDevice(&dev) != cudaSuccess) return CLOTHB200_ERR_NO_DEVICE;
    cudaDeviceProp pr;
    if (cudaGetDeviceProperties(&pr, dev) != cudaSuccess) return CLOTHB200_ERR_NO_DEVICE;
    if (sm_count) *sm_count = pr.multiProcessorCount;
    if (cc_major) *cc_major = pr.major;
    if (cc_minor) *cc_minor = pr.minor;
    if (smem_per_sm) *smem_per_sm = (int)pr.sharedMemPerMultiprocessor;
    return CLOTHB200_OK;
}

int clothb200_step_kernel_info(const ClothB200Params *p, int is_f64, int mode, int rest_table, int per_env_physics, int *ctas_per_sm,
                               int *registers, int *local_bytes, int *smem_bytes) {
    if (!p) return CLOTHB200_ERR_ARG;
    if (mode != CLOTHB200_MODE_REFERENCE_ORDER && mode != CLOTHB200_MODE_COLOURED) return CLOTHB200_ERR_UNSUPPORTED;
    int out[4] = {0, 0, 0, 0};
    const int rc = is_f64 ? kernel_info_f64(p, mode, rest_table, per_env_physics, out) : kernel_info_f32(p, mode, rest_table, per_env_physics, out);
    if (rc) return rc;
    if (ctas_per_sm) *ctas_per_sm = out[0];
    if (registers) *registers = out[1];
    if (local_bytes) *local_bytes = out[2];
    if (smem_bytes) *smem_bytes = out[3];
    return CLOTHB200_OK;
}

int clothb200_occupancy(const ClothB200Params *p, int is_f64, int *ctas_per_sm, int *smem_bytes, int *threads) {
    if (!p) return CLOTHB200_ERR_ARG;
    const size_t sm = is_f64 ? step_smem_f64(p) : step_smem_f32(p);
    if (smem_bytes) *smem_bytes = (int)sm;
    if (threads) *threads = threads_per_cloth(p->num_width_points);
    if (ctas_per_sm) {
        const int by_smem = (int)((228 * 1024) / (sm + 1024));
        const int by_thr = 2048 / threads_per_cloth(p->num_width_points);
        int v = by_smem < by_thr ? by_smem : by_thr;
        *ctas_per_sm = v < 32 ? v : 32;
    }
    return CLOTHB200_OK;
}

int clothb200_params_default(ClothB200Params *p) {
    if (!p) return CLOTHB200_ERR_ARG;
    memset(p, 0, sizeof(*p));
    p->num_width_points = 25; p->num_height_points = 25;
    p->width = 1.0; p->height = 1.0;
    p->density = 200.0; p->ks = 10000.0; p->damping = 2.0; p->thickness = 0.02;
    p->plane_friction = 1.0; p->tear_thresh = 2.0;
    p->gravity = -9.8; p->minimum_z = 0.0;
    p->frames_per_sec = 30; p->simulation_steps = 30;
    p->iters_up = 50; p->iters_up_rest = 80; p->iters_grip_rest = 300; p->iters_rest = 1000;
    p->iters_pull_max = 400; p->max_actions = 10;
    p->reduce_factor = 0.002; p->grip_radius = 0.003; p->gripper_height = 1.0;
    p->clip_act_space = 1; p->delta_actions = 1;
    return CLOTHB200_OK;
}

int clothb200_params_validate(const ClothB200Params *p) {
    if (!p) return CLOTHB200_ERR_ARG;
    if (p->num_width_points != p->num_height_points || p->num_width_points < 3) return CLOTHB200_ERR_CONFIG;
    if (p->num_width_points * p->num_height_points >= 32768) return CLOTHB200_ERR_UNSUPPORTED;
    if (!(p->thickness > 0) || !(p->density > 0) || p->frames_per_sec <= 0 || p->simulation_steps <= 0) return CLOTHB200_ERR_CONFIG;
    if (!(p->gripper_height / p->thickness < 4096)) return CLOTHB200_ERR_UNSUPPORTED;
    if (p->reward_type != CLOTHB200_REWARD_COVERAGE_DELTA && p->reward_type != CLOTHB200_REWARD_COVERAGE) return CLOTHB200_ERR_CONFIG;
    return CLOTHB200_OK;
}

int clothb200_init_grid_f32(const ClothB200Params *p, int t, const double *nz, int side, float *a, float *b, float *r) { return init_grid<float>(p, t, nz, side, a, b, r); }
int clothb200_init_grid_f64(const ClothB200Params *p, int t, const double *nz, int side, double *a, double *b, double *r) { return init_grid<double>(p, t, nz, side, a, b, r); }

int clothb200_broadcast_state_f32(int np, int n, const float *a, const float *b, float *c, float *d, void *st) { return broadcast_state_f32(np, n, a, b, c, d, (cudaStream_t)st); }
int clothb200_broadcast_state_f64(int np, int n, const double *a, const double *b, double *c, double *d, void *st) { return broadcast_state_f64(np, n, a, b, c, d, (cudaStream_t)st); }

// cloth_env.py:401-470 in IEEE double with libm pow() for `**2` (what CPython's float_pow calls)
int clothb200_decode_actions_host(const ClothB200Params *P, int n_env, const double *actions, ClothB200Plan *plans) {
    if (!P || n_env < 0 || (n_env > 0 && (!actions || !plans))) return CLOTHB200_ERR_ARG;
    double lo[4], hi[4];
    const double pi_f32 = 3.1415927410125732;   // spaces.Box casts its bounds to float32 (cloth_env.py:178-181)
    if (P->clip_act_space) { for (int i = 0; i < 4; i++) { lo[i] = -1.0; hi[i] = 1.0; } }
    else if (P->delta_actions) { lo[0] = 0; lo[1] = 0; lo[2] = -1; lo[3] = -1; hi[0] = hi[1] = hi[2] = hi[3] = 1; }
    else { lo[0] = -0.25; lo[1] = -0.25; lo[2] = 0.0; lo[3] = -pi_f32; hi[0] = 1.25; hi[1] = 1.25; hi[2] = 1.0; hi[3] = pi_f32; }
    for (int e = 0; e < n_env; e++) {
        const double *a = actions + 4 * e;
        if (a[0] != a[0] || a[1] != a[1] || a[2] != a[2] || a[3] != a[3]) {
            // NaN survives np.clip and the reference's `while True: current_l += ...; if current_l >= total` loop
            // (cloth_env.py:462-467) would never exit: the plan is marked bad, the step does nothing and reports BADSTATE
            plans[e].gx = 0.5; plans[e].gy = 0.5; plans[e].dxr = 0.0; plans[e].dyr = 0.0; plans[e].iters_pull = 0;
            plans[e].reserved = CLOTHB200_PLAN_BAD_ACTION;
            continue;
        }
        double x = clampd(a[0], lo[0], hi[0]), y = clampd(a[1], lo[1], hi[1]);
        const double a2 = clampd(a[2], lo[2], hi[2]), a3 = clampd(a[3], lo[3], hi[3]);
        double length = a2, radians = a3;
        if (P->clip_act_space) {
            x = (x / 2.0) + 0.5; y = (y / 2.0) + 0.5;
            if (!P->delta_actions) { length = (length / 2.0) + 0.5; radians = radians * 3.141592653589793; }
        }
        double xd, yd, total = 0.0;
        if (P->delta_actions) {
            total = sqrt(pow(a2, 2.0) + pow(a3, 2.0));
            xd = a2 / (total + 1e-5); yd = a3 / (total + 1e-5);
        } else { xd = cos(radians); yd = sin(radians); }
        const double xr = xd * P->reduce_factor, yr = yd * P->reduce_factor;
        int ip;
        if (P->delta_actions) {
            const double stepl = sqrt(pow(xr, 2.0) + pow(yr, 2.0));
            int ii = 0;
            if (stepl > 0.0) { double cur = 0; for (;;) { cur += stepl; if (cur >= total || ii >= CLOTHB200_MAX_ITERS_PULL) break; ii += 1; } }
            ip = ii;
        } else ip = (int)(P->iters_pull_max * length);
        plans[e].gx = x; plans[e].gy = y; plans[e].dxr = xr; plans[e].dyr = yr; plans[e].iters_pull = ip; plans[e].reserved = 0;
    }
    return CLOTHB200_OK;
}
int clothb200_decode_actions_f32(const ClothB200Params *p, int n, const float *a, ClothB200Plan *plans, void *st) { return decode_actions_f32(p, n, a, plans, (cudaStream_t)st); }
int clothb200_decode_actions_f64(const ClothB200Params *p, int n, const double *a, ClothB200Plan *plans, void *st) { return decode_actions_f64(p, n, a, plans, (cudaStream_t)st); }

// physics == NULL: the batch's material (the plain entry points below are these with NULL)
int clothb200_step_plans_phys_f32(const ClothB200Params *p, int mode, int n, const ClothB200Plan *plans, const ClothB200Step *io, int init, const ClothB200Physics *ph, void *st) { return step_plans_f32(p, mode, n, plans, io, init, ph, (cudaStream_t)st); }
int clothb200_step_plans_phys_f64(const ClothB200Params *p, int mode, int n, const ClothB200Plan *plans, const ClothB200Step *io, int init, const ClothB200Physics *ph, void *st) { return step_plans_f64(p, mode, n, plans, io, init, ph, (cudaStream_t)st); }
int clothb200_step_plans_f32(const ClothB200Params *p, int mode, int n, const ClothB200Plan *plans, const ClothB200Step *io, int init, void *st) { return clothb200_step_plans_phys_f32(p, mode, n, plans, io, init, nullptr, st); }
int clothb200_step_plans_f64(const ClothB200Params *p, int mode, int n, const ClothB200Plan *plans, const ClothB200Step *io, int init, void *st) { return clothb200_step_plans_phys_f64(p, mode, n, plans, io, init, nullptr, st); }

int clothb200_step_actions_phys_f32(const ClothB200Params *p, int mode, int n, const float *actions, ClothB200Plan *scratch, const ClothB200Step *io, int init, const ClothB200Physics *ph, void *st) {
    int rc = decode_actions_f32(p, n, actions, scratch, (cudaStream_t)st);
    if (rc) return rc;
    return step_plans_f32(p, mode, n, scratch, io, init, ph, (cudaStream_t)st);
}
int clothb200_step_actions_phys_f64(const ClothB200Params *p, int mode, int n, const double *actions, ClothB200Plan *scratch, const ClothB200Step *io, int init, const ClothB200Physics *ph, void *st) {
    int rc = decode_actions_f64(p, n, actions, scratch, (cudaStream_t)st);
    if (rc) return rc;
    return step_plans_f64(p, mode, n, scratch, io, init, ph, (cudaStream_t)st);
}
int clothb200_step_actions_f32(const ClothB200Params *p, int mode, int n, const float *actions, ClothB200Plan *scratch, const ClothB200Step *io, int init, void *st) {
    return clothb200_step_actions_phys_f32(p, mode, n, actions, scratch, io, init, nullptr, st);
}
int clothb200_step_actions_f64(const ClothB200Params *p, int mode, int n, const double *actions, ClothB200Plan *scratch, const ClothB200Step *io, int init, void *st) {
    return clothb200_step_actions_phys_f64(p, mode, n, actions, scratch, io, init, nullptr, st);
}

int clothb200_update_n_phys_f32(const ClothB200Params *p, int mode, int n, int k, const ClothB200Step *io, const ClothB200Physics *ph, void *st) { return update_n_f32(p, mode, n, k, io, ph, (cudaStream_t)st); }
int clothb200_update_n_phys_f64(const ClothB200Params *p, int mode, int n, int k, const ClothB200Step *io, const ClothB200Physics *ph, void *st) { return update_n_f64(p, mode, n, k, io, ph, (cudaStream_t)st); }
int clothb200_update_n_f32(const ClothB200Params *p, int mode, int n, int k, const ClothB200Step *io, void *st) { return clothb200_update_n_phys_f32(p, mode, n, k, io, nullptr, st); }
int clothb200_update_n_f64(const ClothB200Params *p, int mode, int n, int k, const ClothB200Step *io, void *st) { return clothb200_update_n_phys_f64(p, mode, n, k, io, nullptr, st); }

int clothb200_grab_top_f32(const ClothB200Params *p, int n, const double *xy, double r, const ClothB200Step *io, void *st) { return grab_top_f32(p, n, xy, r, io, (cudaStream_t)st); }
int clothb200_grab_top_f64(const ClothB200Params *p, int n, const double *xy, double r, const ClothB200Step *io, void *st) { return grab_top_f64(p, n, xy, r, io, (cudaStream_t)st); }
int clothb200_gripper_adjust_f32(int np, int n, double x, double y, double z, float *pos, float *prev, void *st) { return gripper_adjust_f32(np, n, x, y, z, pos, prev, (cudaStream_t)st); }
int clothb200_gripper_adjust_f64(int np, int n, double x, double y, double z, double *pos, double *prev, void *st) { return gripper_adjust_f64(np, n, x, y, z, pos, prev, (cudaStream_t)st); }
int clothb200_gripper_release_f32(int np, int n, float *pos, float *prev, void *st) { return gripper_release_f32(np, n, pos, prev, (cudaStream_t)st); }
int clothb200_gripper_release_f64(int np, int n, double *pos, double *prev, void *st) { return gripper_release_f64(np, n, pos, prev, (cudaStream_t)st); }
size_t clothb200_sizeof_scene(void) { return sizeof(ClothB200Scene); }
int clothb200_scene_default(ClothB200Scene *s) {
    if (!s) return CLOTHB200_ERR_ARG;
    memset(s, 0, sizeof(*s));
    s->height = 224; s->width = 224; s->samples = 2;
    s->lens_mm = 40.f; s->sensor_mm = 36.f;
    s->cam_pos[0] = 0.5f; s->cam_pos[1] = 0.5f; s->cam_pos[2] = 1.45f;
    s->lamp_pos[0] = 4.07625f; s->lamp_pos[1] = 1.00545f; s->lamp_pos[2] = 5.90386f;
    s->lamp_energy = 1.5f; s->diffuse_intensity = 0.8f; s->horizon = 0.051f;
    s->bed_z = -0.05f; s->bed_x0 = 0.f; s->bed_x1 = 1.f; s->bed_y0 = 0.f; s->bed_y1 = 1.f;
    s->floor_z = -0.25f; s->floor_x0 = -0.5f; s->floor_x1 = 1.5f; s->floor_y0 = -0.25f; s->floor_y1 = 1.25f;
    s->front[0] = 0.070f; s->front[1] = 0.050f; s->front[2] = 0.600f;
    s->back[0] = 0.070f; s->back[1] = 0.300f; s->back[2] = 0.900f;
    s->bed[0] = 1.f; s->bed[1] = 1.f; s->bed[2] = 1.f;
    return CLOTHB200_OK;
}
int clothb200_render_rgb_f32(const ClothB200Params *p, const ClothB200Scene *sc, const ClothB200SceneEnv *env, int n, const float *pos, uint8_t *out, void *st) { return render_f32(p, sc, env, n, pos, 0, out, nullptr, nullptr, (cudaStream_t)st); }
int clothb200_render_rgb_f64(const ClothB200Params *p, const ClothB200Scene *sc, const ClothB200SceneEnv *env, int n, const double *pos, uint8_t *out, void *st) { return render_f64(p, sc, env, n, pos, 0, out, nullptr, nullptr, (cudaStream_t)st); }
int clothb200_render_depth_f32(const ClothB200Params *p, const ClothB200Scene *sc, const ClothB200SceneEnv *env, int n, const float *pos, float *zbuf, uint32_t *mm, uint8_t *out, void *st) { return render_f32(p, sc, env, n, pos, 1, out, zbuf, mm, (cudaStream_t)st); }
int clothb200_render_depth_f64(const ClothB200Params *p, const ClothB200Scene *sc, const ClothB200SceneEnv *env, int n, const double *pos, float *zbuf, uint32_t *mm, uint8_t *out, void *st) { return render_f64(p, sc, env, n, pos, 1, out, zbuf, mm, (cudaStream_t)st); }
int clothb200_post_depth(int n, int H, int W, const uint8_t *gray, const float *sub, const float *noise, uint8_t *out, void *st) {
    if (n < 0 || H < 2 || W < 2 || (n > 0 && (!gray || !out))) return CLOTHB200_ERR_ARG;
    if (n == 0) return CLOTHB200_OK;
    const size_t tot = (size_t)n * H * W;
    post_depth_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)st>>>(n, H, W, gray, sub, noise, out);
    g_launch_count++;
    return check_cuda(cudaGetLastError(), "post_depth launch");
}
int clothb200_post_rgb(int n, int H, int W, uint8_t *bgr, const uint8_t *lut, const float *noise, void *st) {
    if (n < 0 || H < 1 || W < 1 || (n > 0 && !bgr)) return CLOTHB200_ERR_ARG;
    if (n == 0 || (!lut && !noise)) return CLOTHB200_OK;
    const size_t tot = (size_t)n * H * W * 3;
    post_rgb_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)st>>>(n, H, W, bgr, lut, noise);
    g_launch_count++;
    return check_cuda(cudaGetLastError(), "post_rgb launch");
}
int clothb200_measure_f32(const ClothB200Params *p, int n, const ClothB200Step *io, void *st) { return measure_f32(p, n, io, (cudaStream_t)st); }
int clothb200_measure_f64(const ClothB200Params *p, int n, const ClothB200Step *io, void *st) { return measure_f64(p, n, io, (cudaStream_t)st); }

#define STEP_HOST_BODY(SFX, T)                                                                                                           \
    if (!p || !io || n < 0 || (n > 0 && !actions)) return CLOTHB200_ERR_ARG;                                                             \
    if (n == 0) return CLOTHB200_OK;                                                                                                     \
    if ((obs && !io->obs) || (reward && !io->reward) || (done && !io->done) || (coverage && !io->coverage) ||                            \
        (variance_inv && !io->variance_inv) || (flags && !io->flags) || (sim_steps && !io->sim_steps))                                   \
        return CLOTHB200_ERR_ARG;                                                                                                        \
    cudaStream_t s = (cudaStream_t)st;                                                                                                   \
    int rc = g_scratch.ensure(n);                                                                                                        \
    if (rc) return rc;                                                                                                                   \
    rc = clothb200_decode_actions_host(p, n, actions, g_scratch.pinned);                                                                 \
    if (rc) return rc;                                                                                                                   \
    rc = check_cuda(cudaMemcpyAsync(g_scratch.dev, g_scratch.pinned, sizeof(ClothB200Plan) * (size_t)n, cudaMemcpyHostToDevice, s), "H2D plans"); \
    if (rc) return rc;                                                                                                                   \
    rc = step_plans_##SFX(p, mode, n, g_scratch.dev, io, initialize, physics, s);                                                        \
    if (rc) return rc;                                                                                                                   \
    const size_t N3 = (size_t)3 * p->num_width_points * p->num_height_points;                                                            \
    if (obs) rc |= check_cuda(cudaMemcpyAsync(obs, io->obs, sizeof(T) * N3 * n, cudaMemcpyDeviceToHost, s), "D2H obs");                  \
    if (reward) rc |= check_cuda(cudaMemcpyAsync(reward, io->reward, 8 * (size_t)n, cudaMemcpyDeviceToHost, s), "D2H reward");           \
    if (done) rc |= check_cuda(cudaMemcpyAsync(done, io->done, 4 * (size_t)n, cudaMemcpyDeviceToHost, s), "D2H done");                   \
    if (coverage) rc |= check_cuda(cudaMemcpyAsync(coverage, io->coverage, 8 * (size_t)n, cudaMemcpyDeviceToHost, s), "D2H coverage");   \
    if (variance_inv) rc |= check_cuda(cudaMemcpyAsync(variance_inv, io->variance_inv, 8 * (size_t)n, cudaMemcpyDeviceToHost, s), "D2H variance"); \
    if (flags) rc |= check_cuda(cudaMemcpyAsync(flags, io->flags, 4 * (size_t)n, cudaMemcpyDeviceToHost, s), "D2H flags");               \
    if (sim_steps) rc |= check_cuda(cudaMemcpyAsync(sim_steps, io->sim_steps, 4 * (size_t)n, cudaMemcpyDeviceToHost, s), "D2H sim_steps"); \
    if (rc) return CLOTHB200_ERR_CUDA;                                                                                                   \
    return check_cuda(cudaStreamSynchronize(s), "cudaStreamSynchronize");

int clothb200_step_host_phys_f32(const ClothB200Params *p, int mode, int n, const double *actions, const ClothB200Step *io, int initialize,
                                 float *obs, double *reward, int32_t *done, double *coverage, double *variance_inv, int32_t *flags,
                                 int32_t *sim_steps, const ClothB200Physics *physics, void *st) {
    STEP_HOST_BODY(f32, float)
}
int clothb200_step_host_phys_f64(const ClothB200Params *p, int mode, int n, const double *actions, const ClothB200Step *io, int initialize,
                                 double *obs, double *reward, int32_t *done, double *coverage, double *variance_inv, int32_t *flags,
                                 int32_t *sim_steps, const ClothB200Physics *physics, void *st) {
    STEP_HOST_BODY(f64, double)
}
int clothb200_step_host_f32(const ClothB200Params *p, int mode, int n, const double *actions, const ClothB200Step *io, int initialize,
                            float *obs, double *reward, int32_t *done, double *coverage, double *variance_inv, int32_t *flags,
                            int32_t *sim_steps, void *st) {
    return clothb200_step_host_phys_f32(p, mode, n, actions, io, initialize, obs, reward, done, coverage, variance_inv, flags, sim_steps, nullptr, st);
}
int clothb200_step_host_f64(const ClothB200Params *p, int mode, int n, const double *actions, const ClothB200Step *io, int initialize,
                            double *obs, double *reward, int32_t *done, double *coverage, double *variance_inv, int32_t *flags,
                            int32_t *sim_steps, void *st) {
    return clothb200_step_host_phys_f64(p, mode, n, actions, io, initialize, obs, reward, done, coverage, variance_inv, flags, sim_steps, nullptr, st);
}

static int time_kernel(void (*launch)(int, float *, cudaStream_t), int iters, cudaStream_t s, float *ms_out) {
    float *sink = nullptr;
    int rc = check_cuda(cudaMalloc((void **)&sink, 64), "cudaMalloc(sink)");
    if (rc) return rc;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    launch(iters / 8 + 1, sink, s);   // warm-up
    cudaEventRecord(e0, s);
    launch(iters, sink, s);
    cudaEventRecord(e1, s);
    rc = check_cuda(cudaEventSynchronize(e1), "microbenchmark");
    cudaEventElapsedTime(ms_out, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(sink);
    return rc;
}
static int g_bench_blocks = 148 * 2;
static void launch_smem(int iters, float *sink, cudaStream_t s) { smem_bw_kernel<<<g_bench_blocks, 1024, 0, s>>>(iters, sink); g_launch_count++; }
static void launch_fma(int iters, float *sink, cudaStream_t s) { fp32_fma_kernel<<<g_bench_blocks, 1024, 0, s>>>(iters, sink); g_launch_count++; }

int clothb200_bench_smem_bandwidth(int iters, double *gb_per_s, void *st) {
    if (!gb_per_s || iters <= 0) return CLOTHB200_ERR_ARG;
    int sms = 148;
    clothb200_device_info(-1, &sms, nullptr, nullptr, nullptr);
    g_bench_blocks = sms * 2;
    float ms = 0.f;
    int rc = time_kernel(launch_smem, iters, (cudaStream_t)st, &ms);
    if (rc) return rc;
    const double bytes = (double)g_bench_blocks * 1024.0 * 8.0 * 16.0 * iters;
    *gb_per_s = bytes / (ms * 1e-3) / 1e9;
    return CLOTHB200_OK;
}
int clothb200_bench_fp32_flops(int iters, double *tflop_per_s, void *st) {
    if (!tflop_per_s || iters <= 0) return CLOTHB200_ERR_ARG;
    int sms = 148;
    clothb200_device_info(-1, &sms, nullptr, nullptr, nullptr);
    g_bench_blocks = sms * 2;
    float ms = 0.f;
    int rc = time_kernel(launch_fma, iters, (cudaStream_t)st, &ms);
    if (rc) return rc;
    const double flops = (double)g_bench_blocks * 1024.0 * 16.0 * 8.0 * 2.0 * iters;
    *tflop_per_s = flops / (ms * 1e-3) / 1e12;
    return CLOTHB200_OK;
}

}  // extern "C"
