// cloth_device.cuh - device-side building blocks of the batched cloth step (sm_100a).
//
// One CTA owns one cloth.  pos/prev of all N points live in shared memory for the whole action
// (staged in and out with TMA bulk copies); every phase of Cloth.update() (cloth.pyx:169-214) runs
// there.  REFERENCE_ORDER mode reproduces the sequential Gauss-Seidel semantics of the Cython loops
// exactly (bit-exact in the double instantiation) while still exposing parallelism:
//   - Hooke (cloth.pyx:221-237) is a Jacobi phase: per-point gather of its <=12 springs in global
//     spring order gives the same per-point summation order as the reference's scatter loop.
//   - self-collision (cloth.pyx:313-343) is sequential only inside one hash bucket.  All points are
//     first evaluated against the post-Verlet snapshot; a bucket whose snapshot has no hit is final;
//     in a bucket with hits the first hit point (lowest index) takes its snapshot correction and only
//     the points after it are replayed in index order by one warp (lanes = candidates).
//   - the 10 % stretch limit (cloth.pyx:258-296) modifies a spring's end points only if it is longer
//     than 1.1 x rest.  All springs are tested against the snapshot in parallel; flagged springs go
//     into a bitmask priority queue ordered by spring index and are replayed in order by one warp;
//     every applied correction re-tests the <=22 later springs incident to the moved points, so a
//     spring is processed exactly when the sequential loop would have found it stretched.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/clothb200.h"

namespace clothb200 {

// ------------------------------------------------------------------------------------------------
// scalar helpers
// ------------------------------------------------------------------------------------------------
template <typename T> struct V4;
template <> struct V4<float> { typedef float4 type; };
template <> struct V4<double> { typedef double4 type; };

__device__ __forceinline__ float4 mk4(float x, float y, float z, float w) { return make_float4(x, y, z, w); }
__device__ __forceinline__ double4 mk4(double x, double y, double z, double w) { return make_double4(x, y, z, w); }

__device__ __forceinline__ float sqrt_t(float x) { return sqrtf(x); }
__device__ __forceinline__ double sqrt_t(double x) { return sqrt(x); }
__device__ __forceinline__ float floor_t(float x) { return floorf(x); }
__device__ __forceinline__ double floor_t(double x) { return floor(x); }

// cloth.pyx:17-18 fastnorm: sqrt(x*x + y*y + z*z), left-to-right
template <typename T> __device__ __forceinline__ T norm3(T x, T y, T z) { return sqrt_t(x * x + y * y + z * z); }

// The reward terms and the grip test in double, one rounding per operator as in the oracle (-ffp-contract=off): the
// f32 units allow FMA contraction, which would also fuse these double products and sums; ptxas never fuses the _rn
// intrinsics.  (-fmad=false makes the f64 units round every operator anyway: there these compile as before.)
// dx*dx + dy*dy
__device__ __forceinline__ double dist2_rn(double dx, double dy) { return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)); }
// ax*by - ay*bx: the monotone chain's turn test and the shoelace term
__device__ __forceinline__ double cross_rn(double ax, double ay, double bx, double by) { return __dsub_rn(__dmul_rn(ax, by), __dmul_rn(ay, bx)); }

template <typename T> struct DevParams {
    int W, H, N;
    int table_size, table_shift; // hash table: power of two >= 1.6 N
    int ev_words;                // ceil(6N/32) words of the stretched-spring queue
    int n_levels;                // grab_top z levels (gripper.pyx:31-41)
    int max_actions;
    T mg;                        // mass*gravity (cloth.pyx:179)
    T kk_struct, kk_bend;        // ks*1.0, ks*0.2 (cloth.pyx:225-232)
    T dsdm, damp;                // (dt*dt)/mass, 1-damping/100 (cloth.pyx:240-241)
    T cell_w, cell_h, cell_t;    // 3dx, 3dy, max (cloth.pyx:308-310)
    T inv_cell_w, inv_cell_h, inv_cell_t;
    int cell_pow2;               // cell sizes are powers of two: x/w == x*(1/w) exactly
    T thresh, thresh2;           // 2*thickness (cloth.pyx:317) and its square
    T sim_steps;                 // simulation_steps as scalar (cloth.pyx:338-340)
    T min_z, fric1, surf_off;    // minimum_z, 1-plane_friction, 1e-4 (cloth.pyx:345-370)
    T tear_thresh;
    T rest_k[6];                 // rest lengths of the flat grid per spring kind k (used when rest == NULL)
    T kkrest_k[6];               // ks * kc * rest_k[k]: the constant of the f32 Hooke form kk - kkrest / l
    T limit_c2_k[6];             // min(rest_k * 1.1, rest_k * tear_thresh)^2: squared length beyond which a spring needs the limit pass
    double grip_radius, thickness, gripper_height;
    double iu, iur, igr, ir;     // iters_up, iters_up_rest, iters_grip_rest, iters_rest
    // static wavefront schedule of _limit_spring_changes: springs grouped by dependency level (level(s) = 1 + max level
    // of the earlier springs that share a point with s), sweep_lw entries per level: a | q << 12 | k << 24, ~0u = empty
    const uint32_t *sweep_tbl;
    int sweep_levels, sweep_lw, sweep_thresh;
    int relax_iters;             // coloured mode: limit passes per update (>= 1; the reference does exactly one)
    int reward_abs;              // reward_type 'coverage': rew += coverage, not its delta (cloth_env.py:657-659)
    int force_grab;              // cfg env.force_grab: grow the grip radius by 0.02 until something is gripped (cloth_env.py:434-444)
};

// The material constants of one cloth: what density, ks, damping, plane_friction, tear_thresh and gravity become.
// DevParams carries the batch's; the per-environment step kernel reads one row of these per cloth instead, through the
// read-only path.  The fields Hooke/Verlet reads every substep come first (44 of the 80 bytes of an f32 row; rows are not
// padded to 64 bytes, so these span two or three 32-byte sectors, loaded once per CTA into L1).
template <typename T> struct DevMaterial {
    T mg, kk_struct, kk_bend, dsdm, damp;
    T kkrest_k[6];
    T fric1, tear_thresh;
    T limit_c2_k[6];
    int valid;                   // 0: a non-finite value or density <= 0 (the cloth is not stepped, BADSTATE)
};

// cloth.pyx:175-186, 240-241: the constants in double as the reference derives them, then rounded to T once; the
// per-kind products are formed in T from those.  The one place this arithmetic lives (make_dev_params and the
// per-environment rows both call it), so the same material gives the same bits either way.
template <typename T>
__host__ __device__ inline void derive_material(double density, double ks, double damping, double plane_friction, double tear_thresh,
                                                double gravity, int W, int H, double frames_per_sec, int simulation_steps,
                                                const T *rest_k, DevMaterial<T> &m) {
    const double mass = density / W / H;
    const double delta_t = 1.0 / frames_per_sec / simulation_steps;
    m.mg = (T)(mass * gravity);
    m.kk_struct = (T)(ks * 1.0);
    m.kk_bend = (T)(ks * 0.2);
    m.dsdm = (T)((delta_t * delta_t) / mass);
    m.damp = (T)(1.0 - damping / 100.0);
    m.fric1 = (T)(1. - plane_friction);
    m.tear_thresh = (T)tear_thresh;
    for (int k = 0; k < 6; k++) {
        m.kkrest_k[k] = (k >= 4 ? m.kk_bend : m.kk_struct) * rest_k[k];
        const T a = rest_k[k] * T(1.1), b = rest_k[k] * m.tear_thresh, c = a < b ? a : b;    // ClothCTA::limit_c
        m.limit_c2_k[k] = c * c;
    }
    m.valid = isfinite(density) && isfinite(ks) && isfinite(damping) && isfinite(plane_friction) && isfinite(tear_thresh) &&
              isfinite(gravity) && density > 0;
}

template <typename T> struct StepArgs {
    T *pos, *prev;
    const T *rest;
    long long rest_env_stride;
    const ClothB200Plan *plans;  // NULL => plain update mode (n_updates x Cloth.update())
    const double *grab_xy;       // grab-only mode (clothb200_grab_top_*)
    double grab_radius;
    int n_updates;
    int mode;                    // 0 step, 1 update_n, 2 grab only, 3 measure only
    int initialize;
    int n_env;
    int32_t *flags, *sim_steps, *n_grabbed;
    uint32_t *grab_mask;
    double *coverage, *variance_inv;
    T *obs;
    double *prev_coverage;
    int32_t *num_steps, *num_sim_steps;
    double *reward;
    int32_t *done;
    const double *iters_up_env;
    const int32_t *env_order;
    long long *prof;             // optional [n_env][16] cycle / event counters (debug)
    float *cost;                 // optional [n_env] in/out: SM cycles per substep of the env's last step
    int debug_flags;             // CLOTHB200_DEBUG env var: 1 = no warp-role rotation
    // time-sliced mode (KMODE_STEP only, slice > 0): a persistent grid takes (item = position in the launch order)
    // tickets from a queue, runs `slice` substeps of that cloth, stores it and re-queues it behind everything else
    int slice, qcap;
    int yield_slack;             // a cloth keeps its slot unless the waiting one has more than this many substeps more left
    int endgame_slices, endgame_shift;   // the last endgame_slices slices of an action run in slices of slice >> endgame_shift
    unsigned long long *queue;   // [qcap] (ticket + 1) << 32 | substeps left << 16 | item
    const unsigned long long *sorted_keys;   // plan_work_kernel's keys after the sort (substeps per item)
    int *qctl;                   // [0] tickets taken, [1] tickets issued, [2] cloths finished
    int *progress, *ngrab_s;     // [qcap] per item: substeps done, number of gripped points
    float *cycles_s;             // [qcap] per item: SM cycles spent so far
    const DevMaterial<T> *mat;   // [n_env] by launch position (item): per-environment material (the PHYS kernels only)
};

enum { KMODE_STEP = 0, KMODE_UPDATE = 1, KMODE_GRAB = 2, KMODE_MEASURE = 3 };

// ------------------------------------------------------------------------------------------------
// TMA bulk copy + mbarrier (PTX).  cp.async.bulk needs 16-byte aligned addresses and sizes.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_wait() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// the stored bytes are complete in global memory (not just read out of shared memory) when this returns
__device__ __forceinline__ void bulk_commit_wait_all() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void fence_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// ---- work queue of the time-sliced step kernel (one thread per CTA calls these) ----
// A ring of qcap slots; ticket t lives in slot t % qcap, tagged t + 1 (0 = empty).  At most qcap cloths are alive,
// but a slot can still be wanted by ticket t + qcap while the holder of ticket t has not read it yet (the other
// cloths can be re-queued in the meantime), so the reader empties the slot and the writer waits for an empty slot.
// Every wait is for an event of a strictly older ticket held by a running CTA: no cycle.
template <typename A_t> __device__ __forceinline__ int queue_pop(const A_t &A) {
    const int t = atomicAdd(&A.qctl[0], 1);
    volatile unsigned long long *slot = A.queue + (t % A.qcap);
    volatile int *done = A.qctl + 2;
    unsigned ns = 100u;
    for (;;) {
        const unsigned long long v = *slot;
        if ((int)(v >> 32) == t + 1) {
            __threadfence();
            *slot = 0ull;
            return (int)(v & 0xffffull);
        }
        if (*done >= A.qcap) return -1;
        __nanosleep(ns);                      // idle slots at the end of a launch: back off, the SM belongs to the working cloths
        if (ns < 4000u) ns += ns;
    }
}
template <typename A_t> __device__ __forceinline__ void queue_push(const A_t &A, int item, int remaining) {
    __threadfence();
    const int t = atomicAdd(&A.qctl[1], 1);
    const unsigned rem = (unsigned)(remaining > 65535 ? 65535 : remaining);
    volatile unsigned long long *slot = A.queue + (t % A.qcap);
    while (*slot != 0ull) __nanosleep(100);
    atomicExch(A.queue + (t % A.qcap), ((unsigned long long)(unsigned)(t + 1) << 32) | (rem << 16) | (unsigned)item);
}
// substeps left of the cloth at the head of the queue (0 if nothing is waiting); a racy peek, only a heuristic
template <typename A_t> __device__ __forceinline__ int queue_head_remaining(const A_t &A) {
    const int h = *(volatile int *)&A.qctl[0];
    const unsigned long long v = *(volatile unsigned long long *)(A.queue + (h % A.qcap));
    return (int)(v >> 32) == h + 1 ? (int)((v >> 16) & 0xffffull) : 0;
}

// ------------------------------------------------------------------------------------------------
// The per-CTA cloth.  NT threads; WC = compile-time grid width (0 = runtime).
// ------------------------------------------------------------------------------------------------
// slot classes of the collision work list (ClothCTA::collide_buckets): SLOT | buckets per warp << 8 | ceil(256 / SLOT) << 16
static __device__ __constant__ uint32_t kSlotClass[11] = {
    64u | 1u << 8 | 4u << 16,  32u | 1u << 8 | 8u << 16,  16u | 2u << 8 | 16u << 16, 10u | 3u << 8 | 26u << 16,
    8u | 4u << 8 | 32u << 16,  7u | 4u << 8 | 37u << 16,  6u | 5u << 8 | 43u << 16,  5u | 6u << 8 | 52u << 16,
    4u | 8u << 8 | 64u << 16,  3u | 10u << 8 | 86u << 16, 2u | 16u << 8 | 128u << 16};

#define CLOTH_KEY_EMPTY 0x7fffffff
#define CLOTH_FIRST_NONE 0x7ffffffe

template <typename T, int NT, int WC, bool REST_TABLE, bool COLOURED = false, bool PHYS = false> struct ClothCTA {
    typedef typename V4<T>::type P4;
    static constexpr int NWARPS = NT / 32;
    // f32 production math (rsqrt / squared-distance forms of the reference's expressions); the f64 build evaluates the
    // reference's expressions themselves.  CLOTHB200_F32_REFERENCE_FORMS builds the float kernels that way too (study
    // variant libclothb200_f32ieee.so: IEEE div/sqrt, no flush-to-zero - gym_cloth_b200/build.py, scripts/f32_drift.py).
#ifdef CLOTHB200_F32_REFERENCE_FORMS
    static constexpr bool FAST = false;
#else
    static constexpr bool FAST = (sizeof(T) == 4);
#endif

    const DevParams<T> &P;
    const int W, H, N;
    const int tid, lane, warp;
    P4 *pos, *prev;          // [N]
    int *tkey;               // [TS]   hash keys, later the bucket's first hit point
    uint32_t *tinfo;         // [TS]   count | (end offset << 16)
    uint16_t *pslot;         // [N]    bucket slot of each point (bit 15: this point allocates the bucket)
    uint16_t *lstA, *lstB;   // [N]    bucket member lists: unordered / index-ordered; lstA later = fix-up work list
    int *cls;                // [2*NCLS] work-list class counters of the reference-order collision (see NCLS)
    uint32_t *ev;            // [ev_words] stretched-spring queue
    int *misc;               // [16] counters/flags: 0 total, 1 nwork, 2 tear, 3 bad, 4.. scratch
    float2 *kc;              // [8] per spring kind: {rest*1.1, (rest*tear_thresh)^2} (f32, constant rest lengths)
    const T *rest;           // rest table of this env (REST_TABLE)
    const DevMaterial<T> *mat;   // material row of this env (PHYS), read through the read-only path where a phase uses it
    int rot;                 // blockIdx-derived rotation of the warp roles (spreads serial phases over the 4 SM sub-partitions)
    long long *pacc;         // [16] smem: thread 0's cycles per phase + event counters when profiling
    long long plast;
    bool prof_on;

    __device__ ClothCTA(const DevParams<T> &P_, unsigned char *smem, const T *rest_, const DevMaterial<T> *mat_ = nullptr)
        : P(P_), W(WC ? WC : P_.W), H(WC ? WC : P_.H), N(WC ? WC * WC : P_.N), tid(threadIdx.x), lane(threadIdx.x & 31),
          warp(threadIdx.x >> 5), rest(rest_), mat(mat_), rot((int)blockIdx.x), plast(0), prof_on(false) {
        size_t o = 0;
        pos = reinterpret_cast<P4 *>(smem + o); o += sizeof(P4) * (size_t)N;
        prev = reinterpret_cast<P4 *>(smem + o); o += sizeof(P4) * (size_t)N;
        tkey = reinterpret_cast<int *>(smem + o); o += 4 * (size_t)P.table_size;
        tinfo = reinterpret_cast<uint32_t *>(smem + o); o += 4 * (size_t)P.table_size;
        misc = reinterpret_cast<int *>(smem + o); o += 4 * 16;
        pacc = reinterpret_cast<long long *>(smem + o); o += 8 * 16;
        kc = reinterpret_cast<float2 *>(smem + o); o += 8 * 8;
        // the stretched-spring queue `ev` shares its storage with `pslot`: pslot is dead once the collision replay
        // starts (which zeroes the area), ev lives from the limit snapshot to the end of the update
        const size_t ps_bytes = 2 * (size_t)((N + 7) & ~7), ev_bytes = 4 * (size_t)((P.ev_words + 3) & ~3);
        pslot = reinterpret_cast<uint16_t *>(smem + o);
        ev = reinterpret_cast<uint32_t *>(smem + o); o += ps_bytes > ev_bytes ? ps_bytes : ev_bytes;
        lstA = reinterpret_cast<uint16_t *>(smem + o); o += 2 * (size_t)((N + 7) & ~7);
        cls = reinterpret_cast<int *>(smem + o); o += cls_bytes();
        lstB = reinterpret_cast<uint16_t *>(smem + o); o += 2 * (size_t)((N + 7) & ~7);
        if (!cls_bytes()) cls = reinterpret_cast<int *>(lstB);
    }
    // The class counters sit at the head of lstB when the ordered scatter leaves lstB idle (and the coloured mode has
    // none).  The unordered scatter writes the index-ordered member lists into lstB while other warps may still read
    // the counters, and lstB is smaller than the counters on grids of fewer than 136 points: there they get their own.
    static __host__ __device__ constexpr size_t cls_bytes() { return (ORDERED || COLOURED) ? 0 : 8 * (size_t)NCLS; }
    static __host__ __device__ size_t smem_bytes(int N, int table_size, int ev_words) {
        const size_t ps_bytes = 2 * (size_t)((N + 7) & ~7), ev_bytes = 4 * (size_t)((ev_words + 3) & ~3);
        return sizeof(P4) * (size_t)N * 2 + 8 * (size_t)table_size + 64 + 128 + 64 + (ps_bytes > ev_bytes ? ps_bytes : ev_bytes) +
               2 * ps_bytes + cls_bytes() + 16 /* mbarrier */;
    }

    __device__ __forceinline__ void sync() {
        if (NT == 32) __syncwarp(); else __syncthreads();
    }

    // ---- spring topology (cloth.pyx:135-146).  Spring slot s = q*6 + k: k-th spring created by point q. ----
    // All helpers are branch-free (no jump tables): they sit on the critical path of the serial replays.
    // offset from q back to ptA for kind k: {W, 1, W+1, W-1, 2W, 2} packed 10 bits each
    __device__ __forceinline__ unsigned long long koff_pack() const {
        return (unsigned long long)W | (1ull << 10) | ((unsigned long long)(W + 1) << 20) | ((unsigned long long)(W - 1) << 30) |
               ((unsigned long long)(2 * W) << 40) | (2ull << 50);
    }
    __device__ __forceinline__ int koff(int k) const { return (int)((koff_pack() >> (10 * k)) & 1023ull); }
    // bit k set <=> point (r,c) creates spring kind k
    __device__ __forceinline__ unsigned vmask(int r, int c) const {
        const unsigned r0 = r > 0, c0 = c > 0, cw = c + 1 < W, r1 = r > 1, c1 = c > 1;
        return r0 | (c0 << 1) | ((r0 & c0) << 2) | ((r0 & cw) << 3) | (r1 << 4) | (c1 << 5);
    }
    __device__ __forceinline__ bool kvalid(int r, int c, int k) const { return (vmask(r, c) >> k) & 1u; }
    // per-kind constant selected with compares (k is usually warp-uniform); avoids register-indexed constant loads
    __device__ __forceinline__ T sel6(const T *v, int k) const {
        T lo = k == 0 ? v[0] : (k == 1 ? v[1] : v[2]);
        T hi = k == 3 ? v[3] : (k == 4 ? v[4] : v[5]);
        return k < 3 ? lo : hi;
    }
    // ---- material constants: the launch's (P), or this cloth's row in the per-environment variant ----
    __device__ __forceinline__ T mg() const { if constexpr (PHYS) return __ldg(&mat->mg); else return P.mg; }
    __device__ __forceinline__ T kk_struct() const { if constexpr (PHYS) return __ldg(&mat->kk_struct); else return P.kk_struct; }
    __device__ __forceinline__ T kk_bend() const { if constexpr (PHYS) return __ldg(&mat->kk_bend); else return P.kk_bend; }
    __device__ __forceinline__ T dsdm() const { if constexpr (PHYS) return __ldg(&mat->dsdm); else return P.dsdm; }
    __device__ __forceinline__ T damp() const { if constexpr (PHYS) return __ldg(&mat->damp); else return P.damp; }
    __device__ __forceinline__ T fric1() const { if constexpr (PHYS) return __ldg(&mat->fric1); else return P.fric1; }
    __device__ __forceinline__ T tear_thresh() const { if constexpr (PHYS) return __ldg(&mat->tear_thresh); else return P.tear_thresh; }
    __device__ __forceinline__ T kkrest_k(int k) const { if constexpr (PHYS) return __ldg(&mat->kkrest_k[k]); else return P.kkrest_k[k]; }
    __device__ __forceinline__ T limit_c2_k(int k) const { if constexpr (PHYS) return __ldg(&mat->limit_c2_k[k]); else return P.limit_c2_k[k]; }

    __device__ __forceinline__ T rest_of(int q, int k) const {
        if (REST_TABLE) return __ldg(rest + q * 6 + k);
        return sel6(P.rest_k, k);
    }
    // kk * rest of spring (q, k): a launch constant unless the cloth carries its own rest lengths
    __device__ __forceinline__ T kkrest_of(int q, int k, T kk) const {
        if (REST_TABLE || !FAST) return kk * rest_of(q, k);
        return kkrest_k(k);
    }
    __device__ __forceinline__ T kk_of(int k) const { return k >= 4 ? kk_bend() : kk_struct(); }

    // ---- distance predicates ----
    // f32 build: squared-distance forms (no sqrt).  f64 build: the reference's exact `fastnorm(...) <op> c`
    // decision; a squared-distance pre-filter with a 1e-15 relative guard band decides all but razor-edge
    // cases without the sqrt, the remaining ones evaluate the reference expression itself.
    // true <=> fastnorm(d) > c   (c = rest*1.1 or rest*tear_thresh, as the reference computes it)
    __device__ __forceinline__ bool longer_than(T d0, T d1, T d2, T c) const {
        const T q = d0 * d0 + d1 * d1 + d2 * d2;
        const T c2 = c * c;
        if (FAST) return q > c2;
        if (q > c2 * T(1.000000000000001)) return true;
        if (q < c2 * T(0.999999999999999)) return false;
        return sqrt_t(q) > c;
    }
    // true <=> fastnorm(d) <= thresh  (cloth.pyx:330)
    __device__ __forceinline__ bool within_thresh(T q) const {
        if (FAST) return q <= P.thresh2;
        if (q < P.thresh2 * T(0.999999999999999)) return true;
        if (q > P.thresh2 * T(1.000000000000001)) return false;
        return sqrt_t(q) <= P.thresh;
    }

    // ---- Hooke (cloth.pyx:221-237) gathered per point + Verlet (cloth.pyx:239-256) ----
    // One spring's contribution to point p, selected without branches so that the 12 neighbour loads and
    // the 12 independent force evaluations of a point can overlap.  SIGN=+1: p is ptA, -1: p is ptB.
    // Z_RN: fz -= fm*d2 as a rounded product and a rounded difference (see hooke_verlet)
    template <int SIGN, bool Z_RN = false>
    __device__ __forceinline__ void add_spring(bool valid, const P4 &Pa, const P4 &Pb, T kk, T rst, T kkrst, T &fx, T &fy, T &fz, int &bad) {
        const T d0 = Pb.x - Pa.x, d1 = Pb.y - Pa.y, d2 = Pb.z - Pa.z;
        const T q = d0 * d0 + d1 * d1 + d2 * d2;
        T fm;
        if (FAST) {
            // ks*kc*(l-rest)/l; a spring that does not exist gets coefficient 0, a zero-length one gives inf -> NaN
            // positions, which commit_and_hash() reports as BADSTATE (the reference raises ZeroDivisionError here)
            fm = valid ? kk - kkrst * rsqrtf((float)q) : T(0);
            if (SIGN > 0) { fx += fm * d0; fy += fm * d1; fz += fm * d2; }
            else if constexpr (Z_RN) { fx -= fm * d0; fy -= fm * d1; fz = __fsub_rn(fz, __fmul_rn(fm, d2)); }
            else { fx -= fm * d0; fy -= fm * d1; fz -= fm * d2; }
            return;
        }
        {
            const T l = sqrt_t(q);                               // fastnorm
            fm = kk * (l - rst) / l;
        }
        bad |= (valid && q == T(0)) ? 1 : 0;                     // reference: ZeroDivisionError
        const T f0 = fm * d0, f1 = fm * d1, f2 = fm * d2;
        if (SIGN > 0) { fx = valid ? fx + f0 : fx; fy = valid ? fy + f1 : fy; fz = valid ? fz + f2 : fz; }
        else { fx = valid ? fx + (-f0) : fx; fy = valid ? fy + (-f1) : fy; fz = valid ? fz + (-f2) : fz; }
    }

    // The new position is parked in prev[p].xyz (prev is private to the owner thread); commit_and_hash()
    // swaps it in after the barrier, when no thread reads old positions any more.
    __device__ __forceinline__ void hooke_verlet() {
        int bad = 0;
        if (!COLOURED && tid < 2 * NCLS) size_count()[tid] = 0;     // work-list size classes of this substep
        for (int p = tid; p < N; p += NT) {
            const P4 Pp = pos[p];
            if (Pp.w != T(0)) continue;  // pinned: Verlet skips it, its force is never used
            const int r = p / W, c = p - r * W;
            const bool v0 = r > 0, v1 = c > 0, v2 = v0 && v1, v3 = v0 && (c + 1 < W), v4 = r > 1, v5 = c > 1;
            const bool u0 = c + 1 < W, u1 = c + 2 < W, dn = r + 1 < H, u2 = dn && v1, u3 = dn, u4 = dn && u0, u5 = r + 2 < H;
            // all twelve neighbours first (invalid ones alias p itself: in range, result discarded)
            const P4 A0 = pos[v0 ? p - W : p], A1 = pos[v1 ? p - 1 : p], A2 = pos[v2 ? p - W - 1 : p];
            const P4 A3 = pos[v3 ? p - W + 1 : p], A4 = pos[v4 ? p - 2 * W : p], A5 = pos[v5 ? p - 2 : p];
            const P4 B0 = pos[u0 ? p + 1 : p], B1 = pos[u1 ? p + 2 : p], B2 = pos[u2 ? p + W - 1 : p];
            const P4 B3 = pos[u3 ? p + W : p], B4 = pos[u4 ? p + W + 1 : p], B5 = pos[u5 ? p + 2 * W : p];
            const P4 Q = prev[p];
            // _reset_gravity: f = 0 then f += (0,0,mg)
            T fx = T(0) + T(0), fy = T(0) + T(0), fz = T(0) + mg();
            // springs created by p (p is ptB, ptB.add_force(-F)), creation order k = 0..5.  In the f32 kernels with the
            // batch's material ptxas keeps the first spring's z product apart from mg (FMUL + FADD, not FFMA); with mg
            // read from the cloth's row it would fuse them, so the per-environment variant rounds both explicitly: the
            // same material gives the same bits in either kernel
            add_spring<-1, PHYS && FAST>(v0, A0, Pp, kk_struct(), rest_of(p, 0), kkrest_of(p, 0, kk_struct()), fx, fy, fz, bad);
            add_spring<-1>(v1, A1, Pp, kk_struct(), rest_of(p, 1), kkrest_of(p, 1, kk_struct()), fx, fy, fz, bad);
            add_spring<-1>(v2, A2, Pp, kk_struct(), rest_of(p, 2), kkrest_of(p, 2, kk_struct()), fx, fy, fz, bad);
            add_spring<-1>(v3, A3, Pp, kk_struct(), rest_of(p, 3), kkrest_of(p, 3, kk_struct()), fx, fy, fz, bad);
            add_spring<-1>(v4, A4, Pp, kk_bend(), rest_of(p, 4), kkrest_of(p, 4, kk_bend()), fx, fy, fz, bad);
            add_spring<-1>(v5, A5, Pp, kk_bend(), rest_of(p, 5), kkrest_of(p, 5, kk_bend()), fx, fy, fz, bad);
            // springs created by later points in which p is ptA, in creation order:
            // q = p+1 (k=1), p+2 (k=5), p+W-1 (k=3), p+W (k=0), p+W+1 (k=2), p+2W (k=4)
            add_spring<1>(u0, Pp, B0, kk_struct(), rest_of(u0 ? p + 1 : p, 1), kkrest_of(u0 ? p + 1 : p, 1, kk_struct()), fx, fy, fz, bad);
            add_spring<1>(u1, Pp, B1, kk_bend(), rest_of(u1 ? p + 2 : p, 5), kkrest_of(u1 ? p + 2 : p, 5, kk_bend()), fx, fy, fz, bad);
            add_spring<1>(u2, Pp, B2, kk_struct(), rest_of(u2 ? p + W - 1 : p, 3), kkrest_of(u2 ? p + W - 1 : p, 3, kk_struct()), fx, fy, fz, bad);
            add_spring<1>(u3, Pp, B3, kk_struct(), rest_of(u3 ? p + W : p, 0), kkrest_of(u3 ? p + W : p, 0, kk_struct()), fx, fy, fz, bad);
            add_spring<1>(u4, Pp, B4, kk_struct(), rest_of(u4 ? p + W + 1 : p, 2), kkrest_of(u4 ? p + W + 1 : p, 2, kk_struct()), fx, fy, fz, bad);
            add_spring<1>(u5, Pp, B5, kk_bend(), rest_of(u5 ? p + 2 * W : p, 4), kkrest_of(u5 ? p + 2 * W : p, 4, kk_bend()), fx, fy, fz, bad);
            // Verlet: new = x + damp*(x-px) + f*dsdm
            T nx = Pp.x + (damp() * (Pp.x - Q.x)) + (fx * dsdm());
            T ny = Pp.y + (damp() * (Pp.y - Q.y)) + (fy * dsdm());
            T nz = Pp.z + (damp() * (Pp.z - Q.z)) + (fz * dsdm());
            prev[p] = mk4(nx, ny, nz, Q.w);
        }
        if (bad) misc[3] = 1;
    }

    // ---- commit Verlet + build_spatial_map pass 1 (cloth.pyx:298-311): find/insert bucket, count ----
    __device__ __forceinline__ int cell(T v, T w, T inv_w) {
        // floor(v / w); when w is a power of two the product with 1/w is the same number
        T f = floor_t(P.cell_pow2 ? v * inv_w : v / w);
        if (!(f > T(-1048576) && f < T(1048576))) { misc[3] = 1; f = T(0); }  // NaN/huge: reference raises
        return (int)f;
    }
    // Ordered scatter (reference-order mode, compile-time grids of <= 1023 points run by 4 warps): the points are dealt
    // to the warps in contiguous index chunks, pass 1 counts per (bucket, warp) in the four bytes of tinfo[slot], pass 2
    // turns the counts into one list cursor per warp, and in pass 3 every warp appends its chunk row by row in lane
    // order - so every bucket list comes out in point-index order (the dict value order of cloth.pyx:301-305) and
    // nothing has to be ranked or permuted afterwards.
    static constexpr int CHUNK = (((WC * WC + NWARPS - 1) / NWARPS) + 31) & ~31;
    static constexpr bool ORDERED = !COLOURED && WC != 0 && NWARPS == 4 && WC * WC <= 1023 && CHUNK <= 255;
    static constexpr int HASH_ROWS = ORDERED ? CHUNK / 32 : 0;
    __device__ __forceinline__ void commit_and_hash() {
        const int nrows = ORDERED ? HASH_ROWS : (N + NT - 1) / NT;
        for (int i = 0; i < nrows; i++) {
            const int p = ORDERED ? warp * CHUNK + 32 * i + lane : tid + i * NT;
            if (p >= N) continue;
            P4 Pp = pos[p];
            if (Pp.w == T(0)) {
                const P4 Nw = prev[p];
                prev[p] = mk4(Pp.x, Pp.y, Pp.z, Nw.w);
                Pp = mk4(Nw.x, Nw.y, Nw.z, T(0));
                pos[p] = Pp;
            }
            const int key = 961 * cell(Pp.x, P.cell_w, P.inv_cell_w) + 31 * cell(Pp.y, P.cell_h, P.inv_cell_h) +
                            cell(Pp.z, P.cell_t, P.inv_cell_t);
            uint32_t slot = ((uint32_t)key * 2654435761u) >> P.table_shift;
            const uint32_t msk = (uint32_t)P.table_size - 1;
            for (int probes = 0;; probes++) {
                int old = *reinterpret_cast<volatile int *>(&tkey[slot]);
                if (old == key) break;
                if (old == CLOTH_KEY_EMPTY) {
                    old = atomicCAS(&tkey[slot], CLOTH_KEY_EMPTY, key);
                    if (old == CLOTH_KEY_EMPTY || old == key) break;
                }
                // more occupied cells than table slots (> 3x the cells of the flat cloth): not a cloth any more
                if (probes > (int)msk) { misc[3] = 1; break; }
                slot = (slot + 1) & msk;
            }
            const uint32_t r = atomicAdd(&tinfo[slot], ORDERED ? 1u << (8 * warp) : 1u);
            pslot[p] = (uint16_t)(slot | (r == 0 ? 0x8000u : 0u));
        }
    }
    // pass 2: the first arriver of each bucket reserves its range in the member list
    __device__ __forceinline__ void alloc_buckets() {
        for (int p = tid; p < N; p += NT) {
            const uint32_t s = pslot[p];
            if (s & 0x8000u) {
                const uint32_t slot = s & 0x7fffu;
                const uint32_t cnt = tinfo[slot];
                const uint32_t off = (uint32_t)atomicAdd(&misc[0], (int)cnt);
                tinfo[slot] = cnt | (off << 16);
                tkey[slot] = CLOTH_FIRST_NONE;
            }
        }
    }
    // pass 3: unordered scatter (high half of tinfo runs from off to off+cnt)
    __device__ __forceinline__ void scatter_members() {
        for (int p = tid; p < N; p += NT) {
            const uint32_t slot = pslot[p] & 0x7fffu;
            const uint32_t idx = atomicAdd(&tinfo[slot], 0x10000u) >> 16;
            lstA[idx] = (uint16_t)p;
        }
    }
    // pass 4: rank inside the bucket -> index-ordered list (the dict value order of cloth.pyx:301-305), fused with
    // the snapshot collision test: every pair is tested once, by its lower-index point, and only the lowest
    // point index that has a hit is kept per bucket (a hit makes every unpinned end of the pair a "hit point").
    __device__ __forceinline__ void order_and_snapshot() {
        for (int p = tid; p < N; p += NT) {
            const uint32_t slot = pslot[p] & 0x7fffu;
            const uint32_t info = tinfo[slot];
            const int cnt = info & 0xffffu, start = (int)(info >> 16) - cnt;
            int rk = 0;
            if (cnt > 1) {
                const P4 Pp = pos[p];
                int first = CLOTH_FIRST_NONE;
                // a hit makes every unpinned end of the pair a hit point; the pair is tested by its lower index
#define CLOTH_PAIR(q, Q)                                                                                    \
    {                                                                                                       \
        const T d0 = Pp.x - Q.x, d1 = Pp.y - Q.y, d2 = Pp.z - Q.z;                                          \
        const bool hit = q > p && within_thresh(d0 * d0 + d1 * d1 + d2 * d2);                               \
        const int h = Pp.w == T(0) ? p : (Q.w == T(0) ? q : CLOTH_FIRST_NONE);                              \
        first = (hit && h < first) ? h : first;                                                             \
        rk += (q < p) ? 1 : 0;                                                                              \
    }
                int j = 0;
                for (; j + 4 <= cnt; j += 4) {      // four candidates in flight: index and position loads overlap
                    const int q0 = lstA[start + j], q1 = lstA[start + j + 1], q2 = lstA[start + j + 2], q3 = lstA[start + j + 3];
                    const P4 Q0 = pos[q0], Q1 = pos[q1], Q2 = pos[q2], Q3 = pos[q3];
                    CLOTH_PAIR(q0, Q0) CLOTH_PAIR(q1, Q1) CLOTH_PAIR(q2, Q2) CLOTH_PAIR(q3, Q3)
                }
                for (; j < cnt; j++) {
                    const int q0 = lstA[start + j];
                    const P4 Q0 = pos[q0];
                    CLOTH_PAIR(q0, Q0)
                }
#undef CLOTH_PAIR
                if (first != CLOTH_FIRST_NONE) atomicMin(&tkey[slot], first);
            }
            lstB[start + rk] = (uint16_t)p;
        }
    }

    // ---- self_collide (cloth.pyx:313-343) ----
    // _handle_plane_collision (cloth.pyx:345-370)
    __device__ __forceinline__ void plane_point(int p) {
        const P4 Pp = pos[p];
        if (Pp.w != T(0) || Pp.z >= P.min_z) return;
        const P4 Q = prev[p];
        T t = (P.min_z - Q.z) * T(1.0);
        T tx = Q.x + t * T(-0.0), ty = Q.y + t * T(-0.0), tz = Q.z + t * T(-1.0);
        T gx = tx + P.surf_off * T(0.0), gy = ty + P.surf_off * T(0.0), gz = tz + P.surf_off * T(1.0);
        T cx = gx - Q.x, cy = gy - Q.y, cz = gz - Q.z;
        pos[p] = mk4(Q.x + cx * fric1(), Q.y + cy * fric1(), Q.z + cz * fric1(), Pp.w);
    }
    // ordered replay of one bucket by one warp: from the first hit point on (nothing before it moved, so its
    // own evaluation equals the snapshot), in index order; contributions are summed in candidate order.
    // A bucket of up to 32*K members replayed out of registers: lane l keeps members l, l+32, ... (bucket lists are
    // in point-index order, so walking register set 0, then 1, ... visits the subjects in the reference's order and
    // the per-set ballots add the contributions in candidate order).  Crumpled cloths pile 40-100 points into one
    // cell; the shared-memory path below costs them 4x more per member.
    template <int K> __device__ __forceinline__ void replay_bucket_regs(const uint16_t *lstB, const int start, const int cnt, const int j0) {
        int mine[K];
        P4 Pm[K];
        bool dirty[K];
#pragma unroll
        for (int k = 0; k < K; k++) {
            const int m = k * 32 + lane;
            mine[k] = m < cnt ? lstB[start + m] : 0;
            Pm[k] = mk4(T(0), T(0), T(0), T(1));
            if (m < cnt) Pm[k] = pos[mine[k]];
            dirty[k] = false;
        }
#pragma unroll
        for (int kj = 0; kj < K; kj++) {
            if (kj * 32 < cnt) {
                // pinned members never move and are skipped as subjects (cloth.pyx:314-315)
                unsigned todo = __ballot_sync(0xffffffffu, kj * 32 + lane < cnt && kj * 32 + lane >= j0 && Pm[kj].w == T(0));
                while (todo) {
                    const int jl = __ffs(todo) - 1;
                    todo &= todo - 1;
                    const T px = __shfl_sync(0xffffffffu, Pm[kj].x, jl), py = __shfl_sync(0xffffffffu, Pm[kj].y, jl),
                            pz = __shfl_sync(0xffffffffu, Pm[kj].z, jl);
                    T t0 = T(0), t1 = T(0), t2 = T(0);
                    int n = 0;
#pragma unroll
                    for (int k = 0; k < K; k++) {
                        if (k * 32 < cnt) {
                            const T d0 = px - Pm[k].x, d1 = py - Pm[k].y, d2 = pz - Pm[k].z;
                            const T qq = d0 * d0 + d1 * d1 + d2 * d2;
                            const bool hit = k * 32 + lane < cnt && !(k == kj && lane == jl) && within_thresh(qq);
                            unsigned m = __ballot_sync(0xffffffffu, hit);
                            if (m) {
                                T c0 = T(0), c1 = T(0), c2 = T(0);
                                if (hit) {
                                    if (qq == T(0)) misc[3] = 1;
                                    T factor;
                                    if (FAST) factor = P.thresh * rsqrtf((float)qq) - T(1);
                                    else { const T d = sqrt_t(qq); factor = (P.thresh - d) / d; }
                                    c0 = d0 * factor; c1 = d1 * factor; c2 = d2 * factor;
                                }
                                n += __popc(m);
                                while (m) {
                                    const int l = __ffs(m) - 1;
                                    m &= m - 1;
                                    t0 += __shfl_sync(0xffffffffu, c0, l);
                                    t1 += __shfl_sync(0xffffffffu, c1, l);
                                    t2 += __shfl_sync(0xffffffffu, c2, l);
                                }
                            }
                        }
                    }
                    if (n) {
                        const T nf = (T)n;
                        T cx, cy, cz;
                        if (FAST) { const T inv = T(1) / (nf * P.sim_steps); cx = t0 * inv; cy = t1 * inv; cz = t2 * inv; }
                        else { cx = t0 / nf / P.sim_steps; cy = t1 / nf / P.sim_steps; cz = t2 / nf / P.sim_steps; }
                        if (lane == jl) { Pm[kj] = mk4(px + cx, py + cy, pz + cz, Pm[kj].w); dirty[kj] = true; }
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < K; k++) {
            if (k * 32 + lane < cnt) {
                // plane collision (cloth.pyx:345-370) of my member, then one write-back
                if (Pm[k].w == T(0) && !(Pm[k].z >= P.min_z)) {
                    const P4 Q = prev[mine[k]];
                    T t = (P.min_z - Q.z) * T(1.0);
                    T tx = Q.x + t * T(-0.0), ty = Q.y + t * T(-0.0), tz = Q.z + t * T(-1.0);
                    T gx = tx + P.surf_off * T(0.0), gy = ty + P.surf_off * T(0.0), gz = tz + P.surf_off * T(1.0);
                    T ex = gx - Q.x, ey = gy - Q.y, ez = gz - Q.z;
                    Pm[k] = mk4(Q.x + ex * fric1(), Q.y + ey * fric1(), Q.z + ez * fric1(), Pm[k].w);
                    dirty[k] = true;
                }
                if (dirty[k]) pos[mine[k]] = Pm[k];
            }
        }
    }

    // ==================================================================================================
    // Reference-order self-collision, bucket-centric.  self_collide (cloth.pyx:313-343) is sequential only inside one
    // cell, so every cell with >= 2 points is one unit of work: its members sit in the lanes of a warp in point-index
    // order (the dict value order of cloth.pyx:301-305), subject j is broadcast with shuffles, all candidates are
    // tested at once, the hits are summed in candidate order and lane j takes the correction before subject j+1 is
    // looked at.  Cells are small (9 points on a flat cloth), so consecutive cells of the work list are packed side
    // by side into the 32 lanes ("segments") and advance in lock step.  No snapshot pre-test, no per-point gather.
    // ==================================================================================================
    // The work list is kept sorted by SLOT class, largest first: a bucket of n members is given a slot of SLOT >= n
    // lanes (n > 32: a "pile", its own path), and 32 / SLOT buckets of one class sit side by side in a warp, so a group
    // of the work list is just (class, i-th group of the class) - nothing is packed, scanned or negotiated at run time:
    //     class        0     1      2      3     4   5   6   7   8   9   10
    //     members    > 32  17-32  11-16  9-10    8   7   6   5   4   3    2
    //     SLOT         -    32     16     10     8   7   6   5   4   3    2
    //     per group    1     1      2      3     4   4   5   6   8  10   16
    // Class counters, fill counters and the per-class offsets live in `cls` (ordered scatter: the head of lstB, which
    // has no other use); hooke_verlet() zeroes them.  The list itself: behind them (ordered scatter) or in the key area
    // (dead after pass 1).
    static constexpr int NCLS = 34;                                  // ints reserved per counter block
    static constexpr int NSC = 11;                                   // slot classes
    __device__ __forceinline__ static int cls_of(uint32_t cnt) {
        return cnt > 32u ? 0 : (cnt > 16u ? 1 : (cnt > 10u ? 2 : (cnt > 8u ? 3 : 12 - (int)cnt)));
    }
    __device__ __forceinline__ static int cls_slot(int c) { return (int)(kSlotClass[c] & 255u); }
    __device__ __forceinline__ static int cls_cap(int c) { return (int)((kSlotClass[c] >> 8) & 255u); }
    __device__ __forceinline__ static int cls_mul(int c) { return (int)(kSlotClass[c] >> 16); }   // ceil(256 / SLOT): lane / SLOT = lane * mul >> 8
    __device__ __forceinline__ int *size_count() const { return cls; }
    __device__ __forceinline__ int *size_fill() const { return cls + NCLS; }
    __device__ __forceinline__ int *group_off() const { return size_fill() + NSC; }       // first group of each class
    __device__ __forceinline__ int *item_off() const { return size_fill() + 2 * NSC; }    // first work-list index of each class
    __device__ __forceinline__ uint16_t *worklist() const { return ORDERED ? lstB + 4 * NCLS : reinterpret_cast<uint16_t *>(tkey); }
    // member list of the buckets in point-index order
    __device__ __forceinline__ const uint16_t *ordered_list() const { return ORDERED ? lstA : lstB; }
    // tinfo[slot] after pass 2.  Unordered scatter: cnt | (end offset << 16), the high half running from start to end
    // during pass 3.  Ordered scatter: cnt | start << 10 | warp 0's cursor << 20, the cursors of warps 1-3 in tkey[slot].
    __device__ __forceinline__ void bucket_range(uint32_t info, int &cnt, int &start) const {
        if (ORDERED) { cnt = (int)(info & 1023u); start = (int)((info >> 10) & 1023u); }
        else { cnt = (int)(info & 0xffffu); start = (int)(info >> 16) - cnt; }
    }
    // pass 2: the first arriver of each bucket reserves its range and counts the bucket in its slot class
    __device__ __forceinline__ void alloc_buckets_ro() {
        int *szc = size_count();
        for (int p = tid; p < N; p += NT) {
            const uint32_t s = pslot[p];
            if (s & 0x8000u) {
                const uint32_t slot = s & 0x7fffu;
                const uint32_t info = tinfo[slot];
                uint32_t cnt = info;
                if (ORDERED) cnt = (info & 255u) + ((info >> 8) & 255u) + ((info >> 16) & 255u) + (info >> 24);
                const uint32_t off = (uint32_t)atomicAdd(&misc[0], (int)cnt);
                if (ORDERED) {
                    const uint32_t c1 = off + (info & 255u), c2 = c1 + ((info >> 8) & 255u), c3 = c2 + ((info >> 16) & 255u);
                    tinfo[slot] = cnt | (off << 10) | (off << 20);
                    tkey[slot] = (int)(c1 | (c2 << 10) | (c3 << 20));
                } else {
                    tinfo[slot] = cnt | (off << 16);
                }
                if (cnt > 1u) atomicAdd(&szc[cls_of(cnt)], 1);
            }
        }
    }
    // pass 3: scatter of the members; the first arriver also files the bucket in the class-sorted work list.
    // A point alone in its cell cannot collide and gets its plane collision right away.
    __device__ __forceinline__ void scatter_members_ro() {
        const unsigned FULL = 0xffffffffu;
        uint16_t *wl = worklist();
        int *szf = size_fill();
        // every warp scans the class counters itself (lane l <-> class l): first work-list index of each class; warp 0
        // also leaves the tables collide_buckets() reads: per class its first group and first item, and the group total
        int cls_off = lane < NSC ? size_count()[lane] : 0;
        {
            const int cnt_l = cls_off;
            const int cap_l = cls_cap(lane < NSC ? lane : 0);
            int incl = cnt_l, gincl = (cnt_l + cap_l - 1) / cap_l;
            const int g_l = gincl;
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) {
                const int v = __shfl_up_sync(FULL, incl, o), w = __shfl_up_sync(FULL, gincl, o);
                if (lane >= o) { incl += v; gincl += w; }
            }
            cls_off = incl - cnt_l;
            if (warp == 0) {
                if (lane < NSC) { group_off()[lane] = gincl - g_l; item_off()[lane] = cls_off; }
                if (lane == NSC - 1) misc[1] = gincl;                // number of groups
            }
        }
        const int nrows = ORDERED ? HASH_ROWS : (N + NT - 1) / NT;
        for (int i = 0; i < nrows; i++) {
            const int p = ORDERED ? warp * CHUNK + 32 * i + lane : tid + i * NT;
            const bool on = p < N;
            uint32_t s = 0u, cnt = 0u, at = 0u;
            if (ORDERED) {
                s = on ? pslot[p] : 0u;
                const uint32_t slot = s & 0x7fffu;
                // the lanes of this row that share my bucket, in lane (= point index) order
                const unsigned peers = __match_any_sync(FULL, on ? slot : 0x10000u + lane);
                const int leader = __ffs(peers) - 1;
                uint32_t cur = 0u;
                if (on && lane == leader) {
                    const uint32_t n = (uint32_t)__popc(peers);
                    if (warp == 0) cur = atomicAdd(&tinfo[slot], n << 20) >> 20;
                    else cur = ((uint32_t)atomicAdd(&tkey[slot], (int)(n << (10 * (warp - 1)))) >> (10 * (warp - 1))) & 1023u;
                }
                cur = __shfl_sync(FULL, cur, leader);
                at = (cur & 1023u) + (uint32_t)__popc(peers & ((1u << lane) - 1u));
                cnt = on ? (tinfo[slot] & 1023u) : 0u;
            } else if (on) {
                s = pslot[p];
                const uint32_t old = atomicAdd(&tinfo[s & 0x7fffu], 0x10000u);
                cnt = old & 0xffffu; at = old >> 16;
            }
            const bool files = on && (s & 0x8000u) && cnt > 1u;
            const int cls = files ? cls_of(cnt) : 0;
            const int off = __shfl_sync(FULL, cls_off, cls);
            if (files) wl[off + atomicAdd(&szf[cls], 1)] = (uint16_t)(s & 0x7fffu);
            if (on) {
                if (cnt == 1u) plane_point(p);
                else lstA[at] = (uint16_t)p;
            }
        }
    }
    // index-ordered copy of a bucket of any size: lstA[start..start+cnt) -> lstB (one warp)
    __device__ __forceinline__ void order_bucket(const int start, const int cnt) {
        for (int base = 0; base < cnt; base += 32) {
            const bool on = base + lane < cnt;
            const int mine = on ? lstA[start + base + lane] : 0;
            int rk = 0;
            for (int cb = 0; cb < cnt; cb += 32) {
                const int oth = cb + lane < cnt ? lstA[start + cb + lane] : 0x7fffffff;
                const int nj = min(32, cnt - cb);
                for (int j = 0; j < nj; j++) rk += __shfl_sync(0xffffffffu, oth, j) < mine ? 1 : 0;
            }
            if (on) lstB[start + rk] = (uint16_t)mine;
        }
        __syncwarp();
    }
    __device__ __forceinline__ void collide_buckets() {
        const unsigned FULL = 0xffffffffu;
        for (int j = tid; j < P.ev_words; j += NT) ev[j] = 0u;   // pslot is dead from here on: its storage becomes the spring queue
        const int ngroups = misc[1];
        const uint16_t *wl = worklist();
        const uint16_t *lst = ordered_list();
        const int my_goff = lane < NSC ? group_off()[lane] : 0x7fffffff, my_ioff = lane < NSC ? item_off()[lane] : 0,
                  my_cnt = lane < NSC ? size_count()[lane] : 0;
        int badq = 0;                                            // coincident points (reference: ZeroDivisionError)
        for (;;) {
            int g = 0;
            if (lane == 0) g = atomicAdd(&misc[6], 1);
            g = __shfl_sync(FULL, g, 0);
            if (g >= ngroups) break;
            // class of group g: the last class whose first group is <= g (empty classes share the offset of the next one)
            const int c = __popc(__ballot_sync(FULL, my_goff <= g)) - 1;
            const int gi = g - __shfl_sync(FULL, my_goff, c);
            const int cap = cls_cap(c), slot = cls_slot(c);
            const int item0 = __shfl_sync(FULL, my_ioff, c) + gi * cap;
            const int k = min(cap, __shfl_sync(FULL, my_cnt, c) - gi * cap);
            if (c == 0) {
                // a pile of more than 32 points: members in 2 or 4 registers per lane, or the shared-memory path
                int cnt, start;
                bucket_range(tinfo[wl[item0]], cnt, start);
                if (prof_on && lane == 0) { atomicAdd((unsigned long long *)&pacc[15], (unsigned long long)cnt * (unsigned long long)(cnt - 1)); atomicAdd((unsigned long long *)&pacc[5], 1ull); }
                if (!ORDERED) order_bucket(start, cnt);
                if (cnt <= 64) replay_bucket_regs<2>(lst, start, cnt, 0);
                else if (cnt <= 128) replay_bucket_regs<4>(lst, start, cnt, 0);
                else replay_bucket_smem(lst, start, cnt, 0);
                __syncwarp();
                continue;
            }
            // ---- lane -> (segment, member) ----
            const int seg = (lane * cls_mul(c)) >> 8, seg_base = seg * slot, li = lane - seg_base;
            int seg_cnt = 0, s_start = 0;
            if (seg < k) bucket_range(tinfo[wl[item0 + seg]], seg_cnt, s_start);
            const bool valid = li < seg_cnt;
            if (!valid) seg_cnt = 0;
            const int maxcnt = __reduce_max_sync(FULL, seg_cnt);
            int mine = valid ? lstA[s_start + li] : 0;
            if (!ORDERED) {
                // members into point-index order: rank inside the segment, permute through the bucket's lstB range
                // (the scatter often leaves a bucket sorted already: one compare with the left neighbour tells)
                const int left = __shfl_up_sync(FULL, mine, 1);
                if (__any_sync(FULL, valid && li > 0 && left > mine)) {
                    int rk = 0;
#pragma unroll 1
                    for (int j = 0; j < maxcnt; j++) {
                        const int oth = __shfl_sync(FULL, mine, seg_base + j);
                        rk += (j < seg_cnt && oth < mine) ? 1 : 0;
                    }
                    if (valid) lstB[s_start + rk] = (uint16_t)mine;
                    __syncwarp();
                    if (valid) mine = lstB[s_start + li];
                }
            }
            P4 Pm = mk4(T(0), T(0), T(0), T(1));
            if (valid) Pm = pos[mine];                               // idle lanes read nothing: another warp may be writing any point
            bool dirty = false;
            const unsigned segmask = slot >= 32 ? FULL : ((1u << slot) - 1u);
            // bit j <=> member j of my segment is a subject I am a candidate for: it exists, is not pinned (pinned
            // members never move and are skipped as subjects, cloth.pyx:314-315) and is not me
            const unsigned subj_seg = (__ballot_sync(FULL, valid && Pm.w == T(0)) >> seg_base) & segmask & ~(1u << li);
            const unsigned subj = valid ? subj_seg : 0u;             // the padding lanes of a slot are nobody's candidate
            if (prof_on) {   // members, buckets and ordered pair tests n(n-1) of this group (SURVEY.md 8d's P)
                const int pairs = __reduce_add_sync(FULL, valid ? seg_cnt - 1 : 0);
                const unsigned vm = __ballot_sync(FULL, valid);
                if (lane == 0) {
                    atomicAdd((unsigned long long *)&pacc[14], (unsigned long long)__popc(vm)); atomicAdd((unsigned long long *)&pacc[11], (unsigned long long)k);
                    atomicAdd((unsigned long long *)&pacc[15], (unsigned long long)pairs); atomicAdd((unsigned long long *)&pacc[6], (unsigned long long)maxcnt);
                }
            }
#pragma unroll 1
            for (int j = 0; j < maxcnt; j++) {
                const int src = seg_base + j;
                const T px = __shfl_sync(FULL, Pm.x, src), py = __shfl_sync(FULL, Pm.y, src), pz = __shfl_sync(FULL, Pm.z, src);
                const T d0 = px - Pm.x, d1 = py - Pm.y, d2 = pz - Pm.z;
                const T qq = d0 * d0 + d1 * d1 + d2 * d2;
                const bool hit = (subj & (1u << j)) && within_thresh(qq);
                const unsigned m = __ballot_sync(FULL, hit);
                if (m) {
                    T c0 = T(0), c1 = T(0), c2 = T(0);
                    if (hit) {
                        badq |= qq == T(0) ? 1 : 0;
                        T factor;
                        if (FAST) factor = P.thresh * rsqrtf((float)qq) - T(1);
                        else { const T d = sqrt_t(qq); factor = (P.thresh - d) / d; }
                        c0 = d0 * factor; c1 = d1 * factor; c2 = d2 * factor;
                    }
                    unsigned mm = (m >> seg_base) & segmask;        // hits of my segment's subject, bit = member
                    const int n = __popc(mm);
                    int rounds = __reduce_max_sync(FULL, n);
                    T t0 = T(0), t1 = T(0), t2 = T(0);
#pragma unroll 1
                    do {                                            // candidate order
                        const int l = seg_base + (mm ? __ffs(mm) - 1 : 0);
                        const T v0 = __shfl_sync(FULL, c0, l), v1 = __shfl_sync(FULL, c1, l), v2 = __shfl_sync(FULL, c2, l);
                        if (mm) { t0 += v0; t1 += v1; t2 += v2; }
                        mm &= mm - 1u;
                    } while (--rounds > 0);
                    if (n && li == j) {
                        const T nf = (T)n;
                        T cx, cy, cz;
                        if (FAST) { const T inv = T(1) / (nf * P.sim_steps); cx = t0 * inv; cy = t1 * inv; cz = t2 * inv; }
                        else { cx = t0 / nf / P.sim_steps; cy = t1 / nf / P.sim_steps; cz = t2 / nf / P.sim_steps; }
                        Pm = mk4(px + cx, py + cy, pz + cz, Pm.w);
                        dirty = true;
                    }
                }
            }
            if (valid) {
                // plane collision (cloth.pyx:345-370) of my member, then one write-back
                if (Pm.w == T(0) && !(Pm.z >= P.min_z)) {
                    const P4 Q = prev[mine];
                    T t = (P.min_z - Q.z) * T(1.0);
                    T tx = Q.x + t * T(-0.0), ty = Q.y + t * T(-0.0), tz = Q.z + t * T(-1.0);
                    T gx = tx + P.surf_off * T(0.0), gy = ty + P.surf_off * T(0.0), gz = tz + P.surf_off * T(1.0);
                    T ex = gx - Q.x, ey = gy - Q.y, ez = gz - Q.z;
                    Pm = mk4(Q.x + ex * fric1(), Q.y + ey * fric1(), Q.z + ez * fric1(), Pm.w);
                    dirty = true;
                }
                if (dirty) pos[mine] = Pm;
            }
            __syncwarp();
        }
        if (badq) misc[3] = 1;
    }

    // a bucket of more than 128 points, replayed through shared memory (lstB ordered)
    __device__ __forceinline__ void replay_bucket_smem(const uint16_t *lstB, const int start, const int cnt, const int j0) {
        for (int j = j0; j < cnt; j++) {
            const int p = lstB[start + j];
            const P4 Pp = pos[p];
            if (Pp.w != T(0)) continue;
            T t0 = T(0), t1 = T(0), t2 = T(0);
            int n = 0;
            for (int base = 0; base < cnt; base += 32) {
                const int cj = base + lane;
                const bool valid = cj < cnt && cj != j;
                T c0 = T(0), c1 = T(0), c2 = T(0);
                bool hit = false;
                if (valid) {
                    const P4 Pq = pos[lstB[start + cj]];
                    const T d0 = Pp.x - Pq.x, d1 = Pp.y - Pq.y, d2 = Pp.z - Pq.z;
                    const T qq = d0 * d0 + d1 * d1 + d2 * d2;
                    if (within_thresh(qq)) {
                        if (qq == T(0)) misc[3] = 1;
                        else {
                            T factor;
                            if (FAST) factor = P.thresh * rsqrtf((float)qq) - T(1);
                            else { const T d = sqrt_t(qq); factor = (P.thresh - d) / d; }
                            c0 = d0 * factor; c1 = d1 * factor; c2 = d2 * factor;
                            hit = true;
                        }
                    }
                }
                unsigned m = __ballot_sync(0xffffffffu, hit);
                n += __popc(m);
                while (m) {
                    const int l = __ffs(m) - 1;
                    m &= m - 1;
                    t0 += __shfl_sync(0xffffffffu, c0, l);
                    t1 += __shfl_sync(0xffffffffu, c1, l);
                    t2 += __shfl_sync(0xffffffffu, c2, l);
                }
            }
            if (n && lane == 0) {
                const T nf = (T)n;
                const T cx = t0 / nf / P.sim_steps, cy = t1 / nf / P.sim_steps, cz = t2 / nf / P.sim_steps;
                pos[p] = mk4(Pp.x + cx, Pp.y + cy, Pp.z + cz, Pp.w);
            }
            __syncwarp();
        }
        for (int base = 0; base < cnt; base += 32)
            if (base + lane < cnt) plane_point(lstB[start + base + lane]);
    }

    // ---- _limit_spring_changes (cloth.pyx:258-296) ----
    // c_min = min(rest*1.1, rest*tear_thresh): a spring longer than that needs the sequential treatment
    __device__ __forceinline__ T limit_c(T rst) const {
        const T a = rst * T(1.1), b = rst * tear_thresh();
        return a < b ? a : b;
    }
    __device__ __forceinline__ bool spring_flagged(const P4 &Pa, const P4 &Pb, T rst, int k) const {
        if (Pa.w != T(0) && Pb.w != T(0)) return false;
        if (FAST && !REST_TABLE) {       // per-kind constant: the same product limit_c() forms, squared once on the host side
            const T d0 = Pa.x - Pb.x, d1 = Pa.y - Pb.y, d2 = Pa.z - Pb.z;
            return d0 * d0 + d1 * d1 + d2 * d2 > limit_c2_k(k);
        }
        return longer_than(Pa.x - Pb.x, Pa.y - Pb.y, Pa.z - Pb.z, limit_c(rst));
    }
    // snapshot test of all springs; also clears the hash table for the next substep
    __device__ __forceinline__ void limit_snapshot() {
        for (int j = tid; j < P.table_size; j += NT) { tkey[j] = CLOTH_KEY_EMPTY; tinfo[j] = 0u; }
        // the previous substep swept and still shortened many springs: the sweep is exact whatever the flags say,
        // so the flag pass is skipped until a sweep comes back short
        if (misc[7]) return;
        for (int p = tid; p < N; p += NT) {
            const P4 Pb = pos[p];
            const int r = p / W, c = p - r * W;
            const bool v0 = r > 0, v1 = c > 0, v2 = v0 && v1, v3 = v0 && (c + 1 < W), v4 = r > 1, v5 = c > 1;
            const P4 A0 = pos[v0 ? p - W : p], A1 = pos[v1 ? p - 1 : p], A2 = pos[v2 ? p - W - 1 : p];
            const P4 A3 = pos[v3 ? p - W + 1 : p], A4 = pos[v4 ? p - 2 * W : p], A5 = pos[v5 ? p - 2 : p];
            uint32_t bits = 0;
            bits |= (v0 && spring_flagged(A0, Pb, rest_of(p, 0), 0)) ? 1u : 0u;
            bits |= (v1 && spring_flagged(A1, Pb, rest_of(p, 1), 1)) ? 2u : 0u;
            bits |= (v2 && spring_flagged(A2, Pb, rest_of(p, 2), 2)) ? 4u : 0u;
            bits |= (v3 && spring_flagged(A3, Pb, rest_of(p, 3), 3)) ? 8u : 0u;
            bits |= (v4 && spring_flagged(A4, Pb, rest_of(p, 4), 4)) ? 16u : 0u;
            bits |= (v5 && spring_flagged(A5, Pb, rest_of(p, 5), 5)) ? 32u : 0u;
            if (bits) {
                const int s = p * 6;
                const int sh = s & 31;
                const uint32_t lo = bits << sh, hi = sh > 26 ? bits >> (32 - sh) : 0u;
                if (lo) atomicOr(&ev[s >> 5], lo);
                if (hi) atomicOr(&ev[(s >> 5) + 1], hi);
            }
        }
    }
    // lowest flagged slot >= from (warp-wide, all lanes get the result); 0x7fffffff if none
    __device__ __forceinline__ int next_flagged(int from) const {
        const int nw = P.ev_words;
        for (int base = from >> 5; base < nw; base += 32) {
            const int wi = base + lane;
            uint32_t word = wi < nw ? ev[wi] : 0u;
            if (wi == (from >> 5)) word &= ~((1u << (from & 31)) - 1u);
            const int cand = word ? (wi << 5) + __ffs(word) - 1 : 0x7fffffff;
            const int s = __reduce_min_sync(0xffffffffu, cand);
            if (s != 0x7fffffff) return s;
        }
        return 0x7fffffff;
    }
    // Ordered replay by one warp.  Every lane evaluates the popped spring redundantly (no broadcast needed);
    // lanes 0-23 additionally own one of the <= 2 x 12 springs incident to its end points (a fixed per-lane
    // geometry) and re-test it in registers against the updated end point, so that the next pop is
    // min(already flagged, newly flagged) without a round trip through shared memory.
    __device__ __forceinline__ void limit_replay(int replay_warp) {
        if (warp != replay_warp) return;
        // per-lane incident spring: i in 0..11 relative to end point x (lanes 0-11: ptA, 12-23: ptB of the event)
        const int i = lane < 12 ? lane : lane - 12;
        // springs 0..5 are created by x itself (x is ptB); 6..11 by x+1, x+2, x+W-1, x+W, x+W+1, x+2W with x as ptA
        const int inc_dq = i < 6 ? 0 : (i == 6 ? 1 : (i == 7 ? 2 : (i == 8 ? W - 1 : (i == 9 ? W : (i == 10 ? W + 1 : 2 * W)))));
        const int inc_k = i < 6 ? i : (i == 6 ? 1 : (i == 7 ? 5 : (i == 8 ? 3 : (i == 9 ? 0 : (i == 10 ? 2 : 4)))));
        const int inc_other = i < 6 ? -koff(inc_k) : inc_dq;   // the end point that is not x, relative to x
        // spring kind inc_k exists at creating point qq=(r,c) <=> qq >= minq && cmin <= c <= cmax   (cloth.pyx:135-146)
        const int minq = lane >= 24 ? 0x40000000 : ((inc_k == 0 || inc_k == 2 || inc_k == 3) ? W : (inc_k == 4 ? 2 * W : 0));
        const int cmin = (inc_k == 1 || inc_k == 2) ? 1 : (inc_k == 5 ? 2 : 0);
        const int cmax = inc_k == 3 ? W - 2 : W - 1;
        const T c_lane = REST_TABLE ? T(0) : limit_c(sel6(P.rest_k, inc_k));
        const unsigned long long kp = koff_pack();
        const int nw = P.ev_words;
        int npop = 0, nmove = 0;
        int s = next_flagged(0);
        while (s != 0x7fffffff) {
            const int q = (int)(((unsigned)s * 43691u) >> 18);   // s / 6 for s < 2^17
            const int k = s - q * 6;
            const int a = q - (int)((kp >> (10 * k)) & 1023ull);
            // flags already queued beyond s: loaded now, consumed at the end of the iteration
            const int wi0 = (s + 1) >> 5;
            uint32_t word = (wi0 + lane < nw) ? ev[wi0 + lane] : 0u;
            if (lane == 0) word &= ~((1u << ((s + 1) & 31)) - 1u);
            P4 Pa = pos[a], Pb = pos[q];
            // my incident spring
            const int x = lane < 12 ? a : q;
            const int qq = x + inc_dq;
            const int s2 = qq * 6 + inc_k;
            const int c2 = qq - (qq / W) * W;
            const bool inc_ok = qq >= minq && qq < N && s2 > s && c2 >= cmin && c2 <= cmax;
            const P4 Po = pos[inc_ok ? x + inc_other : x];
            npop++;
            const bool pa = Pa.w != T(0), pb = Pb.w != T(0);
            bool moved = false;
            if (FAST) {
                // branch-free: the correction factor is always computed, the stores and the re-test are predicated
                float c11, ct2;
                if (REST_TABLE) { const float r = (float)__ldg(rest + s), ct = r * (float)tear_thresh(); c11 = r * 1.1f; ct2 = ct * ct; }
                else { const float2 c = kc[k]; c11 = c.x; ct2 = c.y; }
                const float e0 = (float)(Pa.x - Pb.x), e1 = (float)(Pa.y - Pb.y), e2 = (float)(Pa.z - Pb.z);
                const float qd = e0 * e0 + e1 * e1 + e2 * e2;
                const bool live = !(pa && pb);
                moved = live && qd > c11 * c11;
                if (live && qd > ct2) misc[2] = 1;
                const float fac = 1.0f - c11 * rsqrtf(fmaxf(qd, 1e-30f));
                const float fa = (!moved || pa) ? 0.0f : (pb ? fac : fac * 0.5f);
                const float fb = (!moved || pb) ? 0.0f : (pa ? fac : fac * 0.5f);
                Pa = mk4((T)((float)Pa.x - e0 * fa), (T)((float)Pa.y - e1 * fa), (T)((float)Pa.z - e2 * fa), Pa.w);
                Pb = mk4((T)((float)Pb.x + e0 * fb), (T)((float)Pb.y + e1 * fb), (T)((float)Pb.z + e2 * fb), Pb.w);
            } else if (!(pa && pb)) {
                const T rst = REST_TABLE ? __ldg(rest + s) : sel6(P.rest_k, k);
                const T e0 = Pa.x - Pb.x, e1 = Pa.y - Pb.y, e2 = Pa.z - Pb.z;
                const T c11 = rst * T(1.1);
                const T l = norm3(e0, e1, e2);
                if (l > rst * tear_thresh()) misc[2] = 1;
                if (l > c11) {
                    const T d0 = e0 / l, d1 = e1 / l, d2 = e2 / l;
                    const T extra = l - c11;
                    moved = true;
                    if (pa) { Pb = mk4(Pb.x + d0 * extra, Pb.y + d1 * extra, Pb.z + d2 * extra, Pb.w); }
                    else if (pb) { Pa = mk4(Pa.x - d0 * extra, Pa.y - d1 * extra, Pa.z - d2 * extra, Pa.w); }
                    else {
                        const T ed = extra * T(0.5);
                        Pa = mk4(Pa.x - d0 * ed, Pa.y - d1 * ed, Pa.z - d2 * ed, Pa.w);
                        Pb = mk4(Pb.x + d0 * ed, Pb.y + d1 * ed, Pb.z + d2 * ed, Pb.w);
                    }
                }
            }
            int cand = 0x7fffffff;
            nmove += moved ? 1 : 0;
            __syncwarp();                                            // every lane has read its points before lane 0 stores
            if (lane == 0 && moved) { if (!pa) pos[a] = Pa; if (!pb) pos[q] = Pb; }
            {
                // re-test my incident spring against the updated end point, in registers.  The squared terms make
                // the test independent of which end is ptA, so no lane-divergent code is needed.
                const bool x_moved = lane < 12 ? !pa : !pb;
                const P4 Px = lane < 12 ? Pa : Pb;
                const T cl = REST_TABLE ? limit_c(__ldg(rest + (inc_ok ? s2 : s))) : c_lane;
                const bool flag = moved && inc_ok && x_moved && !(Px.w != T(0) && Po.w != T(0)) &&
                                  longer_than(Px.x - Po.x, Px.y - Po.y, Px.z - Po.z, cl);
                if (flag) { atomicOr(&ev[s2 >> 5], 1u << (s2 & 31)); cand = s2; }
            }
            // next pop = min(flags already in the queue, flags raised just now)
            if (word) { const int e = ((wi0 + lane) << 5) + __ffs(word) - 1; cand = e < cand ? e : cand; }
            int nxt = __reduce_min_sync(0xffffffffu, cand);
            __syncwarp();
            if (nxt == 0x7fffffff && wi0 + 32 < nw) nxt = next_flagged((wi0 + 32) << 5);
            s = nxt;
        }
        // the queue is left clean for the next substep
        __syncwarp();
        for (int j = lane; j < nw; j += 32) ev[j] = 0u;
        if (prof_on && lane == 0) { pacc[12] += npop; pacc[13] += nmove; }
    }

    // Wavefront sweep of the whole limit pass by one warp: level order is a topological order of the sequential
    // loop (two springs that share a point are never in the same level), so evaluating every spring level by level
    // with lanes = springs of the level gives exactly the sequential result at a cost independent of how many
    // springs are stretched.  Used when the queue is long.
    // one dependency level of the sweep.  f32: branch-free (idle lanes run a dummy spring 0-0, the correction factor is
    // computed unconditionally and stores are predicated), because divergence is what a lone warp pays most for.
    __device__ __forceinline__ int sweep_level(uint32_t cur, T rst_tab, int &torn_acc) {
        if (FAST) {
            // idle lanes run a pinned-pinned dummy spring between two copies of a point nobody writes (misc[8..11] =
            // (0,0,0,1)): no predication anywhere, and no lane reads a point another lane may be storing
            const bool on = cur != 0xffffffffu;
            const uint32_t dummy = (uint32_t)(reinterpret_cast<const unsigned char *>(misc + 8) - reinterpret_cast<const unsigned char *>(pos));
            const uint32_t ao = on ? (cur & 0xfffu) * (uint32_t)sizeof(P4) : dummy, qo = on ? ((cur >> 12) & 0xfffu) * (uint32_t)sizeof(P4) : dummy;
            const int k = (cur >> 24) & 7u;
            P4 *pa_ptr = reinterpret_cast<P4 *>(reinterpret_cast<unsigned char *>(pos) + ao), *pb_ptr = reinterpret_cast<P4 *>(reinterpret_cast<unsigned char *>(pos) + qo);
            const P4 Pa = *pa_ptr, Pb = *pb_ptr;
            float c11, ct2;
            if (REST_TABLE) { c11 = (float)rst_tab * 1.1f; const float ct = (float)rst_tab * (float)tear_thresh(); ct2 = ct * ct; }
            else { const float2 c = kc[k]; c11 = c.x; ct2 = c.y; }
            const bool pa = Pa.w != T(0), pb = Pb.w != T(0);
            const float e0 = (float)(Pa.x - Pb.x), e1 = (float)(Pa.y - Pb.y), e2 = (float)(Pa.z - Pb.z);
            const float qd = e0 * e0 + e1 * e1 + e2 * e2;
            const bool live = !(pa && pb);
            const bool str = live && qd > c11 * c11;
            torn_acc |= (live && qd > ct2) ? 1 : 0;
            const float fac = 1.0f - c11 * rsqrtf(fmaxf(qd, 1e-30f));
            const float half = fac * 0.5f;
            const float fa = pb ? fac : half, fb = pa ? fac : half;      // a pinned end is never stored
            if (str && !pa) *pa_ptr = mk4((T)((float)Pa.x - e0 * fa), (T)((float)Pa.y - e1 * fa), (T)((float)Pa.z - e2 * fa), Pa.w);
            if (str && !pb) *pb_ptr = mk4((T)((float)Pb.x + e0 * fb), (T)((float)Pb.y + e1 * fb), (T)((float)Pb.z + e2 * fb), Pb.w);
            __syncwarp();
            return str ? 1 : 0;
        }
        int moved = 0;
        if (cur != 0xffffffffu) {
            const int a = cur & 0xfffu, q = (cur >> 12) & 0xfffu, k = (cur >> 24) & 7u;
            P4 Pa = pos[a], Pb = pos[q];
            const bool pa = Pa.w != T(0), pb = Pb.w != T(0);
            if (!(pa && pb)) {
                const T rst = REST_TABLE ? rst_tab : rest_of(q, k);
                const T e0 = Pa.x - Pb.x, e1 = Pa.y - Pb.y, e2 = Pa.z - Pb.z;
                const T c11 = rst * T(1.1);
                const T l = norm3(e0, e1, e2);
                if (l > rst * tear_thresh()) misc[2] = 1;
                if (l > c11) {
                    const T d0 = e0 / l, d1 = e1 / l, d2 = e2 / l;
                    const T extra = l - c11;
                    if (pa) { pos[q] = mk4(Pb.x + d0 * extra, Pb.y + d1 * extra, Pb.z + d2 * extra, Pb.w); }
                    else if (pb) { pos[a] = mk4(Pa.x - d0 * extra, Pa.y - d1 * extra, Pa.z - d2 * extra, Pa.w); }
                    else {
                        const T ed = extra * T(0.5);
                        pos[a] = mk4(Pa.x - d0 * ed, Pa.y - d1 * ed, Pa.z - d2 * ed, Pa.w);
                        pos[q] = mk4(Pb.x + d0 * ed, Pb.y + d1 * ed, Pb.z + d2 * ed, Pb.w);
                    }
                    moved = 1;
                }
            }
        }
        __syncwarp();
        return moved;
    }
    __device__ __forceinline__ T sweep_rest(uint32_t e) const {
        if (!REST_TABLE || e == 0xffffffffu) return T(0);
        return __ldg(rest + ((e >> 12) & 0xfffu) * 6 + ((e >> 24) & 7u));
    }
    __device__ __forceinline__ void limit_sweep() {
        const int nl = P.sweep_levels;
        // the schedule: rows of 32 entries (idle lanes and the padding rows hold ~0u), padded to a multiple of eight
        // levels plus eight more, so that the loads below need neither bounds nor lane predicates.  Entries (and, with
        // a rest table, the rest lengths) are fetched eight levels ahead: the table lives in L2, shared memory leaves
        // little L1
        const uint32_t *tp = P.sweep_tbl + lane;
        uint32_t cur[8], nxt[8];
        T rcur[8], rnxt[8];
#pragma unroll
        for (int u = 0; u < 8; u++) cur[u] = __ldg(tp + 32 * u);
#pragma unroll
        for (int u = 0; u < 8; u++) rcur[u] = sweep_rest(cur[u]);
        int nmove = 0, torn = 0;
        for (int L = 0; L < nl; L += 8) {
            tp += 256;
#pragma unroll
            for (int u = 0; u < 8; u++) nxt[u] = __ldg(tp + 32 * u);
#pragma unroll
            for (int u = 0; u < 8; u++) {
                nmove += sweep_level(cur[u], rcur[u], torn);
                if (u == 3) {
#pragma unroll
                    for (int v = 0; v < 8; v++) rnxt[v] = sweep_rest(nxt[v]);
                }
            }
#pragma unroll
            for (int u = 0; u < 8; u++) { cur[u] = nxt[u]; rcur[u] = rnxt[u]; }
        }
        if (torn) misc[2] = 1;
        for (int j = lane; j < P.ev_words; j += 32) ev[j] = 0u;
        nmove = __reduce_add_sync(0xffffffffu, nmove);
        if (lane == 0) {
            misc[7] = nmove >= P.sweep_thresh ? 1 : 0;
            if (prof_on) pacc[13] += nmove;
        }
    }
    // the replay warp picks the cheaper exact strategy for this substep
    __device__ __forceinline__ void limit_resolve(int replay_warp) {
        if (warp != replay_warp) return;
        if (P.sweep_tbl != nullptr) {
            if (misc[7]) { limit_sweep(); return; }
            int cnt = 0;
            for (int j = lane; j < P.ev_words; j += 32) cnt += __popc(ev[j]);
            cnt = __reduce_add_sync(0xffffffffu, cnt);
            if (cnt >= P.sweep_thresh) { limit_sweep(); return; }
        }
        limit_replay(replay_warp);
    }

    __device__ __forceinline__ void ptick(int k) {
        if (prof_on && tid == 0) { const long long t = clock64(); pacc[k] += t - plast; plast = t; }
    }
    // ==================================================================================================
    // Graph-coloured mode (CLOTHB200_MODE_COLOURED): same phases, but the two Gauss-Seidel passes are made parallel.
    //  - self-collision: Jacobi - every point is corrected from the post-Verlet snapshot of its bucket (the reference
    //    applies corrections in place in point order; the corrections carry a 1/simulation_steps factor, so the
    //    difference is second order);
    //  - 10 % limit: the springs are edge-coloured into 12 classes (6 kinds x 2 parity classes) whose members share no
    //    point; classes run one after the other, all springs of a class in parallel, each on live positions.  This is
    //    Gauss-Seidel in colour order instead of creation order.  relax_iters > 1 repeats the pass.
    // Not bit-comparable with the reference.  The f64 build equals the oracle's own coloured update bit for bit
    // (oracle_update_coloured, tests/test_gpu_coloured_oracle.py); the f32 build is held to measured bounds against it.
    // ==================================================================================================
    static constexpr int PPT = WC ? (WC * WC + NT - 1) / NT : 1;   // points per thread (compile-time grids only)

    __device__ __forceinline__ void collide_jacobi() {
        T cx[PPT], cy[PPT], cz[PPT];
#pragma unroll
        for (int i = 0; i < PPT; i++) {
            cx[i] = cy[i] = cz[i] = T(0);
            const int p = tid + i * NT;
            if (p >= N) continue;
            const P4 Pp = pos[p];
            if (Pp.w != T(0)) continue;
            const uint32_t slot = pslot[p] & 0x7fffu;
            if (tkey[slot] == CLOTH_FIRST_NONE) continue;          // no hit anywhere in this bucket
            const uint32_t info = tinfo[slot];
            const int cnt = info & 0xffffu, start = (int)(info >> 16) - cnt;
            T t0 = T(0), t1 = T(0), t2 = T(0);
            int n = 0;
#define CLOTH_JAC(q, Pq)                                                                                    \
    {                                                                                                       \
        const T d0 = Pp.x - Pq.x, d1 = Pp.y - Pq.y, d2 = Pp.z - Pq.z;                                       \
        const T qq = d0 * d0 + d1 * d1 + d2 * d2;                                                           \
        if (q != p && within_thresh(qq)) {                                                                  \
            if (qq == T(0)) misc[3] = 1;                                                                    \
            else {                                                                                          \
                T factor;                                                                                   \
                if (FAST) factor = P.thresh * rsqrtf((float)qq) - T(1);                                     \
                else { const T d = sqrt_t(qq); factor = (P.thresh - d) / d; }                               \
                t0 += d0 * factor; t1 += d1 * factor; t2 += d2 * factor;                                    \
                n += 1;                                                                                     \
            }                                                                                               \
        }                                                                                                   \
    }
            int j = 0;
            for (; j + 4 <= cnt; j += 4) {                           // index order: deterministic summation
                const int q0 = lstB[start + j], q1 = lstB[start + j + 1], q2 = lstB[start + j + 2], q3 = lstB[start + j + 3];
                const P4 Q0 = pos[q0], Q1 = pos[q1], Q2 = pos[q2], Q3 = pos[q3];
                CLOTH_JAC(q0, Q0) CLOTH_JAC(q1, Q1) CLOTH_JAC(q2, Q2) CLOTH_JAC(q3, Q3)
            }
            for (; j < cnt; j++) {
                const int q0 = lstB[start + j];
                const P4 Q0 = pos[q0];
                CLOTH_JAC(q0, Q0)
            }
#undef CLOTH_JAC
            if (n) { const T nf = (T)n; cx[i] = t0 / nf / P.sim_steps; cy[i] = t1 / nf / P.sim_steps; cz[i] = t2 / nf / P.sim_steps; }
        }
        sync();   // every point has read the snapshot
#pragma unroll
        for (int i = 0; i < PPT; i++) {
            const int p = tid + i * NT;
            if (p >= N) continue;
            const P4 Pp = pos[p];
            if (Pp.w != T(0)) continue;
            if (cx[i] != T(0) || cy[i] != T(0) || cz[i] != T(0)) pos[p] = mk4(Pp.x + cx[i], Pp.y + cy[i], Pp.z + cz[i], Pp.w);
            plane_point(p);
        }
    }

    // one colour class: kind k, parity par (of r for k = 0,2,3; of c for k = 1; of r/2 for k = 4; of c/2 for k = 5)
    template <int k, int par> __device__ __forceinline__ void limit_colour() {
        const int off = koff(k);
        for (int p = tid; p < N; p += NT) {
            const int r = p / W, c = p - r * W;
            const int key = (k == 1) ? c : (k == 4 ? (r >> 1) : (k == 5 ? (c >> 1) : r));
            if ((key & 1) != par || !kvalid(r, c, k)) continue;
            const int a = p - off;
            const P4 Pa = pos[a], Pb = pos[p];
            const bool pa = Pa.w != T(0), pb = Pb.w != T(0);
            if (pa && pb) continue;
            const T rst = rest_of(p, k);
            const T e0 = Pa.x - Pb.x, e1 = Pa.y - Pb.y, e2 = Pa.z - Pb.z;
            const T c11 = rst * T(1.1);
            const T qd = e0 * e0 + e1 * e1 + e2 * e2;
            const T ct = rst * tear_thresh();
            if (qd > ct * ct) misc[2] = 1;
            if (qd > c11 * c11) {
                T fac;
                if (FAST) fac = T(1) - c11 * rsqrtf((float)qd);
                else { const T l = sqrt_t(qd); fac = (l - c11) / l; }
                const T fa = pa ? T(0) : (pb ? fac : fac * T(0.5));
                const T fb = pb ? T(0) : (pa ? fac : fac * T(0.5));
                if (!pa) pos[a] = mk4(Pa.x - e0 * fa, Pa.y - e1 * fa, Pa.z - e2 * fa, Pa.w);
                if (!pb) pos[p] = mk4(Pb.x + e0 * fb, Pb.y + e1 * fb, Pb.z + e2 * fb, Pb.w);
            }
        }
    }

    __device__ __forceinline__ void update_coloured() {
        if (prof_on && tid == 0) plast = clock64();
        hooke_verlet();            sync(); ptick(0);
        commit_and_hash();         sync(); ptick(1);
        alloc_buckets();           sync(); ptick(2);
        scatter_members();         sync(); ptick(3);
        order_and_snapshot();      sync(); ptick(4);
        collide_jacobi();          sync(); ptick(6);
        for (int j = tid; j < P.table_size; j += NT) { tkey[j] = CLOTH_KEY_EMPTY; tinfo[j] = 0u; }
        for (int it = 0; it < P.relax_iters; it++) {
            limit_colour<0, 0>(); sync(); limit_colour<0, 1>(); sync();
            limit_colour<1, 0>(); sync(); limit_colour<1, 1>(); sync();
            limit_colour<2, 0>(); sync(); limit_colour<2, 1>(); sync();
            limit_colour<3, 0>(); sync(); limit_colour<3, 1>(); sync();
            limit_colour<4, 0>(); sync(); limit_colour<4, 1>(); sync();
            limit_colour<5, 0>(); sync(); limit_colour<5, 1>(); sync();
        }
        if (tid == 0) { misc[0] = 0; misc[1] = 0; misc[6] = 0; }
        sync(); ptick(8);
    }

    __device__ __forceinline__ void update() { if (COLOURED) update_coloured(); else update_reference_order(); }

    // ---- one Cloth.update() (cloth.pyx:169-214), reference order ----
    __device__ __forceinline__ void update_reference_order() {
        if (prof_on && tid == 0) plast = clock64();
        hooke_verlet();            sync(); ptick(0);
        commit_and_hash();         sync(); ptick(1);
        alloc_buckets_ro();        sync(); ptick(2);
        scatter_members_ro();      sync(); ptick(3);
        collide_buckets();         sync(); ptick(7);
        limit_snapshot();          sync(); ptick(8);
        limit_resolve(rot % NWARPS);
        if (tid == 0) { misc[0] = 0; misc[1] = 0; misc[6] = 0; }
        sync(); ptick(9);
    }

    // ---- Gripper (gripper.pyx) ----
    // adjust (gripper.pyx:55-66): a point listed m times in grabbed_pts is moved m times
    __device__ __forceinline__ void gripper_adjust(T dx, T dy, T dz) {
        for (int p = tid; p < N; p += NT) {
            P4 Q = prev[p];
            if (Q.w > T(0)) {
                P4 Pp = pos[p];
                const int m = (int)Q.w;
                for (int i = 0; i < m; i++) {
                    Q = mk4(Pp.x, Pp.y, Pp.z, Q.w);
                    Pp = mk4(dx + Pp.x, dy + Pp.y, dz + Pp.z, Pp.w);
                }
                pos[p] = Pp; prev[p] = Q;
            }
        }
    }
    // release (gripper.pyx:68-73)
    __device__ __forceinline__ void gripper_release() {
        for (int p = tid; p < N; p += NT) {
            P4 Q = prev[p];
            if (Q.w > T(0)) {
                P4 Pp = pos[p];
                Pp.w = T(0); Q.w = T(0);
                pos[p] = Pp; prev[p] = Q;
            }
        }
    }
    // grab_top (gripper.pyx:23-42) in double, the radius test rounded as the oracle's (dist2_rn): both builds grip the
    // oracle's set on their own state.  Returns len(grabbed_pts) afterwards (all threads).
    // scratch: doubles in the (idle) hash table area.
    __device__ __forceinline__ int grab_top(double x, double y, double radius) {
        double *levels = reinterpret_cast<double *>(tkey);
        const int nlev = P.n_levels;
        if (tid == 0) {
            double curZ = P.gripper_height;
            for (int i = 0; i < nlev; i++) { levels[i] = curZ; curZ -= P.thickness; }
            misc[4] = 0x7fffffff; misc[5] = 0;
        }
        sync();
        const double band = 2 * P.thickness;
        int mylev_min = 0x7fffffff;
        for (int p = tid; p < N; p += NT) {
            const P4 Pp = pos[p];
            const double px = (double)Pp.x, py = (double)Pp.y, pz = (double)Pp.z;
            if (dist2_rn(px - x, py - y) < radius) {
                for (int i = 0; i < nlev && i < mylev_min; i++)
                    if (fabs(pz - levels[i]) < band) { mylev_min = i; break; }
            }
        }
        if (mylev_min != 0x7fffffff) atomicMin(&misc[4], mylev_min);
        sync();
        const int lev = misc[4];
        int cnt = 0;
        for (int p = tid; p < N; p += NT) {
            P4 Pp = pos[p];
            P4 Q = prev[p];
            bool sel = false;
            if (lev != 0x7fffffff) {
                const double px = (double)Pp.x, py = (double)Pp.y, pz = (double)Pp.z;
                sel = (dist2_rn(px - x, py - y) < radius) && (fabs(pz - levels[lev]) < band);
            }
            if (sel) {
                Pp.w = T(1); Q.w = Q.w + T(1);
                pos[p] = Pp; prev[p] = Q;
            }
            cnt += (int)Q.w;
        }
        if (cnt) atomicAdd(&misc[5], cnt);
        sync();
        const int total = misc[5];
        sync();
        // restore the hash table area
        for (int j = tid; j < P.table_size; j += NT) { tkey[j] = CLOTH_KEY_EMPTY; tinfo[j] = 0u; }
        sync();
        return total;
    }

    // bit p set <=> point p is in gripper.grabbed_pts
    __device__ __forceinline__ void write_grab_mask(uint32_t *out) {
        const int nwords = (N + 31) >> 5;
        for (int wi = tid; wi < nwords; wi += NT) {
            uint32_t word = 0;
            for (int b = 0; b < 32; b++) { const int p = wi * 32 + b; if (p < N && prev[p].w > T(0)) word |= 1u << b; }
            out[wi] = word;
        }
    }

    // ---- coverage: area of the convex hull of the clipped (x,y) (cloth_env.py:1086-1098) ----
    __device__ __forceinline__ void clipped_xy(int p, double &x, double &y) const {
        const P4 Pp = pos[p];
        double vx = (double)Pp.x, vy = (double)Pp.y;
        vx = (0.0 > vx) ? 0.0 : vx; vx = (1.0 < vx) ? 1.0 : vx;   // min(max(p.x,0),1)
        vy = (0.0 > vy) ? 0.0 : vy; vy = (1.0 < vy) ? 1.0 : vy;
        x = vx; y = vy;
    }
    __device__ __forceinline__ bool xy_less(int a, int b) const {
        if (a >= N) return false;   // padding sorts last
        if (b >= N) return true;
        double ax, ay, bx, by;
        clipped_xy(a, ax, ay); clipped_xy(b, bx, by);
        return (ax < bx) || (ax == bx && ay < by);
    }
    // Andrew monotone chain + shoelace in double, same operations in the same order as oracle_hull_area, each rounded
    // once (cross_rn) in both builds: the f32 build's coverage is the oracle's of its own (widened) state, bit for bit.
    // Uses the hash table area as scratch (the table is rebuilt from scratch every substep).
    __device__ __forceinline__ double hull_area() {
        uint16_t *idx = reinterpret_cast<uint16_t *>(tkey);   // [np2] spans tkey+tinfo (8*table_size bytes, table_size >= np2/4)
        // [< 2N] from lstA on, over cls and lstB (contiguous, idle outside update()).  Points in convex position fill
        // N + 1 entries, one more than lstA holds when N % 8 == 0: the last lands at the head of cls (or of lstB where
        // cls aliases it), which every substep rewrites before it reads it.
        uint16_t *hull = lstA;
        int np2 = 1; while (np2 < N) np2 <<= 1;
        for (int i = tid; i < np2; i += NT) idx[i] = (uint16_t)i;
        sync();
        for (int k = 2; k <= np2; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tid; i < np2; i += NT) {
                    const int l = i ^ j;
                    if (l > i) {
                        const int a = idx[i], b = idx[l];
                        const bool up = (i & k) == 0;
                        if (up ? xy_less(b, a) : xy_less(a, b)) { idx[i] = (uint16_t)b; idx[l] = (uint16_t)a; }
                    }
                }
                sync();
            }
        }
        double area = 0.0;
        if (tid == 0) {
            int kk = 0;
            double ox, oy, ax, ay, bx, by;
            for (int i = 0; i < N; i++) {
                clipped_xy(idx[i], bx, by);
                while (kk >= 2) {
                    clipped_xy(hull[kk - 2], ox, oy); clipped_xy(hull[kk - 1], ax, ay);
                    if (cross_rn(ax - ox, ay - oy, bx - ox, by - oy) <= 0) kk--; else break;
                }
                hull[kk++] = idx[i];
            }
            for (int i = N - 2, t = kk + 1; i >= 0; i--) {
                clipped_xy(idx[i], bx, by);
                while (kk >= t) {
                    clipped_xy(hull[kk - 2], ox, oy); clipped_xy(hull[kk - 1], ax, ay);
                    if (cross_rn(ax - ox, ay - oy, bx - ox, by - oy) <= 0) kk--; else break;
                }
                hull[kk++] = idx[i];
            }
            kk--;
            double a2 = 0.0, hx, hy;
            clipped_xy(hull[0], hx, hy);
            for (int i = 0; i < kk; i++) {
                clipped_xy(hull[i], ax, ay);
                clipped_xy(hull[(i + 1) % kk], bx, by);
                a2 = __dadd_rn(a2, cross_rn(ax - hx, ay - hy, bx - hx, by - hy));
            }
            area = (kk >= 3) ? 0.5 * fabs(a2) : 0.0;
        }
        sync();
        for (int j = tid; j < P.table_size; j += NT) { tkey[j] = CLOTH_KEY_EMPTY; tinfo[j] = 0u; }
        sync();
        return area;  // valid in thread 0
    }

    // block-wide double sum (result valid in all threads); scratch = first words of tinfo, which is
    // idle (all zero) outside update() and is zeroed again before returning
    __device__ __forceinline__ double block_sum(double v) {
        double *buf = reinterpret_cast<double *>(tinfo);
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        sync();
        if (lane == 0) buf[warp] = v;
        sync();
        double s = 0.0;
        for (int w = 0; w < NWARPS; w++) s += buf[w];
        sync();
        if (tid < 2 * NWARPS) tinfo[tid] = 0u;
        sync();
        return s;
    }
    // _compute_variance (cloth_env.py:1075-1084): per-thread strided sums, block_sum's order, one rounding per operator
    __device__ __forceinline__ double variance_inv() {
        double s = 0.0;
        for (int p = tid; p < N; p += NT) s += (double)pos[p].z;
        const double mean = block_sum(s) / N;
        double v = 0.0;
        for (int p = tid; p < N; p += NT) { const double d = __dsub_rn((double)pos[p].z, mean); v = __dadd_rn(v, __dmul_rn(d, d)); }
        const double var = block_sum(v) / N;
        return (var < 0.000001) ? 1000.0 : 0.001 / var;
    }
    // _out_of_bounds (cloth_env.py:1020-1045): bounds (1,1,1), slack 0.25
    __device__ __forceinline__ bool out_of_bounds() {
        int bad = 0;
        for (int p = tid; p < N; p += NT) {
            const P4 Pp = pos[p];
            const double x = (double)Pp.x, y = (double)Pp.y, z = (double)Pp.z;
            bad |= (x >= 1 + 0.25) || (x < -0.25) || (y >= 1 + 0.25) || (y < -0.25) || (z >= 1) || (z < 0);
        }
        if (NT == 32) return __any_sync(0xffffffffu, bad) != 0;
        return __syncthreads_or(bad) != 0;
    }
};

}  // namespace clothb200
