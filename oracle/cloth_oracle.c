/*
 * cloth_oracle.c - CPU restatement (IEEE double, sequential) of gym-cloth's per-step hot path.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may build, load or call this file.
 * The shipped path (gym_cloth_b200/) never links or imports it.
 *
 * Parity status: PINNED.  tests/test_oracle_vs_reference.py runs this restatement side by
 * side with the reference's own compiled Cython physics (oracle/_ref, built by
 * oracle/build_ref.py from /root/reference/gym_cloth/physics/*.pyx) and requires
 * bit-identical positions/previous positions/pinned sets/tear flags; the committed
 * fixtures under tests/golden/ were produced by the reference itself
 * (tests/golden/make_golden.py) and are checked on every CPU test run.
 *
 * Each function cites the reference lines it follows (paths relative to /root/reference).
 * Compile with -O2 -ffp-contract=off (no FMA contraction: the reference performs one
 * rounded IEEE operation per Python-level operator).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORACLE_OK 0
#define ORACLE_ERR_ZERODIV (-1)   /* reference raises ZeroDivisionError (cloth.pyx:232, :331) */
#define ORACLE_ERR_NONFINITE (-2) /* reference raises ValueError/OverflowError in math.floor (cloth.pyx:311) */
#define ORACLE_ERR_ARG (-3)

typedef struct {
    /* cfg['cloth'] (cfg/t1_rgbd.yaml:5-22), read per update at cloth.pyx:175-186 */
    int32_t num_width_points, num_height_points;
    double width, height;
    double density, ks, damping, thickness, plane_friction, tear_thresh;
    /* Cloth.__init__ defaults (cloth.pyx:24-26) */
    double gravity, minimum_z;
    int32_t frames_per_sec, simulation_steps;
    /* cfg['env'] (cfg/t1_rgbd.yaml:32-43), read at cloth_env.py:91-106 */
    double iters_up, iters_up_rest, iters_grip_rest, iters_rest; /* doubles: tier-3 reset sets a float iters_up (cloth_env.py:960) */
    int32_t iters_pull_max;
    double reduce_factor, grip_radius, gripper_height;
    int32_t clip_act_space, delta_actions, max_actions;
    int32_t pad_;
} OracleParams;

typedef struct {
    OracleParams P;
    int N, S;
    double *pos, *prev, *force; /* [N][3] */
    uint8_t *pinned;            /* [N] */
    int32_t *sa, *sb;           /* spring endpoints, ptA (earlier point) / ptB (creating point) */
    uint8_t *stype;             /* 0 structural, 1 shearing, 2 bending */
    uint8_t *skind;             /* creation kind k = 0..5 of cloth.pyx:135-146 (ptA = ptB - {W,1,W+1,W-1,2W,2}[k]) */
    double *rest;               /* [S] */
    int32_t *grabbed;           /* gripper.grabbed_pts, multiplicity preserved */
    int n_grabbed, cap_grabbed;
    int tear;                   /* cloth.cloth_have_tear (sticky) */
    int init_side;
    /* spatial map scratch (cloth.pyx:298-305): chained lists in index order */
    int32_t *map_next, *map_head, *map_tail;
    int64_t *map_key;
    int map_cap;
    /* graph-coloured mode (oracle_update_coloured): not part of the reference */
    int mode, relax_iters;
    int32_t *corder;            /* spring indices by colour class, creation order within a class */
    int32_t cstart[13];         /* class j = corder[cstart[j] .. cstart[j+1]) */
    double *snap;               /* [N][3] post-Verlet snapshot of the Jacobi collision */
    /* instrumentation (not part of the reference): counters for design studies */
    int64_t n_updates, n_pair_tests, n_collide_hits, n_stretched, n_plane;
    int32_t *rec; int rec_cap, rec_n;   /* optional: indices of the springs shortened by the last limit pass */
} OracleCloth;

/* cloth.pyx:17-18  fastnorm */
static inline double fastnorm(double x, double y, double z) { return sqrt(x * x + y * y + z * z); }

void oracle_params_default(OracleParams *p) {
    /* values of cfg/t1_rgbd.yaml (identical in t2/t3 except init.type) */
    memset(p, 0, sizeof(*p));
    p->num_width_points = 25; p->num_height_points = 25;
    p->width = 1.0; p->height = 1.0;
    p->density = 200.0; p->ks = 10000.0; p->damping = 2.0; p->thickness = 0.02;
    p->plane_friction = 1.0; p->tear_thresh = 2.0;
    p->gravity = -9.8; p->minimum_z = 0.0;
    p->frames_per_sec = 30; p->simulation_steps = 30;
    p->iters_up = 50; p->iters_up_rest = 80; p->iters_grip_rest = 300; p->iters_rest = 1000;
    p->iters_pull_max = 400;
    p->reduce_factor = 0.002; p->grip_radius = 0.003; p->gripper_height = 1.0;
    p->clip_act_space = 1; p->delta_actions = 1; p->max_actions = 10;
}

int oracle_sizeof_params(void) { return (int)sizeof(OracleParams); }

void oracle_cloth_destroy(OracleCloth *c) {
    if (!c) return;
    free(c->pos); free(c->prev); free(c->force); free(c->pinned);
    free(c->sa); free(c->sb); free(c->stype); free(c->skind); free(c->rest); free(c->grabbed);
    free(c->corder); free(c->snap);
    free(c->map_next); free(c->map_head); free(c->map_tail); free(c->map_key);
    free(c->rec);
    free(c);
}

/* Colour class 2k + parity of spring s, created by ptB = (r, c) with kind k: the parity is that of r for k = 0, 2, 3,
 * of c for k = 1, of r >> 1 for k = 4 and of c >> 1 for k = 5.  Two springs of one class share no point. */
static int spring_class(const OracleCloth *c, int s) {
    int W = c->P.num_width_points, b = c->sb[s], r = b / W, cc = b % W, k = c->skind[s];
    int key = (k == 1) ? cc : (k == 4 ? (r >> 1) : (k == 5 ? (cc >> 1) : r));
    return 2 * k + (key & 1);
}

/* Cloth.__init__ grid + spring construction, cloth.pyx:92-146, Spring.__init__ :411-417.
 * init_type: 1/3 -> flat grid (x=dx*r, y=dy*c, z=0) ; 2 -> vertical sheet with x-noise.
 * noise: N doubles as drawn by np_random.rand()*0.01-0.005 (tier2 only, may be NULL otherwise);
 * the r==0 override to 0 (cloth.pyx:102-103) is applied here. */
OracleCloth *oracle_cloth_create(const OracleParams *P, int init_type, const double *noise, int init_side) {
    int W = P->num_width_points, H = P->num_height_points;
    if (W != H || W < 2) return NULL; /* cloth.pyx:91 assert height == width */
    if (init_type < 1 || init_type > 3) return NULL; /* cloth.pyx:131-132 ValueError */
    OracleCloth *c = (OracleCloth *)calloc(1, sizeof(OracleCloth));
    c->P = *P;
    int N = W * H;
    c->N = N;
    c->pos = (double *)calloc(3 * N, sizeof(double));
    c->prev = (double *)calloc(3 * N, sizeof(double));
    c->force = (double *)calloc(3 * N, sizeof(double));
    c->pinned = (uint8_t *)calloc(N, 1);
    c->sa = (int32_t *)malloc(6 * N * sizeof(int32_t));
    c->sb = (int32_t *)malloc(6 * N * sizeof(int32_t));
    c->stype = (uint8_t *)malloc(6 * N);
    c->skind = (uint8_t *)malloc(6 * N);
    c->corder = (int32_t *)malloc(6 * N * sizeof(int32_t));
    c->snap = (double *)calloc(3 * N, sizeof(double));
    c->rest = (double *)malloc(6 * N * sizeof(double));
    c->cap_grabbed = 64;
    c->grabbed = (int32_t *)malloc(c->cap_grabbed * sizeof(int32_t));
    c->map_cap = 1; while (c->map_cap < 4 * N) c->map_cap <<= 1;
    c->map_next = (int32_t *)malloc(N * sizeof(int32_t));
    c->map_head = (int32_t *)malloc(c->map_cap * sizeof(int32_t));
    c->map_tail = (int32_t *)malloc(c->map_cap * sizeof(int32_t));
    c->map_key = (int64_t *)malloc(c->map_cap * sizeof(int64_t));
    c->init_side = init_side;
    double dx = P->width * 1.0 / (W - 1);  /* cloth.pyx:55 */
    double dy = P->height * 1.0 / (H - 1); /* cloth.pyx:56 */
    int S = 0;
    for (int r = 0; r < H; r++) {
        for (int cc = 0; cc < W; cc++) {
            int p = r * W + cc;
            double x, y, z;
            if (init_type == 2) { /* cloth.pyx:94-116 */
                double nz = noise ? noise[p] : 0.0;
                if (r == 0) nz = 0.0;
                x = init_side ? 0.0 + fabs(nz) : 1.0 - fabs(nz);
                y = dx * cc;
                z = dy * r;
            } else { /* cloth.pyx:117-130 */
                x = dx * r; y = dy * cc; z = 0.0;
            }
            c->pos[3 * p] = x; c->pos[3 * p + 1] = y; c->pos[3 * p + 2] = z;
            c->prev[3 * p] = x; c->prev[3 * p + 1] = y; c->prev[3 * p + 2] = z; /* point.pyx:37-39 */
#define ADD_SPRING(A, T, K)                                                           \
    do {                                                                              \
        int a_ = (A);                                                                 \
        c->sa[S] = a_; c->sb[S] = p; c->stype[S] = (T); c->skind[S] = (K);            \
        c->rest[S] = fastnorm(c->pos[3 * a_] - x, c->pos[3 * a_ + 1] - y,             \
                              c->pos[3 * a_ + 2] - z); /* cloth.pyx:417 ptA - ptB */  \
        S++;                                                                          \
    } while (0)
            if (r > 0) ADD_SPRING((r - 1) * W + cc, 0, 0);                     /* :135-136 */
            if (cc > 0) ADD_SPRING(r * W + cc - 1, 0, 1);                      /* :137-138 */
            if (r > 0 && cc > 0) ADD_SPRING((r - 1) * W + cc - 1, 1, 2);       /* :139-140 */
            if (r > 0 && cc + 1 < W) ADD_SPRING((r - 1) * W + cc + 1, 1, 3);   /* :141-142 */
            if (r > 1) ADD_SPRING((r - 2) * W + cc, 2, 4);                     /* :143-144 */
            if (cc > 1) ADD_SPRING(r * W + cc - 2, 2, 5);                      /* :145-146 */
#undef ADD_SPRING
        }
    }
    c->S = S;
    /* colour classes (DESIGN.md §4 "Coloured mode"): counting sort, stable in creation order */
    memset(c->cstart, 0, sizeof(c->cstart));
    for (int s = 0; s < S; s++) c->cstart[spring_class(c, s) + 1]++;
    for (int j = 0; j < 12; j++) c->cstart[j + 1] += c->cstart[j];
    int fill[12];
    memcpy(fill, c->cstart, sizeof(fill));
    for (int s = 0; s < S; s++) c->corder[fill[spring_class(c, s)]++] = s;
    c->relax_iters = 1;
    return c;
}

int oracle_cloth_num_points(const OracleCloth *c) { return c->N; }
int oracle_cloth_num_springs(const OracleCloth *c) { return c->S; }
int oracle_cloth_tear(const OracleCloth *c) { return c->tear; }
void oracle_cloth_set_tear(OracleCloth *c, int t) { c->tear = t; }
int oracle_cloth_num_grabbed(const OracleCloth *c) { return c->n_grabbed; }
void oracle_cloth_get_grabbed(const OracleCloth *c, int32_t *out) { memcpy(out, c->grabbed, c->n_grabbed * sizeof(int32_t)); }
void oracle_cloth_get_state(const OracleCloth *c, double *pos, double *prev, uint8_t *pinned) {
    if (pos) memcpy(pos, c->pos, 3 * c->N * sizeof(double));
    if (prev) memcpy(prev, c->prev, 3 * c->N * sizeof(double));
    if (pinned) memcpy(pinned, c->pinned, c->N);
}
void oracle_cloth_set_state(OracleCloth *c, const double *pos, const double *prev, const uint8_t *pinned) {
    if (pos) memcpy(c->pos, pos, 3 * c->N * sizeof(double));
    if (prev) memcpy(c->prev, prev, 3 * c->N * sizeof(double));
    if (pinned) memcpy(c->pinned, pinned, c->N);
}
void oracle_cloth_set_grabbed(OracleCloth *c, const int32_t *idx, int n) {
    if (n > c->cap_grabbed) { c->cap_grabbed = n + 64; c->grabbed = (int32_t *)realloc(c->grabbed, c->cap_grabbed * sizeof(int32_t)); }
    memcpy(c->grabbed, idx, n * sizeof(int32_t));
    c->n_grabbed = n;
}
void oracle_cloth_get_force(const OracleCloth *c, double *f) { memcpy(f, c->force, 3 * c->N * sizeof(double)); }
void oracle_cloth_get_springs(const OracleCloth *c, int32_t *a, int32_t *b, uint8_t *t, double *rest) {
    if (a) memcpy(a, c->sa, c->S * sizeof(int32_t));
    if (b) memcpy(b, c->sb, c->S * sizeof(int32_t));
    if (t) memcpy(t, c->stype, c->S);
    if (rest) memcpy(rest, c->rest, c->S * sizeof(double));
}
void oracle_cloth_set_rest(OracleCloth *c, const double *rest) { memcpy(c->rest, rest, c->S * sizeof(double)); }
void oracle_cloth_record_limit(OracleCloth *c, int on) {
    if (on && !c->rec) { c->rec_cap = c->S; c->rec = (int32_t *)malloc(c->S * sizeof(int32_t)); }
    if (!on) { free(c->rec); c->rec = NULL; }
    c->rec_n = 0;
}
int oracle_cloth_get_limit_record(const OracleCloth *c, int32_t *out) { if (c->rec) memcpy(out, c->rec, c->rec_n * sizeof(int32_t)); return c->rec_n; }
void oracle_cloth_get_counters(const OracleCloth *c, int64_t *out5) {
    out5[0] = c->n_updates; out5[1] = c->n_pair_tests; out5[2] = c->n_collide_hits;
    out5[3] = c->n_stretched; out5[4] = c->n_plane;
}

/* cloth.pyx:216-219 + point.pyx:69-71, 83-86 */
void oracle_phase_gravity(OracleCloth *c) {
    double mass = c->P.density / c->P.num_width_points / c->P.num_height_points; /* cloth.pyx:178 */
    double mg = mass * c->P.gravity;                                               /* :179 */
    for (int p = 0; p < c->N; p++) {
        double *f = c->force + 3 * p;
        f[0] = 0.0; f[1] = 0.0; f[2] = 0.0;
        f[0] = f[0] + 0; f[1] = f[1] + 0; f[2] = f[2] + mg;
    }
}

/* cloth.pyx:221-237 */
int oracle_phase_hookes(OracleCloth *c) {
    double ks = c->P.ks;
    for (int s = 0; s < c->S; s++) {
        double kc = (c->stype[s] == 2) ? 0.2 : 1.0;
        const double *pa = c->pos + 3 * c->sa[s], *pb = c->pos + 3 * c->sb[s];
        double l = fastnorm(pb[0] - pa[0], pb[1] - pa[1], pb[2] - pa[2]);
        if (l == 0.0) return ORACLE_ERR_ZERODIV;
        double fm = ks * kc * (l - c->rest[s]) / l;
        double f0 = fm * (pb[0] - pa[0]), f1 = fm * (pb[1] - pa[1]), f2 = fm * (pb[2] - pa[2]);
        double *fa = c->force + 3 * c->sa[s], *fb = c->force + 3 * c->sb[s];
        fa[0] = fa[0] + f0; fa[1] = fa[1] + f1; fa[2] = fa[2] + f2;
        fb[0] = fb[0] + (-f0); fb[1] = fb[1] + (-f1); fb[2] = fb[2] + (-f2);
    }
    return ORACLE_OK;
}

/* cloth.pyx:239-256 */
void oracle_phase_verlet(OracleCloth *c) {
    double mass = c->P.density / c->P.num_width_points / c->P.num_height_points;
    double delta_t = 1.0 / c->P.frames_per_sec / c->P.simulation_steps; /* cloth.pyx:180 */
    double dsdm = (delta_t * delta_t) / mass;                           /* :240 */
    double damping = (1.0 - c->P.damping / 100.0);                      /* :241 */
    for (int p = 0; p < c->N; p++) {
        if (c->pinned[p]) continue;
        double *x = c->pos + 3 * p, *px = c->prev + 3 * p, *f = c->force + 3 * p;
        for (int k = 0; k < 3; k++) {
            double cur = x[k];
            double nw = x[k] + (damping * (x[k] - px[k])) + (f[k] * dsdm);
            x[k] = nw;
            px[k] = cur;
        }
    }
}

/* cloth.pyx:307-311 : (31*31)*floor(x/w) + 31*floor(y/h) + floor(z/t), w=3dx, h=3dy, t=max(w,h) */
static int hash_position(const OracleCloth *c, double x, double y, double z, int64_t *key) {
    double dx = c->P.width * 1.0 / (c->P.num_width_points - 1);
    double dy = c->P.height * 1.0 / (c->P.num_height_points - 1);
    double w = 3 * dx, h = 3 * dy;
    double t = (w > h) ? w : h; /* Python max(w,h): first maximal element; equal values identical */
    double fx = floor(x / w), fy = floor(y / h), fz = floor(z / t);
    if (!isfinite(fx) || !isfinite(fy) || !isfinite(fz)) return ORACLE_ERR_NONFINITE;
    if (fabs(fx) > 1e15 || fabs(fy) > 1e15 || fabs(fz) > 1e15) return ORACLE_ERR_NONFINITE;
    *key = (31 * 31) * (int64_t)fx + 31 * (int64_t)fy + (int64_t)fz;
    return ORACLE_OK;
}

static int map_find_slot(const OracleCloth *c, int64_t key) {
    uint64_t h = (uint64_t)key * 0x9E3779B97F4A7C15ull;
    int slot = (int)(h >> 40) & (c->map_cap - 1);
    while (c->map_head[slot] >= 0 && c->map_key[slot] != key) slot = (slot + 1) & (c->map_cap - 1);
    return slot;
}

/* cloth.pyx:298-305: dict key -> list of points, appended in point-index order */
int oracle_phase_build_map(OracleCloth *c) {
    for (int i = 0; i < c->map_cap; i++) c->map_head[i] = -1;
    for (int p = 0; p < c->N; p++) {
        int64_t key;
        int rc = hash_position(c, c->pos[3 * p], c->pos[3 * p + 1], c->pos[3 * p + 2], &key);
        if (rc) return rc;
        int slot = map_find_slot(c, key);
        c->map_next[p] = -1;
        if (c->map_head[slot] < 0) { c->map_head[slot] = p; c->map_key[slot] = key; }
        else c->map_next[c->map_tail[slot]] = p;
        c->map_tail[slot] = p;
    }
    return ORACLE_OK;
}

/* cloth.pyx:313-343 for one point */
static int self_collide_point(OracleCloth *c, int p) {
    if (c->pinned[p]) return ORACLE_OK;
    double *x = c->pos + 3 * p;
    int64_t key;
    int rc = hash_position(c, x[0], x[1], x[2], &key);
    if (rc) return rc;
    double thresh = 2.0 * c->P.thickness;
    int slot = map_find_slot(c, key);
    if (c->map_head[slot] < 0) return ORACLE_OK; /* `if pthash in self.map` */
    double t0 = 0.0, t1 = 0.0, t2 = 0.0;
    int n = 0;
    for (int q = c->map_head[slot]; q >= 0; q = c->map_next[q]) {
        if (q == p) continue;
        const double *y = c->pos + 3 * q;
        double d = fastnorm(x[0] - y[0], x[1] - y[1], x[2] - y[2]);
        c->n_pair_tests++;
        if (d <= thresh) {
            if (d == 0.0) return ORACLE_ERR_ZERODIV;
            double factor = (thresh - d) / d;
            t0 += (x[0] - y[0]) * factor;
            t1 += (x[1] - y[1]) * factor;
            t2 += (x[2] - y[2]) * factor;
            n += 1;
        }
    }
    if (n != 0) {
        double nf = (double)n;
        int ss = c->P.simulation_steps;
        double c0 = t0 / nf / ss, c1 = t1 / nf / ss, c2 = t2 / nf / ss;
        x[0] = x[0] + c0; x[1] = x[1] + c1; x[2] = x[2] + c2;
        c->n_collide_hits += n;
    }
    return ORACLE_OK;
}

int oracle_phase_self_collide(OracleCloth *c) { /* cloth.pyx:199-200 */
    for (int p = 0; p < c->N; p++) {
        int rc = self_collide_point(c, p);
        if (rc) return rc;
    }
    return ORACLE_OK;
}

/* cloth.pyx:345-370 */
void oracle_phase_plane(OracleCloth *c) {
    double fr = c->P.plane_friction, off = 0.0001, mz = c->P.minimum_z;
    for (int p = 0; p < c->N; p++) {
        double *x = c->pos + 3 * p, *px = c->prev + 3 * p;
        if (c->pinned[p] || x[2] >= mz) continue;
        double t = (mz - px[2]) * 1.0;
        double tx = px[0] + t * (-0.0), ty = px[1] + t * (-0.0), tz = px[2] + t * (-1.0);
        double gx = tx + off * 0.0, gy = ty + off * 0.0, gz = tz + off * 1.0;
        double cx = gx - px[0], cy = gy - px[1], cz = gz - px[2];
        x[0] = px[0] + cx * (1. - fr);
        x[1] = px[1] + cy * (1. - fr);
        x[2] = px[2] + cz * (1. - fr);
        c->n_plane++;
    }
}

/* cloth.pyx:258-296 */
void oracle_phase_limit(OracleCloth *c) {
    double tear_thresh = c->P.tear_thresh;
    c->rec_n = 0;
    for (int s = 0; s < c->S; s++) {
        int a = c->sa[s], b = c->sb[s];
        if (c->pinned[a] && c->pinned[b]) continue;
        double *pa = c->pos + 3 * a, *pb = c->pos + 3 * b;
        double l = fastnorm(pa[0] - pb[0], pa[1] - pb[1], pa[2] - pb[2]);
        double rest = c->rest[s];
        if (l > rest * tear_thresh) c->tear = 1;
        if (l > (rest * 1.1)) {
            double d0 = (pa[0] - pb[0]) / l, d1 = (pa[1] - pb[1]) / l, d2 = (pa[2] - pb[2]) / l;
            double extra = l - rest * 1.1;
            c->n_stretched++;
            if (c->rec && c->rec_n < c->rec_cap) c->rec[c->rec_n++] = s;
            if (c->pinned[a]) {
                pb[0] = pb[0] + d0 * extra; pb[1] = pb[1] + d1 * extra; pb[2] = pb[2] + d2 * extra;
            } else if (c->pinned[b]) {
                pa[0] = pa[0] - d0 * extra; pa[1] = pa[1] - d1 * extra; pa[2] = pa[2] - d2 * extra;
            } else {
                double ed = extra * 0.5;
                pa[0] = pa[0] - d0 * ed; pa[1] = pa[1] - d1 * ed; pa[2] = pa[2] - d2 * ed;
                pb[0] = pb[0] + d0 * ed; pb[1] = pb[1] + d1 * ed; pb[2] = pb[2] + d2 * ed;
            }
        }
    }
}

/* cloth.pyx:169-214 (render branch excluded: side channel, SURVEY.md §2 row 12) */
int oracle_update(OracleCloth *c) {
    int rc;
    oracle_phase_gravity(c);
    if ((rc = oracle_phase_hookes(c))) return rc;
    oracle_phase_verlet(c);
    if ((rc = oracle_phase_build_map(c))) return rc;
    if ((rc = oracle_phase_self_collide(c))) return rc;
    oracle_phase_plane(c);
    oracle_phase_limit(c);
    c->n_updates++;
    return ORACLE_OK;
}

/* ---- Graph-coloured mode (CLOTHB200_MODE_COLOURED, DESIGN.md §4): the specification of the kernel's
 * update_coloured(), NOT the reference's update.  The f64 coloured build equals it bit for bit: the Jacobi sums run
 * in member-index order, and the springs of one colour class share no point, so running them in parallel equals
 * running them in creation order.  Where the kernel's expression form was a free choice (squared compares, e*fac),
 * that form is part of the definition. ---- */
#define ORACLE_MODE_REFERENCE_ORDER 0
#define ORACLE_MODE_COLOURED 1

/* mode of every later update (oracle_update_n, oracle_run_plan); relax_iters limit passes, at least one */
void oracle_cloth_set_mode(OracleCloth *c, int mode, int relax_iters) { c->mode = mode; c->relax_iters = relax_iters; }
void oracle_cloth_get_colours(const OracleCloth *c, int32_t *out) {
    for (int s = 0; s < c->S; s++) out[s] = spring_class(c, s);
}

/* Jacobi self-collision: every unpinned point is corrected from the post-Verlet snapshot of its bucket (members in
 * index order, pinned members count); needs oracle_phase_build_map on the same positions. */
int oracle_phase_self_collide_jacobi(OracleCloth *c) {
    memcpy(c->snap, c->pos, 3 * c->N * sizeof(double));
    double thresh = 2.0 * c->P.thickness;
    int ss = c->P.simulation_steps;
    for (int p = 0; p < c->N; p++) {
        if (c->pinned[p]) continue;
        const double *x = c->snap + 3 * p;
        int64_t key;
        int rc = hash_position(c, x[0], x[1], x[2], &key);
        if (rc) return rc;
        int slot = map_find_slot(c, key);
        double t0 = 0.0, t1 = 0.0, t2 = 0.0;
        int n = 0;
        for (int q = c->map_head[slot]; q >= 0; q = c->map_next[q]) {
            if (q == p) continue;
            const double *y = c->snap + 3 * q;
            double d = fastnorm(x[0] - y[0], x[1] - y[1], x[2] - y[2]);
            c->n_pair_tests++;
            if (d <= thresh) {
                if (d == 0.0) return ORACLE_ERR_ZERODIV;
                double factor = (thresh - d) / d;
                t0 += (x[0] - y[0]) * factor;
                t1 += (x[1] - y[1]) * factor;
                t2 += (x[2] - y[2]) * factor;
                n += 1;
            }
        }
        if (n != 0) {
            double nf = (double)n, *w = c->pos + 3 * p;
            double c0 = t0 / nf / ss, c1 = t1 / nf / ss, c2 = t2 / nf / ss;
            w[0] = w[0] + c0; w[1] = w[1] + c1; w[2] = w[2] + c2;
            c->n_collide_hits += n;
        }
    }
    return ORACLE_OK;
}

/* The 10 % limit in colour order: classes (k, parity) for k = 0..5, parity 0, 1; max(1, relax_iters) passes.
 * Squared compares for the tear and the limit, correction e*fac with fac = (l - rest*1.1)/l. */
void oracle_phase_limit_coloured(OracleCloth *c, int relax_iters) {
    double tear_thresh = c->P.tear_thresh;
    int passes = relax_iters > 1 ? relax_iters : 1;
    c->rec_n = 0;
    for (int it = 0; it < passes; it++) {
        for (int j = 0; j < c->cstart[12]; j++) {
            int s = c->corder[j], a = c->sa[s], b = c->sb[s];
            int pa_ = c->pinned[a], pb_ = c->pinned[b];
            if (pa_ && pb_) continue;
            double *pa = c->pos + 3 * a, *pb = c->pos + 3 * b;
            double e0 = pa[0] - pb[0], e1 = pa[1] - pb[1], e2 = pa[2] - pb[2];
            double qd = e0 * e0 + e1 * e1 + e2 * e2;
            double rest = c->rest[s], c11 = rest * 1.1, ct = rest * tear_thresh;
            if (qd > ct * ct) c->tear = 1;
            if (qd > c11 * c11) {
                double l = sqrt(qd), fac = (l - c11) / l;
                double fa = pa_ ? 0.0 : (pb_ ? fac : fac * 0.5);
                double fb = pb_ ? 0.0 : (pa_ ? fac : fac * 0.5);
                c->n_stretched++;
                if (c->rec && c->rec_n < c->rec_cap) c->rec[c->rec_n++] = s;
                if (!pa_) { pa[0] = pa[0] - e0 * fa; pa[1] = pa[1] - e1 * fa; pa[2] = pa[2] - e2 * fa; }
                if (!pb_) { pb[0] = pb[0] + e0 * fb; pb[1] = pb[1] + e1 * fb; pb[2] = pb[2] + e2 * fb; }
            }
        }
    }
}

int oracle_update_coloured(OracleCloth *c) {
    int rc;
    oracle_phase_gravity(c);
    if ((rc = oracle_phase_hookes(c))) return rc;
    oracle_phase_verlet(c);
    if ((rc = oracle_phase_build_map(c))) return rc;
    if ((rc = oracle_phase_self_collide_jacobi(c))) return rc;
    oracle_phase_plane(c);
    oracle_phase_limit_coloured(c, c->relax_iters);
    c->n_updates++;
    return ORACLE_OK;
}

static int update_in_mode(OracleCloth *c) {
    return c->mode == ORACLE_MODE_COLOURED ? oracle_update_coloured(c) : oracle_update(c);
}

int oracle_update_n(OracleCloth *c, int n) {
    for (int i = 0; i < n; i++) {
        int rc = update_in_mode(c);
        if (rc) return rc;
    }
    return ORACLE_OK;
}

/* ---- Gripper (gripper.pyx) ---- */
static void grabbed_push(OracleCloth *c, int p) {
    if (c->n_grabbed == c->cap_grabbed) {
        c->cap_grabbed *= 2;
        c->grabbed = (int32_t *)realloc(c->grabbed, c->cap_grabbed * sizeof(int32_t));
    }
    c->grabbed[c->n_grabbed++] = p;
}

/* gripper.pyx:23-42.  grip_radius is passed explicitly because force_grab mutates it
 * (cloth_env.py:436-442).  Returns the number of points appended. */
int oracle_grab_top(OracleCloth *c, double x, double y, double grip_radius) {
    double curZ = c->P.gripper_height;
    double thickness = c->P.thickness;
    int n0 = c->n_grabbed;
    while (curZ > 0) {
        for (int p = 0; p < c->N; p++) {
            const double *q = c->pos + 3 * p;
            if ((q[0] - x) * (q[0] - x) + (q[1] - y) * (q[1] - y) < grip_radius &&
                fabs(q[2] - curZ) < 2 * thickness) {
                c->pinned[p] = 1;
                grabbed_push(c, p);
            }
        }
        if (c->n_grabbed > n0) break;
        curZ -= thickness;
    }
    return c->n_grabbed - n0;
}

/* gripper.pyx:44-53 */
int oracle_grab(OracleCloth *c, double x, double y, double grip_radius) {
    int n0 = c->n_grabbed;
    for (int p = 0; p < c->N; p++) {
        const double *q = c->pos + 3 * p;
        if ((q[0] - x) * (q[0] - x) + (q[1] - y) * (q[1] - y) < grip_radius) {
            c->pinned[p] = 1;
            grabbed_push(c, p);
        }
    }
    return c->n_grabbed - n0;
}

/* gripper.pyx:55-66 */
void oracle_adjust(OracleCloth *c, double x, double y, double z) {
    for (int i = 0; i < c->n_grabbed; i++) {
        int p = c->grabbed[i];
        double *q = c->pos + 3 * p, *pq = c->prev + 3 * p;
        pq[0] = q[0]; pq[1] = q[1]; pq[2] = q[2];
        q[0] = x + q[0]; q[1] = y + q[1]; q[2] = z + q[2];
    }
}

/* gripper.pyx:68-73 */
void oracle_release(OracleCloth *c) {
    for (int i = 0; i < c->n_grabbed; i++) c->pinned[c->grabbed[i]] = 0;
    c->n_grabbed = 0;
}

/* ---- ClothEnv.step (cloth_env.py:369-534) ---- */
typedef struct {
    double gx, gy;        /* grip point after un-clipping (cloth_env.py:417-421) */
    double dxr, dyr;      /* per-substep pull delta = unit dir * reduce_factor (:455-456) */
    int32_t iters_pull;   /* :460-470 */
    int32_t pad_;
} OraclePlan;

static double clampd(double v, double lo, double hi) {
    /* max(min(v, hi), lo) as written at cloth_env.py:406-409 */
    double m = (hi < v) ? hi : v; /* Python min(v, hi): hi only if hi < v */
    return (lo > m) ? lo : m;     /* Python max(m, lo): lo only if lo > m */
}

/* cloth_env.py:401-470.  `**2` is CPython float_pow -> libm pow(x, 2.0) (differs from x*x in
 * ~0.085 % of inputs), np.sqrt on a Python float is IEEE sqrt. */
void oracle_decode_action(const OracleParams *P, const double *action, OraclePlan *plan) {
    double lo[4], hi[4];
    const double pi_f32 = 3.1415927410125732; /* spaces.Box casts bounds to float32 (cloth_env.py:178-181) */
    if (P->clip_act_space) { /* cloth_env.py:164-170 */
        for (int i = 0; i < 4; i++) { lo[i] = -1.0; hi[i] = 1.0; }
    } else if (P->delta_actions) { /* :172-176 */
        lo[0] = 0; lo[1] = 0; lo[2] = -1; lo[3] = -1; hi[0] = hi[1] = hi[2] = hi[3] = 1;
    } else { /* :177-181, slack 0.25, bounds (1,1,1) */
        lo[0] = -0.25; lo[1] = -0.25; lo[2] = 0.0; lo[3] = -pi_f32;
        hi[0] = 1.25; hi[1] = 1.25; hi[2] = 1.0; hi[3] = pi_f32;
    }
    double x = clampd(action[0], lo[0], hi[0]);
    double y = clampd(action[1], lo[1], hi[1]);
    double a2 = clampd(action[2], lo[2], hi[2]);
    double a3 = clampd(action[3], lo[3], hi[3]);
    double length = a2, radians = a3;
    if (P->clip_act_space) { /* :417-426 */
        x = (x / 2.0) + 0.5;
        y = (y / 2.0) + 0.5;
        if (!P->delta_actions) {
            length = (length / 2.0) + 0.5;
            radians = radians * 3.141592653589793;
        }
    }
    double xd, yd, total_length = 0.0;
    if (P->delta_actions) { /* :448-451 */
        total_length = sqrt(pow(a2, 2.0) + pow(a3, 2.0));
        xd = a2 / (total_length + 1e-5);
        yd = a3 / (total_length + 1e-5);
    } else { /* :452-454 */
        xd = cos(radians);
        yd = sin(radians);
    }
    double xr = xd * P->reduce_factor, yr = yd * P->reduce_factor; /* :455-456 */
    int ip;
    if (P->delta_actions) { /* :460-468 */
        int ii = 0;
        double cur = 0; /* Python int 0, first += makes it a float */
        double stepl = sqrt(pow(xr, 2.0) + pow(yr, 2.0));
        if (!(stepl > 0.0)) {
            ip = 0; /* reference would spin forever when total_length>0; only dx=dy=0 reaches here and breaks at once */
        } else {
            for (;;) {
                cur += stepl;
                if (cur >= total_length) break;
                ii += 1;
            }
            ip = ii;
        }
    } else {
        ip = (int)(P->iters_pull_max * length); /* :470 int() truncates toward zero */
    }
    plan->gx = x; plan->gy = y; plan->dxr = xr; plan->dyr = yr; plan->iters_pull = ip; plan->pad_ = 0;
}

/* cloth_env.py:472-515 with a decoded plan.  Returns number of cloth.update() calls executed
 * (num_sim_steps increment) or a negative error.  out_ngrab = len(gripper.grabbed_pts) after
 * grab_top (0 => exit_early, :490-493).  force_grab as at :434-444. */
int oracle_run_plan(OracleCloth *c, const OraclePlan *plan, int force_grab, int *out_ngrab) {
    const OracleParams *P = &c->P;
    oracle_grab_top(c, plan->gx, plan->gy, P->grip_radius);
    if (force_grab) {
        double r = P->grip_radius;
        while (c->n_grabbed == 0) {
            r += 0.02; /* self._radius_inc, cloth_env.py:110 */
            oracle_grab_top(c, plan->gx, plan->gy, r);
        }
    }
    if (out_ngrab) *out_ngrab = c->n_grabbed;
    double iu = P->iters_up, iur = P->iters_up_rest, igr = P->iters_grip_rest, ir = P->iters_rest;
    double ip = (double)plan->iters_pull;
    double iterations = iu + iur + ip + igr + ir; /* :475, left-associative */
    if (c->n_grabbed == 0) iterations = 0;        /* :490-493 */
    int i = 0, nupd = 0;
    while ((double)i < iterations) {
        /* _pull, cloth_env.py:352-367 */
        if ((double)i < iu) oracle_adjust(c, 0.0, 0.0, 0.0025);
        else if ((double)i < iu + iur) { }
        else if ((double)i < iu + iur + ip) oracle_adjust(c, plan->dxr, plan->dyr, 0.0);
        else if ((double)i < iu + iur + ip + igr) { }
        else oracle_release(c);
        int rc = update_in_mode(c);
        if (rc) return rc;
        nupd++;
        if (c->tear) break; /* :511-514 */
        i += 1;
    }
    return nupd;
}

int oracle_step_action(OracleCloth *c, const double *action, int force_grab, int *out_ngrab, int *out_iters_pull) {
    OraclePlan plan;
    oracle_decode_action(&c->P, action, &plan);
    if (out_iters_pull) *out_iters_pull = plan.iters_pull;
    return oracle_run_plan(c, &plan, force_grab, out_ngrab);
}

/* ---- coverage / variance / bounds (cloth_env.py:628-638, 1020-1045, 1075-1098) ---- */
typedef struct { double x, y; } P2;
static int p2cmp(const void *a, const void *b) {
    const P2 *p = (const P2 *)a, *q = (const P2 *)b;
    if (p->x < q->x) return -1;
    if (p->x > q->x) return 1;
    if (p->y < q->y) return -1;
    if (p->y > q->y) return 1;
    return 0;
}
static double cross2(P2 o, P2 a, P2 b) { return (a.x - o.x) * (b.y - o.y) - (a.y - o.y) * (b.x - o.x); }

/* Area of the convex hull of n 2-D points (= scipy.spatial.ConvexHull(points).volume in 2-D,
 * computed there by Qhull - third-party, not in /root/reference; SciPy version unpinned by the
 * reference's requirements.txt.  Restated as Andrew's monotone chain + shoelace; agreement
 * with SciPy 1.18.1 is checked to 1e-12 in tests).  Degenerate (collinear) input -> 0, the value
 * the reference's QhullError branch assigns (cloth_env.py:634-637). */
double oracle_hull_area(const double *xy, int n) {
    if (n < 3) return 0.0;
    P2 *pts = (P2 *)malloc(n * sizeof(P2));
    P2 *h = (P2 *)malloc(2 * n * sizeof(P2));
    for (int i = 0; i < n; i++) { pts[i].x = xy[2 * i]; pts[i].y = xy[2 * i + 1]; }
    qsort(pts, n, sizeof(P2), p2cmp);
    int k = 0;
    for (int i = 0; i < n; i++) {
        while (k >= 2 && cross2(h[k - 2], h[k - 1], pts[i]) <= 0) k--;
        h[k++] = pts[i];
    }
    for (int i = n - 2, t = k + 1; i >= 0; i--) {
        while (k >= t && cross2(h[k - 2], h[k - 1], pts[i]) <= 0) k--;
        h[k++] = pts[i];
    }
    k--; /* last point equals the first */
    double a2 = 0.0;
    for (int i = 0; i < k; i++) {
        P2 p = h[i], q = h[(i + 1) % k];
        a2 += (p.x - h[0].x) * (q.y - h[0].y) - (q.x - h[0].x) * (p.y - h[0].y);
    }
    free(pts); free(h);
    return (k >= 3) ? 0.5 * fabs(a2) : 0.0;
}

/* cloth_env.py:1086-1098 / 628-638 */
double oracle_coverage(const OracleCloth *c) {
    double *xy = (double *)malloc(2 * c->N * sizeof(double));
    for (int p = 0; p < c->N; p++) {
        double x = c->pos[3 * p], y = c->pos[3 * p + 1];
        /* min(max(p.x,0),1) */
        double mx = (0 > x) ? 0.0 : x; mx = (1 < mx) ? 1.0 : mx;
        double my = (0 > y) ? 0.0 : y; my = (1 < my) ? 1.0 : my;
        xy[2 * p] = mx; xy[2 * p + 1] = my;
    }
    double a = oracle_hull_area(xy, c->N);
    free(xy);
    return a;
}

/* cloth_env.py:1075-1084 : np.var(z) (population variance); summation order differs from
 * numpy's pairwise sum, so parity is to ~1e-13 relative, not bitwise. */
double oracle_variance_inv(const OracleCloth *c) {
    double m = 0.0;
    for (int p = 0; p < c->N; p++) m += c->pos[3 * p + 2];
    m /= c->N;
    double v = 0.0;
    for (int p = 0; p < c->N; p++) { double d = c->pos[3 * p + 2] - m; v += d * d; }
    v /= c->N;
    if (v < 0.000001) return 1000.0;
    return 0.001 / v;
}

/* cloth_env.py:1020-1045, bounds (1,1,1), slack 0.25 */
int oracle_out_of_bounds(const OracleCloth *c) {
    double mxx = -INFINITY, mnx = INFINITY, mxy = -INFINITY, mny = INFINITY, mxz = -INFINITY, mnz = INFINITY;
    for (int p = 0; p < c->N; p++) {
        double x = c->pos[3 * p], y = c->pos[3 * p + 1], z = c->pos[3 * p + 2];
        if (x > mxx) mxx = x; if (x < mnx) mnx = x;
        if (y > mxy) mxy = y; if (y < mny) mny = y;
        if (z > mxz) mxz = z; if (z < mnz) mnz = z;
    }
    return (mxx >= 1 + 0.25) || (mnx < -0.25) || (mxy >= 1 + 0.25) || (mny < -0.25) || (mxz >= 1) || (mnz < 0);
}

/* ---- batch driver for the CPU baseline ("kind":"port"): n independent cloths, one call ---- */
int oracle_batch_step(OracleCloth **cloths, int n, const double *actions, int32_t *sim_steps, double *coverage) {
    for (int e = 0; e < n; e++) {
        int ng, ip;
        int rc = oracle_step_action(cloths[e], actions + 4 * e, 0, &ng, &ip);
        sim_steps[e] = rc;
        coverage[e] = oracle_coverage(cloths[e]);
    }
    return ORACLE_OK;
}
