/*
 * oracle/strict.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Strict CPU restatement of the geometric hot path of jlx-dxl/Point-Cloud-Interpolation-
 * (the reference is pure Python/torch; paths below are relative to the reference root).
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may link or call
 * this file.  The shipped CUDA library never does.
 *
 * What "strict" means: every fp32 rounding step of the reference's torch-CPU path is
 * spelled out (fmaf where MKL's K=3 sgemm fuses, separate mul/add where torch does not),
 * and every selection is by the total order (distance, index), which is one valid
 * outcome of the reference's unstable topk/sort and the only one that is deterministic.
 *
 * Pinning: pinned against outputs of the real reference executed in the build container
 * (the .npz files under tests/golden/, made by tests/golden/make_golden.py) for everything that lives in
 * Utils/Pointnet2Utils.py and Utils/Layers.py.  The pytorch3d-backed parts (orc_knn form 2,
 * orc_nearest, orc_chamfer) restate an un-vendored, un-pinned dependency: PARITY UNPINNED for those.
 *
 * Build: see oracle/Makefile  (gcc -O2 -ffp-contract=off -pthread -shared -fPIC).
 * -ffp-contract=off is REQUIRED: the compiler must not fuse a*b+c on its own.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <float.h>

#include <pthread.h>
#include <stdatomic.h>
#include <unistd.h>

/* ------------------------------------------------------------------------------------ */
/* tiny pthread parallel-for (this image's gcc has no libgomp): dynamic chunks of `grain`*/
/* ------------------------------------------------------------------------------------ */
typedef void (*par_body)(int64_t lo, int64_t hi, void *ctx);
typedef struct { par_body fn; void *ctx; int64_t n, grain; atomic_llong next; } par_job;

static int g_threads = 0;
int orc_num_threads(void)
{
    if (g_threads <= 0) {
        const char *e = getenv("ORACLE_THREADS");
        long n = e ? atol(e) : sysconf(_SC_NPROCESSORS_ONLN);
        g_threads = n < 1 ? 1 : (n > 256 ? 256 : (int)n);
    }
    return g_threads;
}
void orc_set_num_threads(int n) { g_threads = n < 1 ? 1 : n; }

static void *par_worker(void *arg)
{
    par_job *j = (par_job *)arg;
    for (;;) {
        int64_t lo = atomic_fetch_add(&j->next, j->grain);
        if (lo >= j->n) break;
        int64_t hi = lo + j->grain < j->n ? lo + j->grain : j->n;
        j->fn(lo, hi, j->ctx);
    }
    return NULL;
}

static void par_for(int64_t n, int64_t grain, par_body fn, void *ctx)
{
    par_job job; job.fn = fn; job.ctx = ctx; job.n = n; job.grain = grain < 1 ? 1 : grain;
    atomic_init(&job.next, 0);
    int nt = orc_num_threads();
    if ((int64_t)nt > (n + job.grain - 1) / job.grain) nt = (int)((n + job.grain - 1) / job.grain);
    if (nt <= 1) { par_worker(&job); return; }
    pthread_t th[256];
    for (int t = 1; t < nt; t++) pthread_create(&th[t], NULL, par_worker, &job);
    par_worker(&job);
    for (int t = 1; t < nt; t++) pthread_join(th[t], NULL);
}

/* ------------------------------------------------------------------------------------ */
/* scalar building blocks                                                               */
/* ------------------------------------------------------------------------------------ */

/* torch.sum(p ** 2, -1) on a [.,3] row: three separate squares, added x,y,z, no FMA.
 * Utils/Pointnet2Utils.py:39-40. */
static inline float sq_norm3(const float *p)
{
    float xx = p[0] * p[0];
    float yy = p[1] * p[1];
    float zz = p[2] * p[2];
    float s = xx + yy;
    return s + zz;
}

/* One entry of torch.matmul(src, dst^T) with K=3 as MKL sgemm produces it on this class
 * of CPU: product of x, then two fused multiply-adds (y, z). Utils/Pointnet2Utils.py:38 */
static inline float dot3_fma(const float *a, const float *b)
{
    float acc = a[0] * b[0];
    acc = fmaf(a[1], b[1], acc);
    acc = fmaf(a[2], b[2], acc);
    return acc;
}

/* square_distance(src,dst)[n,m]: ((-2*dot) + |src|^2) + |dst|^2, two roundings.
 * Utils/Pointnet2Utils.py:38-40 (the in-place += order fixes which norm is added first) */
static inline float sqdist_expanded(const float *s, float ns, const float *d, float nd)
{
    float t = -2.0f * dot3_fma(s, d); /* exact scaling */
    float u = t + ns;
    return u + nd;
}

/* pytorch3d knn_points / chamfer distance entry, direct form with the FMA contraction a
 * CUDA build applies: fma(dz,dz, fma(dy,dy, dx*dx)).  (pytorch3d is not vendored in the
 * reference; call sites Utils/Layers.py:220, Utils/Utils.py:47)  PARITY UNPINNED. */
static inline float sqdist_direct(const float *a, const float *b)
{
    float dx = a[0] - b[0];
    float dy = a[1] - b[1];
    float dz = a[2] - b[2];
    float acc = dx * dx;
    acc = fmaf(dy, dy, acc);
    acc = fmaf(dz, dz, acc);
    return acc;
}

/* ------------------------------------------------------------------------------------ */
/* selection helper: the k smallest FINITE entries of row[0..n) under the total order     */
/* (value, index), then -1 / +inf.                                                       */
/* Done by value-threshold first (quickselect on a scratch copy), then an index-ordered  */
/* sweep, then a tiny sort -- deliberately NOT the streaming insert the CUDA kernels use */
/* ------------------------------------------------------------------------------------ */
static float kth_smallest(float *v, int n, int k) /* k is 0-based; v is clobbered */
{
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        float pivot = v[lo + (hi - lo) / 2];
        int i = lo, j = hi;
        while (i <= j) {
            while (v[i] < pivot) i++;
            while (v[j] > pivot) j--;
            if (i <= j) { float t = v[i]; v[i] = v[j]; v[j] = t; i++; j--; }
        }
        if (k <= j) hi = j;
        else if (k >= i) lo = i;
        else break;
    }
    return v[k];
}

static void select_k(const float *row, int n, int k, float *scratch, int64_t *idx_out, float *val_out)
{
    /* only finite distances are candidates (include/b200pc.h, "Non-finite coordinates"): a NaN has no place in the order,
     * and a +inf distance would tie with the padding below */
    int nf = 0;
    for (int i = 0; i < n; i++)
        if (isfinite(row[i])) scratch[nf++] = row[i];
    int kk = k < nf ? k : nf;
    int cnt = 0;
    if (kk > 0) {
        float tau = kth_smallest(scratch, nf, kk - 1);
        /* strictly below the threshold: all of them belong (a non-finite entry compares false) */
        for (int i = 0; i < n && cnt < kk; i++)
            if (row[i] < tau) { idx_out[cnt] = i; val_out[cnt] = row[i]; cnt++; }
        /* equal to the threshold: lowest indices first until kk are collected */
        for (int i = 0; i < n && cnt < kk; i++)
            if (row[i] == tau) { idx_out[cnt] = i; val_out[cnt] = row[i]; cnt++; }
    }
    /* order the survivors by (value, index) */
    for (int a = 1; a < cnt; a++) {
        float v = val_out[a]; int64_t id = idx_out[a]; int b = a - 1;
        while (b >= 0 && (val_out[b] > v || (val_out[b] == v && idx_out[b] > id))) {
            val_out[b + 1] = val_out[b]; idx_out[b + 1] = idx_out[b]; b--;
        }
        val_out[b + 1] = v; idx_out[b + 1] = id;
    }
    for (; cnt < k; cnt++) { idx_out[cnt] = -1; val_out[cnt] = INFINITY; }   /* fewer than k candidates */
}

/* ------------------------------------------------------------------------------------ */
/* a1: square_distance  Utils/Pointnet2Utils.py:20-41                                    */
/* ------------------------------------------------------------------------------------ */
typedef struct { const float *src, *dst; int B, N, M; float *out; } sqd_ctx;
static void sqd_body(int64_t lo, int64_t hi, void *vc)
{
    sqd_ctx *c = (sqd_ctx *)vc;
    for (int64_t row = lo; row < hi; row++) {
        int b = (int)(row / c->N);
        const float *s = c->src + (size_t)row * 3;
        float ns = sq_norm3(s);
        float *o = c->out + (size_t)row * c->M;
        for (int m = 0; m < c->M; m++) {
            const float *d = c->dst + ((size_t)b * c->M + m) * 3;
            o[m] = sqdist_expanded(s, ns, d, sq_norm3(d));
        }
    }
}
void orc_square_distance(const float *src, const float *dst, int B, int N, int M, float *out)
{
    sqd_ctx c = {src, dst, B, N, M, out};
    par_for((int64_t)B * N, 64, sqd_body, &c);
}

/* ------------------------------------------------------------------------------------ */
/* a4 / a5(search part): k nearest refs per query.                                        */
/* form = 0: expanded, refs are `src` (their norm is added first)  -- kNN, Utils/Layers.py:50-53
 * form = 1: expanded, queries are `src`  -- three-NN Utils/Layers.py:180, Utils/Pointnet2Utils.py:297
 * form = 2: direct (q-r)^2 with FMA accumulation -- pytorch3d.ops.knn_points restated
 *           (PARITY UNPINNED; call sites Utils/Layers.py:220,311,393,430,
 *           PolyPCI/Models/Models_V1.py:113, PointINet20230424/models/layers.py:360,441)  */
/* ------------------------------------------------------------------------------------ */
typedef struct { const float *ref, *qry; const float *rnorm; int B, N, S, k, form; int64_t *idx; float *dist; } knn_ctx;
static void knn_body(int64_t lo, int64_t hi, void *vc)
{
    knn_ctx *c = (knn_ctx *)vc;
    int N = c->N, k = c->k;
    float *row = (float *)malloc((size_t)N * sizeof(float));
    float *scr = (float *)malloc((size_t)N * sizeof(float));
    float *vals = (float *)malloc((size_t)k * sizeof(float));
    for (int64_t qi = lo; qi < hi; qi++) {
        int b = (int)(qi / c->S);
        const float *q = c->qry + (size_t)qi * 3;
        const float *r0 = c->ref + (size_t)b * N * 3;
        const float *rn = c->rnorm + (size_t)b * N;
        float nq = sq_norm3(q);
        if (c->form == 0)      for (int n = 0; n < N; n++) row[n] = sqdist_expanded(r0 + (size_t)n * 3, rn[n], q, nq);
        else if (c->form == 1) for (int n = 0; n < N; n++) row[n] = sqdist_expanded(q, nq, r0 + (size_t)n * 3, rn[n]);
        else                   for (int n = 0; n < N; n++) row[n] = sqdist_direct(q, r0 + (size_t)n * 3);
        select_k(row, N, k, scr, c->idx + (size_t)qi * k, vals);
        if (c->dist) memcpy(c->dist + (size_t)qi * k, vals, (size_t)k * sizeof(float));
    }
    free(row); free(scr); free(vals);
}
void orc_knn(const float *ref, const float *qry, int B, int N, int S, int k, int form,
             int64_t *idx_out, float *dist_out /* may be NULL */)
{
    float *rn = (float *)malloc((size_t)B * N * sizeof(float));
    for (int64_t i = 0; i < (int64_t)B * N; i++) rn[i] = sq_norm3(ref + (size_t)i * 3);
    knn_ctx c = {ref, qry, rn, B, N, S, k, form, idx_out, dist_out};
    par_for((int64_t)B * S, 16, knn_body, &c);
    free(rn);
}

/* ------------------------------------------------------------------------------------ */
/* a2: query_ball_point  Utils/Pointnet2Utils.py:88-108                                  */
/* first `nsample` ref indices (ascending) with d <= r2; pad with the first hit; a       */
/* query with no hit yields N in every slot.  d = square_distance(new_xyz, xyz).         */
/* d <= r2 is the reference's NOT(d > r2) for every distance but NaN: a NaN distance     */
/* (non-finite coordinates) is never a hit here, as in the kernels.                      */
/* r2 is the fp32 rounding of the double radius**2 (computed by the caller).             */
/* ------------------------------------------------------------------------------------ */
typedef struct { float r2; int nsample; const float *xyz, *q; const float *rnorm; int B, N, S; int64_t *out; } ball_ctx;
static void ball_body(int64_t lo, int64_t hi, void *vc)
{
    ball_ctx *c = (ball_ctx *)vc;
    for (int64_t qi = lo; qi < hi; qi++) {
        int b = (int)(qi / c->S);
        const float *q = c->q + (size_t)qi * 3;
        float nq = sq_norm3(q);
        int64_t *o = c->out + (size_t)qi * c->nsample;
        int cnt = 0;
        for (int n = 0; n < c->N && cnt < c->nsample; n++) {
            const float *r = c->xyz + ((size_t)b * c->N + n) * 3;
            float d = sqdist_expanded(q, nq, r, c->rnorm[(size_t)b * c->N + n]);
            if (d <= c->r2) o[cnt++] = n;
        }
        int64_t first = cnt > 0 ? o[0] : (int64_t)c->N;
        for (int j = cnt; j < c->nsample; j++) o[j] = first;
    }
}
void orc_ball_query(float r2, int nsample, const float *xyz, const float *new_xyz, int B, int N, int S,
                    int64_t *out)
{
    float *rn = (float *)malloc((size_t)B * N * sizeof(float));
    for (int64_t i = 0; i < (int64_t)B * N; i++) rn[i] = sq_norm3(xyz + (size_t)i * 3);
    ball_ctx c = {r2, nsample, xyz, new_xyz, rn, B, N, S, out};
    par_for((int64_t)B * S, 16, ball_body, &c);
    free(rn);
}

/* ------------------------------------------------------------------------------------ */
/* a3: farthest_point_sample  Utils/Pointnet2Utils.py:64-85                              */
/* start[b] comes from the caller (the reference draws torch.randint on the CPU RNG).    */
/* dist = ((dx*dx + dy*dy) + dz*dz) with dx = x - cx, no FMA; running min; FIRST argmax. */
/* ------------------------------------------------------------------------------------ */
typedef struct { const float *xyz; int B, N, npoint; const int64_t *start; int64_t *out; } fps_ctx;
static void fps_body(int64_t lo, int64_t hi, void *vc)
{
    fps_ctx *c = (fps_ctx *)vc;
    int N = c->N;
    for (int64_t b = lo; b < hi; b++) {
        const float *p = c->xyz + (size_t)b * N * 3;
        float *mind = (float *)malloc((size_t)N * sizeof(float));
        for (int n = 0; n < N; n++) mind[n] = 1e10f;
        int64_t far = c->start[b];
        for (int i = 0; i < c->npoint; i++) {
            c->out[(size_t)b * c->npoint + i] = far;
            float cx = p[far * 3 + 0], cy = p[far * 3 + 1], cz = p[far * 3 + 2];
            float best = -1.0f; int64_t besti = 0;
            for (int n = 0; n < N; n++) {
                float dx = p[n * 3 + 0] - cx;
                float dy = p[n * 3 + 1] - cy;
                float dz = p[n * 3 + 2] - cz;
                float xx = dx * dx, yy = dy * dy, zz = dz * dz;
                float s = xx + yy;
                float d = s + zz;
                if (d < mind[n]) mind[n] = d;
                if (mind[n] > best) { best = mind[n]; besti = n; } /* strict > keeps the first */
            }
            far = besti;
        }
        free(mind);
    }
}
void orc_fps(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *out)
{
    fps_ctx c = {xyz, B, N, npoint, start, out};
    par_for(B, 1, fps_body, &c);
}

/* ------------------------------------------------------------------------------------ */
/* a6: index_points  Utils/Pointnet2Utils.py:44-61.  idx is flattened to [B, R].         */
/* negative indices wrap (python semantics); out-of-range returns -1 (caller raises).    */
/* ------------------------------------------------------------------------------------ */
int orc_index_points(const float *points, const int64_t *idx, int B, int N, int C, int64_t R, float *out)
{
    int bad = 0;
    for (int b = 0; b < B; b++)
        for (int64_t r = 0; r < R; r++) {
            int64_t i = idx[(size_t)b * R + r];
            if (i < 0) i += N;
            if (i < 0 || i >= N) { bad = 1; continue; }
            memcpy(out + ((size_t)b * R + r) * C, points + ((size_t)b * N + i) * C, (size_t)C * sizeof(float));
        }
    return bad ? -1 : 0;
}

/* ------------------------------------------------------------------------------------ */
/* a5: three-NN inverse-distance weights and interpolation                               */
/* variant 0: Utils/Layers.py:183-186       d<1e-10 -> 1e-10 ; w = (1/d) / sum(1/d)      */
/* variant 1: Utils/Pointnet2Utils.py:301-303   w = 1/(d+1e-8), normalised               */
/* ------------------------------------------------------------------------------------ */
void orc_three_weights(const float *dist, int64_t rows, int variant, float *w)
{
    for (int64_t r = 0; r < rows; r++) {
        float inv[3];
        for (int j = 0; j < 3; j++) {
            float d = dist[r * 3 + j];
            if (variant == 0) { if (d < 1e-10f) d = 1e-10f; inv[j] = 1.0f / d; }
            else { float e = d + 1e-8f; inv[j] = 1.0f / e; }
        }
        float s01 = inv[0] + inv[1];
        float norm = s01 + inv[2];
        for (int j = 0; j < 3; j++) w[r * 3 + j] = inv[j] / norm;
    }
}

/* out[b,n,:] = (f[i0]*w0 + f[i1]*w1) + f[i2]*w2, separate mul/add
 * Utils/Layers.py:187-188, Utils/Pointnet2Utils.py:304 */
typedef struct { const float *feat; const int64_t *idx; const float *w; int B, S, N, C; float *out; } interp_ctx;
static void interp_body(int64_t lo, int64_t hi, void *vc)
{
    interp_ctx *c = (interp_ctx *)vc;
    int C = c->C;
    for (int64_t row = lo; row < hi; row++) {
        int b = (int)(row / c->N);
        const int64_t *id = c->idx + (size_t)row * 3;
        const float *ww = c->w + (size_t)row * 3;
        int64_t i[3]; float wv[3];
        for (int j = 0; j < 3; j++) {      /* the kernels' index rule: wrap once; still out of range -> row 0, weight 0 */
            i[j] = id[j] < 0 ? id[j] + c->S : id[j]; wv[j] = ww[j];
            if (i[j] < 0 || i[j] >= c->S) { i[j] = 0; wv[j] = 0.0f; }
        }
        const float *f0 = c->feat + ((size_t)b * c->S + i[0]) * C;
        const float *f1 = c->feat + ((size_t)b * c->S + i[1]) * C;
        const float *f2 = c->feat + ((size_t)b * c->S + i[2]) * C;
        float *o = c->out + (size_t)row * C;
        for (int ch = 0; ch < C; ch++) {
            float a = f0[ch] * wv[0];
            float bb = f1[ch] * wv[1];
            float cc = f2[ch] * wv[2];
            float ab = a + bb;
            o[ch] = ab + cc;
        }
    }
}
void orc_three_interpolate(const float *feat, const int64_t *idx, const float *w, int B, int S, int N, int C,
                           float *out)
{
    interp_ctx c = {feat, idx, w, B, S, N, C, out};
    par_for((int64_t)B * N, 256, interp_body, &c);
}

/* ------------------------------------------------------------------------------------ */
/* a9: chamfer_loss -> pytorch3d.loss.chamfer_distance defaults (PARITY UNPINNED)        */
/* Utils/Utils.py:39-48.  mean_b[ mean_i min_j d(x_i,y_j) + mean_j min_i d(x_i,y_j) ].   */
/* One direction = for every a_i the nearest b_j (direct form, first minimum wins); a    */
/* point without a finite distance gets -1 / +inf, which makes the loss +inf.            */
/* The scalar is accumulated in double: its contract is 1e-5 relative, not bitwise.      */
/* ------------------------------------------------------------------------------------ */
typedef struct { const float *a, *b; int B, N, M; float *mn; int64_t *arg; } nn1_ctx;
static void nn1_body(int64_t lo, int64_t hi, void *vc)
{
    nn1_ctx *c = (nn1_ctx *)vc;
    for (int64_t row = lo; row < hi; row++) {
        int b = (int)(row / c->N);
        const float *p = c->a + (size_t)row * 3;
        const float *o = c->b + (size_t)b * c->M * 3;
        float best = INFINITY; int64_t bi = -1;     /* d < best: only a finite d is taken */
        for (int j = 0; j < c->M; j++) {
            float d = sqdist_direct(p, o + (size_t)j * 3);
            if (d < best) { best = d; bi = j; }
        }
        c->mn[row] = best; c->arg[row] = bi;
    }
}
void orc_nearest(const float *a, const float *b, int B, int N, int M, float *mn, int64_t *arg)
{
    nn1_ctx c = {a, b, B, N, M, mn, arg};
    par_for((int64_t)B * N, 16, nn1_body, &c);
}
double orc_chamfer(const float *x, const float *y, int B, int N, int M, float *dx_min, int64_t *dx_arg,
                   float *dy_min, int64_t *dy_arg)
{
    orc_nearest(x, y, B, N, M, dx_min, dx_arg);
    orc_nearest(y, x, B, M, N, dy_min, dy_arg);
    double total = 0.0;
    for (int b = 0; b < B; b++) {
        double sx = 0.0, sy = 0.0;
        for (int i = 0; i < N; i++) sx += dx_min[(size_t)b * N + i];
        for (int j = 0; j < M; j++) sy += dy_min[(size_t)b * M + j];
        total += sx / N + sy / M;
    }
    return total / B;
}
