// search.cu -- brute-force neighbour search on FP32 CUDA cores (sm_100a).
//
// One streaming skeleton serves four reference call sites (file:line relative to the reference):
//   * kNN grouping           Utils/Layers.py:50-53          form 0, top-k
//   * three-NN               Utils/Layers.py:180-182,       form 1, top-3
//                            Utils/Pointnet2Utils.py:297-299
//   * pytorch3d knn_points   Utils/Layers.py:220 ...        form 2, top-K   (also Chamfer, K=1)
//   * query_ball_point       Utils/Pointnet2Utils.py:88-108 form 1, first-nsample-by-index
//
// Design (the measurements behind each choice are in DESIGN.md and profiles/):
//   1. pack_refs_kernel turns refs [B,N,3] into 16-byte records grouped in PAIRS:
//      {x0,x1,y0,y1} {z0,z1,w0,w1} with w = |r|^2 (1 - 20 eps), padded to a whole 512-ref tile with records that can
//      never be selected; the 4 pairs of an 8-ref chunk are XOR-swizzled by the chunk number so that
//      lanes re-visiting different chunks spread over the banks.  For top-k searches tile t holds refs t, t + n_tiles, ...
//      (slot_to_ref): a strided sample of the cloud per tile, whatever order the caller's points are in.
//   2. search_kernel: 8 KB tiles stream through a 4-stage shared-memory ring (cp.async.bulk + mbarrier;
//      no producer warp: the warp that releases a stage last refills it).  Every thread OWNS Q queries:
//      their k-best heap lives in shared memory and their threshold tau in a register.
//   3. FILTER.  The prefilter value of a (query, ref) pair is
//          u = fma(z, -2qz, fma(y, -2qy, fma(x, -2qx, |r|^2)))       (3 packed FFMA2 per two refs)
//      which differs from the reference's rounded distance minus |q|^2 by a bounded rounding error, so
//      "u < thr" with thr = (tau - |q|^2) + margin is a CONSERVATIVE test for "distance < tau" in all
//      three reference roundings (filter_threshold derives the margin).  Lane l of a warp keeps chunk
//      c0+l (8 refs) in registers, the warp's 32*Q queries are broadcast one LDS.128 at a time from
//      their shared-memory records {-2qx,-2qy,-2qz,thr}, 8 values are reduced with FMNMX3 and compared
//      once; the ballot of query i is exactly the 32-chunk hit mask lane i needs.  No branch, no list
//      traffic, and one broadcast load feeds 32 x 8 pairs, which keeps the loop on the FMA pipe instead
//      of the shared-memory pipe.  (The first half tile of a ref range uses the mirrored form -- queries
//      in registers, chunks broadcast -- with a drain after 2,2,4,8,16 chunks so that tau tightens fast.)
//   4. DRAIN, once per tile and warp-synchronous: hit chunks are re-tested ref by ref (phase 1), the
//      survivors are evaluated with EXACTLY the reference's arithmetic and rounding order and, if they
//      beat the heap's root key, sifted into the query's max-heap of 64-bit keys (order_key(d) << 32 | index), laid out
//      [rank][query] so that lanes never conflict (phase 2).  The key realises the total order
//      (distance, index): ties go to the lower index whatever the visiting order.
//   5. When there are too few queries to fill 148 SMs the ref range is split over gridDim.z and
//      a small merge kernel combines the partial lists.
//   6. Top-k searches with k >= 3 that are large enough go through an occupancy grid of the refs (section 1b): every
//      query starts from a threshold that provably holds k refs, and the long searches (C2) also visit refs and queries
//      in cell order -- same pairs, same keys, bit-identical results, a third fewer instructions.
#include "search.cuh"

#include <math.h>
#include <stdio.h>
#include <math_constants.h>
#include <stdlib.h>

namespace b200pc {

constexpr int TILE = 512;                  // refs per shared-memory tile
constexpr int TILE_BYTES = TILE * 16;      // 8 KB
constexpr int STAGES = 4;                  // ring depth (3 -> 4 with an 8-entry candidate buffer: -3 % at C2 once the queries are cell-ordered)
constexpr int CHUNK = 8;                   // refs per threshold test
constexpr int REC = 8;                     // 16-byte records per chunk
constexpr int CHUNKS_PER_TILE = TILE / CHUNK;
constexpr int MAX_SPLIT = 32;
constexpr int BAR_BYTES = 128;

// ---------------------------------------------------------------------------------------------
// 1. ref packing
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float torch_sq_norm(float x, float y, float z) {
    // torch.sum(p ** 2, -1): three roundings of the squares, then (xx + yy) + zz, never fused
    return __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
}

// The filter's norm word is |r|^2 deflated by 20 eps: that is the ref's share of the filter's rounding margin
// (filter_threshold), folded into the data so that it scales with THIS ref's magnitude instead of a global bound.
__device__ __forceinline__ float filter_norm(float w) { return __fmul_rn(w, 1.0f - 20.0f * 5.9604645e-8f); }

// Which ref sits in packed slot s.  Top-k searches deal the refs out to the tiles like cards: tile t holds refs
// t, t + n_tiles, t + 2 n_tiles, ... so that every 512-slot tile is an evenly strided sample of the whole cloud.  A streaming
// top-k needs ~k(1 + ln(N/k)) heap inserts per query when the refs arrive in an order unrelated to their position, but many
// times more when they arrive spatially sorted (a raw LiDAR sweep in scan order, a Morton-sorted cloud: measured 6.6 ms
// instead of 0.75 ms on C2).  The heap key carries the ORIGINAL index, so results do not depend on the visiting order.
// The ball query keeps the natural order (its result is "the first nsample by index"): strided = 0.
__device__ __forceinline__ int slot_to_ref(int s, int strided, int n_tiles) {
    return strided ? (s & (TILE - 1)) * n_tiles + (s >> 9) : s;
}
static_assert(TILE == 512, "slot_to_ref assumes 512-slot tiles");

// Ragged batches (item_len, search.cuh): an item's refs are dealt into its OWN ceil(n_b / 512) tiles (slot_to_ref with n_tiles = this count): the slots of those
// tiles past n_b are padding records, the tiles behind them are never packed or visited.  Dense calls: n_b = N, so this is
// the padded tile count and nothing changes.
__device__ __forceinline__ int item_tiles(int n_b) { return (n_b + TILE - 1) / TILE; }

struct GridDesc;
__device__ __forceinline__ void grid_count_ref(const GridDesc *desc, unsigned *counts, int b, float x, float y, float z);

// grid != null: also count the ref into the occupancy grid (section 1b, the variant without sorting)
__global__ void pack_refs_kernel(const float *__restrict__ ref, const int64_t *__restrict__ ref_len, int N, int n_pad, int strided,
                                 float4 *__restrict__ packed, const GridDesc *__restrict__ grid, unsigned *__restrict__ counts) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;  // pair index
    const int b = blockIdx.y;
    const int n_b = item_len(ref_len, b, N), nt_b = item_tiles(n_b);
    if (p >= nt_b * (TILE / 2)) return;
    const float *r = ref + (size_t)b * N * 3;
    float x[2], y[2], z[2], w[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int i = slot_to_ref(2 * p + h, strided, nt_b);
        if (i < n_b) {
            x[h] = r[i * 3 + 0]; y[h] = r[i * 3 + 1]; z[h] = r[i * 3 + 2];
            w[h] = filter_norm(torch_sq_norm(x[h], y[h], z[h]));
            if (grid) grid_count_ref(grid, counts, b, x[h], y[h], z[h]);
        } else {
            // padding: the filter sees u = +inf or NaN (never a hit); every exact form gives +inf or NaN (never selected)
            x[h] = CUDART_INF_F; y[h] = 0.0f; z[h] = 0.0f; w[h] = CUDART_INF_F;
        }
    }
    // a chunk = 4 pairs = 128 bytes = all 32 banks.  Pair q of chunk c is stored in pair-slot q ^ (c & 3), so
    // that lanes re-visiting DIFFERENT chunks in the drain spread over the banks instead of all starting at
    // bank 0 (measured: 11.4 wavefronts per LDS.128 without the swizzle).  The filters take a min over the
    // whole chunk, so the order of the pairs inside a chunk does not matter to them.
    const int chunk = p >> 2, slot = (p & 3) ^ (chunk & 3);
    B200PC_DEV_ASSERT(chunk * 4 + slot < n_pad / 2);
    float4 *o = packed + ((size_t)b * (n_pad / 2) + (size_t)chunk * 4 + slot) * 2;
    o[0] = make_float4(x[0], x[1], y[0], y[1]);
    o[1] = make_float4(z[0], z[1], w[0], w[1]);
}

// ---------------------------------------------------------------------------------------------
// 1b. occupancy grid: cell-sorted refs and queries, and a STARTING threshold for the top-k searches
// ---------------------------------------------------------------------------------------------
// A streaming k-best that starts from tau = +inf pays k(1 + ln(N/k)) heap inserts per query (127 at C2), more than half of
// them in the first tile, and in lock-step a warp pays the maximum over its lanes (profiles/r01_notes.md: the drain is
// 50 % of the kernel).  Nothing forces the search to start blind, or to visit the points in the caller's order:
//   * THRESHOLDS (every gridded search, grid_mode >= 1).  The refs are counted into a uniform grid over their bounding box
//     (<= 128 cells along the longest axis, <= 131072 cells) with a pyramid of four coarser levels; a query starts from
//     tau0 = squared distance to the farthest corner of the first cell box around it (its cell, the 3^3 box at levels
//     0..4, else the bounding box) that holds >= k refs, inflated by the rounding error of the reference's expanded forms.
//   * CELL ORDER (the long searches, grid_mode 2).  Refs and queries are counting-sorted by cell (count, scan, scatter).
//     The 32 queries of a warp are then neighbours in space: their candidates come in the same chunks and in similar
//     numbers, so the lock-step drain idles less.  The tiles are a strided sample of the sorted refs (sorted_slot).
// Every (query, ref) pair still goes through the filter -- this is brute force in a different visiting order with a warm
// start; tau0 is only ever an upper bound and the heap's (distance, index) keys do not depend on the visiting order, so the
// results are bit-identical.  Outputs are written to the rows of the caller's query order.
constexpr int GRID_AXIS = 128;             // cells along the longest axis (level 0)
constexpr int GRID_MAX_CELLS = 131072;     // level-0 cells per batch item
constexpr int GRID_LEVELS = 5;             // level l has cells of size h * 2^l (a count pyramid)
constexpr int GRID_STRIDE = 176128;        // counters per batch item: 131072 + 32768 + 8192 + 2048 + 512 rounded up (688 KB)
constexpr int GRID_SEGS = GRID_MAX_CELLS / 1024;
constexpr long GRID_MIN_PAIRS = 1L << 24;  // searches smaller than this start blind (the grid would cost more than it saves)
constexpr long GRID_SORT_MIN_PAIRS = 1L << 29;   // and smaller than this do not sort (tools/grid_crossover.py: 2 x 16384^2 and 8 x 8192^2 gain 3 %, 16384^2 loses 20 %)

struct GridDesc {            // one per batch item, written by grid_bbox_kernel
    float lo[3], hi[3];      // bounding box of the finite refs
    float h, inv_h;          // level-0 cell size (isotropic) and its reciprocal (0 when all refs coincide)
    int dim[GRID_LEVELS][3]; // cells per axis of every level
    int off[GRID_LEVELS];    // first counter of every level
    int n_finite;            // refs with finite coordinates
    float max_w;             // upper bound of |r|^2 over the finite refs
    int pad[2];
};
static_assert(sizeof(GridDesc) == 128, "GridDesc is 128 bytes");
static_assert(GRID_STRIDE % 4096 == 0, "counters are zeroed 16 bytes at a time");

// Workspace of the grid path, per search call (B batch items).  Everything between `counts` and `tail` is zeroed by ONE memset.
struct GridBufs {
    GridDesc *desc;          // [B]
    unsigned *counts;        // [B][GRID_STRIDE]     refs per cell, all levels
    unsigned *qcend;         // [B][GRID_MAX_CELLS]  queries per level-0 cell, then (in place) the running end of each cell's range
    unsigned *tail;          // [B]                  non-finite refs placed so far (they go behind the finite ones)
    unsigned *cend;          // [B][GRID_MAX_CELLS]  refs: start, then end of each level-0 cell's range in the sorted order
    unsigned *seg, *qseg;    // [B][GRID_SEGS]       counts per 1024-cell segment (refs, queries)
    float4 *sorted;          // [B][N]   refs in cell order {x, y, z, index}
    float4 *qsorted;         // [B][S]   queries in cell order {x, y, z, index}
    int *perm;               // [B][n_pad]  sorted slot -> ref index
    float *seed;             // [B][S]   starting thresholds, in the sorted query order
};
static size_t grid_layout(int B, int N, int S, int n_pad, char *base, GridBufs *g) {
    size_t o = 0;
    auto take = [&](size_t bytes) { char *p = base ? base + o : nullptr; o += align_up(bytes, 256); return p; };
    GridDesc *desc = reinterpret_cast<GridDesc *>(take((size_t)B * sizeof(GridDesc)));
    unsigned *counts = reinterpret_cast<unsigned *>(take((size_t)B * GRID_STRIDE * sizeof(unsigned)));
    unsigned *qcend = reinterpret_cast<unsigned *>(take((size_t)B * GRID_MAX_CELLS * sizeof(unsigned)));
    unsigned *tail = reinterpret_cast<unsigned *>(take((size_t)B * sizeof(unsigned)));
    unsigned *cend = reinterpret_cast<unsigned *>(take((size_t)B * GRID_MAX_CELLS * sizeof(unsigned)));
    unsigned *seg = reinterpret_cast<unsigned *>(take((size_t)B * GRID_SEGS * sizeof(unsigned)));
    unsigned *qseg = reinterpret_cast<unsigned *>(take((size_t)B * GRID_SEGS * sizeof(unsigned)));
    float4 *sorted = reinterpret_cast<float4 *>(take((size_t)B * N * sizeof(float4)));
    float4 *qsorted = reinterpret_cast<float4 *>(take((size_t)B * S * sizeof(float4)));
    int *perm = reinterpret_cast<int *>(take((size_t)B * n_pad * sizeof(int)));
    float *seed = reinterpret_cast<float *>(take((size_t)B * S * sizeof(float)));
    if (g) *g = GridBufs{desc, counts, qcend, tail, cend, seg, qseg, sorted, qsorted, perm, seed};
    return o;
}

__device__ __forceinline__ int grid_cell(float v, float lo, float inv_h, int G) {
    const float f = (v - lo) * inv_h;
    int c = f > 0.0f ? (int)fminf(f, 1.0e6f) : 0;      // NaN -> 0
    return c < G ? c : G - 1;
}
__device__ __forceinline__ int grid_cell_index(const GridDesc &g, float x, float y, float z) {
    const int cx = grid_cell(x, g.lo[0], g.inv_h, g.dim[0][0]), cy = grid_cell(y, g.lo[1], g.inv_h, g.dim[0][1]),
              cz = grid_cell(z, g.lo[2], g.inv_h, g.dim[0][2]);
    B200PC_DEV_ASSERT(cx >= 0 && cy >= 0 && cz >= 0 && (cz * g.dim[0][1] + cy) * g.dim[0][0] + cx < GRID_MAX_CELLS);
    return (cz * g.dim[0][1] + cy) * g.dim[0][0] + cx;
}

// only the item's valid refs (i < n_b) enter the box and n_finite: an item with fewer than k of them starts from +inf, and
// one with none has an empty box (lo = +inf, hi = -inf, one cell)
__global__ void __launch_bounds__(1024) grid_bbox_kernel(const float *__restrict__ ref, const int64_t *__restrict__ ref_len, int N,
                                                         GridDesc *__restrict__ desc) {
    const int b = blockIdx.x;
    const int n_b = item_len(ref_len, b, N);
    const float *r = ref + (size_t)b * N * 3;
    float lo[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, hi[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
    int nf = 0;
    for (int i0 = threadIdx.x; i0 < n_b; i0 += 4 * blockDim.x) {        // four points per thread in flight
        float x[4], y[4], z[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * blockDim.x;
            const bool in = i < n_b;
            x[u] = in ? r[i * 3] : CUDART_NAN_F; y[u] = in ? r[i * 3 + 1] : 0.f; z[u] = in ? r[i * 3 + 2] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (isfinite(x[u]) && isfinite(y[u]) && isfinite(z[u])) {
                lo[0] = fminf(lo[0], x[u]); hi[0] = fmaxf(hi[0], x[u]);
                lo[1] = fminf(lo[1], y[u]); hi[1] = fmaxf(hi[1], y[u]);
                lo[2] = fminf(lo[2], z[u]); hi[2] = fmaxf(hi[2], z[u]);
                ++nf;
            }
    }
    __shared__ float slo[3][32], shi[3][32];
    __shared__ int snf[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
    nf = __reduce_add_sync(0xffffffffu, nf);
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { slo[a][warp] = lo[a]; shi[a][warp] = hi[a]; }
        snf[warp] = nf;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        GridDesc d;
        d.n_finite = 0;
        for (int a = 0; a < 3; ++a) { d.lo[a] = CUDART_INF_F; d.hi[a] = -CUDART_INF_F; }
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
            for (int a = 0; a < 3; ++a) { d.lo[a] = fminf(d.lo[a], slo[a][w]); d.hi[a] = fmaxf(d.hi[a], shi[a][w]); }
            d.n_finite += snf[w];
        }
        float ext[3], emax = 0.0f;
        d.max_w = 0.0f;
        for (int a = 0; a < 3; ++a) {
            ext[a] = d.n_finite > 0 ? d.hi[a] - d.lo[a] : 0.0f;
            emax = fmaxf(emax, ext[a]);
            const float m = fmaxf(fabsf(d.lo[a]), fabsf(d.hi[a]));
            d.max_w += d.n_finite > 0 ? m * m * 1.000001f : 0.0f;
        }
        d.dim[0][0] = d.dim[0][1] = d.dim[0][2] = 1;
        d.h = 0.0f; d.inv_h = 0.0f;
        if (emax > 0.0f && isfinite(emax)) {
            float h = emax / (float)GRID_AXIS;
            for (int it = 0; it < 32; ++it) {
                long cells = 1;
                for (int a = 0; a < 3; ++a) {
                    int g = (int)ceilf(ext[a] / h);
                    g = g < 1 ? 1 : (g > GRID_AXIS ? GRID_AXIS : g);
                    d.dim[0][a] = g;
                    cells *= g;
                }
                if (cells <= GRID_MAX_CELLS) break;
                h *= 2.0f;
            }
            d.h = h; d.inv_h = 1.0f / h;
        }
        int off = 0;
        for (int l = 0; l < GRID_LEVELS; ++l) {
            if (l > 0)
                for (int a = 0; a < 3; ++a) d.dim[l][a] = (d.dim[l - 1][a] + 1) >> 1;
            d.off[l] = off;
            off += d.dim[l][0] * d.dim[l][1] * d.dim[l][2];
        }
        d.pad[0] = d.pad[1] = 0;
        desc[b] = d;
    }
}

__device__ __forceinline__ void grid_count_ref(const GridDesc *desc, unsigned *counts, int b, float x, float y, float z) {
    if (isfinite(x) && isfinite(y) && isfinite(z)) atomicAdd(counts + (size_t)b * GRID_STRIDE + grid_cell_index(desc[b], x, y, z), 1u);
}

// one atomic per point: refs (finite ones) into counts, queries (clamped into the border cells; NaN -> cell 0) into qcend.
// Padded refs and queries of a ragged item are not counted.
__global__ void __launch_bounds__(256) grid_count_kernel(const float *__restrict__ ref, const int64_t *__restrict__ ref_len, int N,
                                                         const float *__restrict__ qry, const int64_t *__restrict__ qry_len, int S,
                                                         const GridDesc *__restrict__ desc, unsigned *__restrict__ counts,
                                                         unsigned *__restrict__ qcend) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (i >= N + S) return;
    if (i < N ? i >= item_len(ref_len, b, N) : i - N >= item_len(qry_len, b, S)) return;
    const GridDesc &g = desc[b];
    const float *p = i < N ? ref + ((size_t)b * N + i) * 3 : qry + ((size_t)b * S + (i - N)) * 3;
    const float x = p[0], y = p[1], z = p[2];
    if (i < N) {
        if (isfinite(x) && isfinite(y) && isfinite(z)) atomicAdd(counts + (size_t)b * GRID_STRIDE + grid_cell_index(g, x, y, z), 1u);
    } else {
        atomicAdd(qcend + (size_t)b * GRID_MAX_CELLS + grid_cell_index(g, x, y, z), 1u);
    }
}

// blockIdx.z = 0: the coarser levels of the ref counts -- every occupied level-0 cell adds its count to its ancestors (a
// few thousand atomics per cloud; counting all five levels per ref tripled the counting kernel's time: the coarse cells
// contend).  Block x owns the cells [1024 x, 1024 x + 1024) and leaves their total in seg[b][x] for grid_scan_kernel.
// blockIdx.z = 1: only the segment totals, of the query counts.
__global__ void __launch_bounds__(256) grid_pyramid_kernel(const GridDesc *__restrict__ desc, unsigned *__restrict__ counts,
                                                           unsigned *__restrict__ seg, const unsigned *__restrict__ qcend,
                                                           unsigned *__restrict__ qseg) {
    const int b = blockIdx.y;
    const bool refs = blockIdx.z == 0;
    const GridDesc &g = desc[b];
    const int cells = g.dim[0][0] * g.dim[0][1] * g.dim[0][2];
    unsigned *base = counts + (size_t)b * GRID_STRIDE;
    const unsigned *src = refs ? base : qcend + (size_t)b * GRID_MAX_CELLS;
    unsigned sum = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = blockIdx.x * 1024 + i * 256 + threadIdx.x;
        const unsigned n = c < cells ? src[c] : 0u;
        sum += n;
        if (n == 0 || !refs) continue;
        const int cx = c % g.dim[0][0], cy = (c / g.dim[0][0]) % g.dim[0][1], cz = c / (g.dim[0][0] * g.dim[0][1]);
#pragma unroll
        for (int l = 1; l < GRID_LEVELS; ++l) {
            B200PC_DEV_ASSERT(g.off[l] + (((cz >> l) * g.dim[l][1] + (cy >> l)) * g.dim[l][0] + (cx >> l)) < GRID_STRIDE);
            atomicAdd(base + g.off[l] + (((cz >> l) * g.dim[l][1] + (cy >> l)) * g.dim[l][0] + (cx >> l)), n);
        }
    }
    __shared__ unsigned sh[8];
    sum = __reduce_add_sync(0xffffffffu, sum);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += sh[w];
        (refs ? seg : qseg)[b * GRID_SEGS + blockIdx.x] = t;
    }
}

// counts -> start offsets (exclusive scan in the linear cell order): cend[c] = points in cells < c.  The scatter below then
// advances cend[c] to the END of cell c (= start of cell c + 1).  z = 0: refs (counts -> cend), z = 1: queries (in place).
__global__ void __launch_bounds__(256) grid_scan_kernel(const GridDesc *__restrict__ desc, const unsigned *__restrict__ counts,
                                                        const unsigned *__restrict__ seg, unsigned *__restrict__ cend,
                                                        unsigned *__restrict__ qcend, const unsigned *__restrict__ qseg) {
    const int b = blockIdx.y, x = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool refs = blockIdx.z == 0;
    const GridDesc &g = desc[b];
    const int cells = g.dim[0][0] * g.dim[0][1] * g.dim[0][2];
    if (x * 1024 >= cells) return;
    const unsigned *sg = (refs ? seg : qseg) + b * GRID_SEGS;
    const unsigned *in = refs ? counts + (size_t)b * GRID_STRIDE : qcend + (size_t)b * GRID_MAX_CELLS;
    unsigned *out = (refs ? cend : qcend) + (size_t)b * GRID_MAX_CELLS;
    __shared__ unsigned sh[9];
    if (warp == 0) {
        unsigned v = 0;
        for (int i = lane; i < x; i += 32) v += sg[i];
        v = __reduce_add_sync(0xffffffffu, v);
        if (lane == 0) sh[8] = v;
    }
    const int c0 = x * 1024 + 4 * threadIdx.x;
    uint4 v = *reinterpret_cast<const uint4 *>(in + c0);    // refs: may run into level 1, masked below
    if (c0 + 0 >= cells) v.x = 0;
    if (c0 + 1 >= cells) v.y = 0;
    if (c0 + 2 >= cells) v.z = 0;
    if (c0 + 3 >= cells) v.w = 0;
    const unsigned mine = v.x + v.y + v.z + v.w;
    unsigned inc = mine;                                   // inclusive scan over the warp, then over the 8 warps
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) sh[warp] = inc;
    __syncthreads();
    unsigned start = sh[8] + inc - mine;
    for (int w = 0; w < warp; ++w) start += sh[w];
    uint4 o4;
    o4.x = start; o4.y = o4.x + v.x; o4.z = o4.y + v.y; o4.w = o4.z + v.z;
    B200PC_DEV_ASSERT(c0 + 3 < GRID_MAX_CELLS);
    *reinterpret_cast<uint4 *>(out + c0) = o4;
}

// Move every point to its cell's range.  Refs: the sorted copy {x, y, z, index} for the seeds, the packed tile records of
// the search (natural slot order = sorted order; layout as in pack_refs_kernel) and the slot -> index table; non-finite
// refs go behind the finite ones, slots N .. n_pad-1 get padding records.  Queries: the sorted copy {x, y, z, index}.
// The order inside a cell depends on the atomics; nothing downstream depends on it (seeds are functions of the SET of
// refs in a box, the heap keys carry the caller's indices).
// Corner bound: every ref of the box is closer than the box's farthest corner, so
//   |q - farthest corner|^2 (1 + 1e-5) + 16 eps (|q|^2 + max|r|^2)
// bounds the k-th smallest distance in the reference's rounding (lev < 0: the whole bounding box holds n_finite >= k refs).
__device__ __forceinline__ float grid_corner_bound(const GridDesc &g, const float (&q)[3], const int (&c)[3], int lev, int rho, float nq) {
    float bound = 0.0f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        float L = g.lo[a], H = g.hi[a];
        if (lev >= 0) {
            const int cl = c[a] >> lev, gl = g.dim[lev][a];
            const int c0 = cl - rho < 0 ? 0 : cl - rho, c1 = cl + rho >= gl ? gl - 1 : cl + rho;
            const float hl = g.h * (float)(1 << lev);
            L = g.lo[a] + (float)c0 * hl;
            const float Hn = g.lo[a] + (float)(c1 + 1) * hl;  // the last cell also takes the refs clamped into it
            H = c1 == gl - 1 ? fmaxf(Hn, g.hi[a]) : Hn;
        }
        // a ref counted in cell c lies in [lo + c h, lo + (c+1) h] up to the rounding of (v - lo) * inv_h: widen by delta
        const float delta = 1e-3f * g.h + 1e-6f * fmaxf(fabsf(g.lo[a]), fabsf(g.hi[a]));
        const float m = fmaxf(fabsf(q[a] - (L - delta)), fabsf((H + delta) - q[a]));
        bound += m * m;
    }
    return bound * 1.00001f + (9.6e-7f * (nq + g.max_w) + 1e-37f);
}

// refs counted in the 3 x 3 x 3 box of level-l cells around level-0 cell c: 27 independent loads
__device__ __forceinline__ unsigned grid_box27(const GridDesc &g, const unsigned *__restrict__ base, const int (&c)[3], int l) {
    const int gx = g.dim[l][0], gy = g.dim[l][1], gz = g.dim[l][2];
    const unsigned *lv = base + g.off[l];
    const int cx = c[0] >> l, cy = c[1] >> l, cz = c[2] >> l;
    unsigned n = 0;
#pragma unroll
    for (int dz = -1; dz <= 1; ++dz)
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
            for (int dx = -1; dx <= 1; ++dx) {
                const int x = cx + dx, y = cy + dy, z = cz + dz;
                const bool in = (unsigned)x < (unsigned)gx && (unsigned)y < (unsigned)gy && (unsigned)z < (unsigned)gz;
                B200PC_DEV_ASSERT(!in || g.off[l] + (z * gy + y) * gx + x < GRID_STRIDE);
                n += in ? __ldg(lv + ((size_t)z * gy + y) * gx + x) : 0u;
            }
    return n;
}

// The first cell box around the query's level-0 cell c that holds >= k refs: the cell itself (lev 0, rho 0), then the 3^3 box
// at levels 0..4 (rho 1); lev = -1 if none does.  n_box = the refs it holds.
__device__ __forceinline__ void grid_find_box(const GridDesc &g, const unsigned *__restrict__ base, const int (&c)[3], int k, int &lev, int &rho,
                                              unsigned &n_box) {
    lev = -1; rho = 1; n_box = 0;
    // own cell and level-0 box are requested together (85 % of the lidar queries stop there); the coarser boxes only when
    // needed -- the callers run a thread per query over hundreds of thousands of queries, loads cost more than round trips
    const unsigned own = __ldg(base + ((size_t)c[2] * g.dim[0][1] + c[1]) * g.dim[0][0] + c[0]);
    const unsigned n0 = grid_box27(g, base, c, 0);
    if (own >= (unsigned)k) { lev = 0; rho = 0; n_box = own; }
    else if (n0 >= (unsigned)k) { lev = 0; n_box = n0; }
    else
        for (int l = 1; l < GRID_LEVELS; ++l) {
            n_box = grid_box27(g, base, c, l);
            if (n_box >= (unsigned)k) { lev = l; break; }
        }
}

// Starting threshold of one query from the counts alone: the corner bound of its box, +inf for a non-finite query or a cloud
// with fewer than k finite refs.
__device__ __forceinline__ float grid_corner_seed(const GridDesc &g, const unsigned *__restrict__ base, const float (&q)[3], int k) {
    if (!(isfinite(q[0]) && isfinite(q[1]) && isfinite(q[2])) || g.n_finite < k) return CUDART_INF_F;
    int c[3], lev, rho;
    unsigned n_box;
#pragma unroll
    for (int a = 0; a < 3; ++a) c[a] = grid_cell(q[a], g.lo[a], g.inv_h, g.dim[0][a]);
    grid_find_box(g, base, c, k, lev, rho, n_box);
    return grid_corner_bound(g, q, c, lev, rho, torch_sq_norm(q[0], q[1], q[2]));
}

// Tile slot of the ref at position p of the cell order: inside the ref range of one split (tps tiles) tile t takes the
// positions t, t + tps, t + 2 tps, ... -- every tile is a uniform sample of the range, as in slot_to_ref, but a chunk of 8
// slots now holds refs from a few neighbouring cells.  (Cutting the tiles straight from the cell order puts all the
// candidates of a warp into 3-4 tiles: 60 % fewer drain iterations in the host simulation, tools/drain_sim.py, but
// measured slower, 0.65 vs 0.56 ms -- the warps of a CTA share the tile ring and every heavy drain stalls the other 13;
// and a query with a loose threshold sweeps towards its neighbourhood with every ref on the way beating the last: 2 ms.)
__device__ __forceinline__ unsigned sorted_slot(unsigned p, int n_tiles, int tps) {
    const unsigned span = (unsigned)tps * TILE, s = p / span, r = p - s * span;
    const unsigned t = min((unsigned)tps, (unsigned)n_tiles - s * (unsigned)tps);      // tiles of this range
    const unsigned q = r / t;
    return s * span + (r - q * t) * TILE + q;
}

// Ragged items: positions n_b .. 512 * item_tiles(n_b) - 1 are the padding of the item's own tiles, the slots behind them
// are left alone (never visited), and only the s_b valid queries enter the sorted copy (positions 0 .. s_b - 1).
__global__ void __launch_bounds__(256) grid_scatter_kernel(const float *__restrict__ ref, const int64_t *__restrict__ ref_len, int N, int n_pad,
                                                           int tps, const float *__restrict__ qry, const int64_t *__restrict__ qry_len, int S,
                                                           const GridDesc *__restrict__ desc, GridBufs gb, float4 *__restrict__ packed, int k_seed) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    const GridDesc &g = desc[b];
    if (i < n_pad) {
        const int n_b = item_len(ref_len, b, N), nt_b = item_tiles(n_b);
        if (i >= nt_b * TILE) return;
        float x = CUDART_INF_F, y = 0.0f, z = 0.0f, w = CUDART_INF_F;    // padding (see pack_refs_kernel)
        unsigned pos = (unsigned)i;
        if (i < n_b) {
            const float *r = ref + ((size_t)b * N + i) * 3;
            x = r[0]; y = r[1]; z = r[2];
            w = filter_norm(torch_sq_norm(x, y, z));
            if (isfinite(x) && isfinite(y) && isfinite(z)) pos = atomicAdd(gb.cend + (size_t)b * GRID_MAX_CELLS + grid_cell_index(g, x, y, z), 1u);
            else pos = (unsigned)g.n_finite + atomicAdd(gb.tail + b, 1u);
            B200PC_DEV_ASSERT(pos < (unsigned)n_b);
            if (k_seed == 0) gb.sorted[(size_t)b * N + pos] = make_float4(x, y, z, __int_as_float(i));   // only grid_seed_kernel reads it
        }
        const unsigned sl = sorted_slot(pos, nt_b, tps);
        B200PC_DEV_ASSERT(sl < (unsigned)(nt_b * TILE));
        gb.perm[(size_t)b * n_pad + sl] = i;
        const unsigned chunk = sl >> 3, slot = ((sl >> 1) & 3u) ^ (chunk & 3u);
        float *o = reinterpret_cast<float *>(packed + ((size_t)b * (n_pad / 2) + (size_t)chunk * 4 + slot) * 2) + (sl & 1u);
        o[0] = x; o[2] = y; o[4] = z; o[6] = w;
    } else if (i - n_pad < item_len(qry_len, b, S)) {
        const int j = i - n_pad;
        const float *qp = qry + ((size_t)b * S + j) * 3;
        const float x = qp[0], y = qp[1], z = qp[2];
        const unsigned pos = atomicAdd(gb.qcend + (size_t)b * GRID_MAX_CELLS + grid_cell_index(g, x, y, z), 1u);
        B200PC_DEV_ASSERT(pos < (unsigned)item_len(qry_len, b, S));
        gb.qsorted[(size_t)b * S + pos] = make_float4(x, y, z, __int_as_float(j));
        if (k_seed > 0) {                                  // the query's starting threshold, here rather than in a launch of its own
            const float q[3] = {x, y, z};
            gb.seed[(size_t)b * S + pos] = grid_corner_seed(g, gb.counts + (size_t)b * GRID_STRIDE, q, k_seed);
        }
    }
}

// Starting threshold of every query: (an upper bound of) the k-th smallest distance to the refs INSIDE the first cell box
// around the query that holds >= k refs (the cell itself, then the 3^3 box at levels 0..4), read from the cell-sorted copy.
// Any k refs bound the k-th distance from above, whatever the geometry, so nothing here depends on how the cells were drawn.
//   * ONE THREAD PER QUERY, queries in cell order: the threads of a warp sit in the same or neighbouring cells, so their
//     box counts, row ranges and refs are the same addresses (one transaction per warp, L1 hits) and their loops have the
//     same trip counts.  (Measured on the way: a thread per query in the CALLER's order 0.61 ms -- every thread chases its
//     own chain of divergent loads; eight lanes per query with the rows flattened into one index range 0.14 ms --
//     20 instructions of bookkeeping per ref.)
//   * the k-th smallest is taken from a per-thread histogram in shared memory, 4 bins per octave of the squared distance,
//     62 bins below the box's farthest corner: tau0 is the upper edge of the bin in which the count reaches k
//     (<= 1.19 d_k); no ordered structure, no dependency between the refs (shared-memory REDs).
//   * in the reference's rounding: the counted refs have |r|^2 <= 2|q|^2 + 2 d, the expanded forms are off by
//     <= 10.03 eps (|q|^2 + |r|^2) <= 10.03 eps (3|q|^2 + 2 d) and this kernel's own fp32 evaluation by a few eps d,
//     hence  tau0 = e (1 + 1e-5) + 16 eps (3|q|^2 + 2 e)  for the bin edge e.
// Queries with no such box take the corner bound of the whole bounding box; non-finite queries and clouds with fewer than
// k finite refs start from +inf.  Boxes of level >= `exact` are not looked into: their queries take the box's corner bound.
constexpr int SEED_THREADS = 128, SEED_BINS = 64, SEED_SHIFT = 21, SEED_MAX_REFS = 192;
__global__ void __launch_bounds__(SEED_THREADS) grid_seed_kernel(const float4 *__restrict__ qsorted, const float *__restrict__ qraw,
                                                                 const int64_t *__restrict__ qry_len, int S, int N, int k,
                                                                 const GridDesc *__restrict__ desc, const unsigned *__restrict__ counts,
                                                                 const unsigned *__restrict__ cend, const float4 *__restrict__ sorted,
                                                                 float *__restrict__ seed, int exact) {
    // [bin][thread pair]: 16-bit counters, two threads to a word (a box is capped at SEED_MAX_REFS refs, so the low half never
    // carries into the high one).  32-bit counters would take 224 KB per SM at 7 resident CTAs and leave the L1 28 KB: every
    // ref load of the walk would go to L2.
    __shared__ __align__(16) unsigned hist_all[SEED_BINS * SEED_THREADS / 2];
    const int b = blockIdx.y, qi = blockIdx.x * SEED_THREADS + threadIdx.x;
    {   // zero the histograms (16 bytes per store)
        uint4 *hz = reinterpret_cast<uint4 *>(hist_all);
        for (int i = threadIdx.x; i < SEED_BINS * SEED_THREADS / 8; i += SEED_THREADS) hz[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();
    if (qi >= item_len(qry_len, b, S)) return;          // padded queries: the search reads no threshold for them
    float q[3];
    if (qsorted) {
        const float4 qv = __ldg(qsorted + (size_t)b * S + qi);
        q[0] = qv.x; q[1] = qv.y; q[2] = qv.z;
    } else {                                                   // the variant without sorting: queries in the caller's order
        const float *qp = qraw + ((size_t)b * S + qi) * 3;
        q[0] = __ldg(qp); q[1] = __ldg(qp + 1); q[2] = __ldg(qp + 2);
    }
    const GridDesc &g = desc[b];
    float tau0 = CUDART_INF_F;
    if (isfinite(q[0]) && isfinite(q[1]) && isfinite(q[2]) && g.n_finite >= k) {
        const float nq = torch_sq_norm(q[0], q[1], q[2]);
        const unsigned *base = counts + (size_t)b * GRID_STRIDE;
        int c[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) c[a] = grid_cell(q[a], g.lo[a], g.inv_h, g.dim[0][a]);
        int lev, rho;
        unsigned n_box;
        grid_find_box(g, base, c, k, lev, rho, n_box);
        const float corner = grid_corner_bound(g, q, c, lev, rho, nq);
        if (qsorted && lev >= 0 && lev < exact && corner < CUDART_INF_F) {
            int lo0[3], hi0[3];                               // the box in level-0 cells
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const int cl = c[a] >> lev, gla = g.dim[lev][a];
                const int c0 = cl - rho < 0 ? 0 : cl - rho, c1 = cl + rho >= gla ? gla - 1 : cl + rho;
                lo0[a] = c0 << lev;
                hi0[a] = min(((c1 + 1) << lev) - 1, g.dim[0][a] - 1);
            }
            const int width = hi0[0] - lo0[0];
            // bins: key = bits(d) >> 21 (8 exponent + 2 mantissa bits); the last bin but one holds the farthest corner, the last = overflow
            const int base_key = max((int)(__float_as_uint(corner) >> SEED_SHIFT) - (SEED_BINS - 2), 0);
            unsigned *hist = hist_all + (threadIdx.x >> 1);
            const unsigned one = (threadIdx.x & 1) ? 0x10000u : 1u, shift = (threadIdx.x & 1) * 16;
            const unsigned *ce = cend + (size_t)b * GRID_MAX_CELLS;
            const float4 *pts = sorted + (size_t)b * N;
            auto count = [&](float4 r) {
                const float dx = r.x - q[0], dy = r.y - q[1], dz = r.z - q[2];
                const float d = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
                int bin = (int)(__float_as_uint(d) >> SEED_SHIFT) - base_key;
                bin = bin < 0 ? 0 : (bin > SEED_BINS - 1 ? SEED_BINS - 1 : bin);
                atomicAdd(hist + bin * (SEED_THREADS / 2), one);  // result unused: a fire-and-forget RED, no read-modify-write chain
            };
            // A dense box is one long serial walk for its thread (1100 refs at C2: 40 us for a warp on its own, the whole
            // kernel waits for it): look at every stride-th ref, ~SEED_MAX_REFS in all.  Any subset of the refs still
            // bounds the k-th distance, only less tightly -- for the few queries at the edge of a dense region.
            const unsigned stride = (n_box + SEED_MAX_REFS - 1) / SEED_MAX_REFS;
            for (int z = lo0[2]; z <= hi0[2]; ++z)
                for (int y = lo0[1]; y <= hi0[1]; ++y) {
                    // the cells of one x-row are neighbours in the linear order: one contiguous range of sorted refs
                    const int lin0 = (z * g.dim[0][1] + y) * g.dim[0][0] + lo0[0];
                    unsigned p = lin0 > 0 ? __ldg(ce + lin0 - 1) : 0u;
                    B200PC_DEV_ASSERT(lin0 >= 0 && lin0 + width < GRID_MAX_CELLS);
                    const unsigned end = __ldg(ce + lin0 + width);
                    B200PC_DEV_ASSERT(p <= end && end <= (unsigned)N);
                    // every ref is read once per warp, i.e. every load waits for L2 (~800 cycles): 16 in flight per thread
                    for (; p + 15 * stride < end; p += 16 * stride) {
                        float4 rr[16];
#pragma unroll
                        for (int u = 0; u < 16; ++u) rr[u] = __ldg(pts + p + u * stride);
#pragma unroll
                        for (int u = 0; u < 16; ++u) count(rr[u]);
                    }
                    for (; p + 3 * stride < end; p += 4 * stride) {
                        const float4 r0 = __ldg(pts + p), r1 = __ldg(pts + p + stride), r2 = __ldg(pts + p + 2 * stride), r3 = __ldg(pts + p + 3 * stride);
                        count(r0); count(r1); count(r2); count(r3);
                    }
                    for (; p < end; p += stride) count(__ldg(pts + p));
                }
            unsigned cum = 0;
            int bin = 0;
            for (; bin < SEED_BINS; ++bin) {
                cum += (hist[bin * (SEED_THREADS / 2)] >> shift) & 0xffffu;
                if (cum >= (unsigned)k) break;
            }
            const float e = __uint_as_float((unsigned)(base_key + bin + 1) << SEED_SHIFT);
            if (bin < SEED_BINS - 1 && e < CUDART_INF_F) tau0 = e * 1.00001f + (9.6e-7f * (3.0f * nq + 2.0f * e) + 1e-37f);
        }
        tau0 = fminf(tau0, corner);
    }
    seed[(size_t)b * S + qi] = tau0;
}

// ---------------------------------------------------------------------------------------------
// 2. distance forms.  SURVEY.md Appendix A: the reference's three roundings of |a-b|^2.
// ---------------------------------------------------------------------------------------------
struct QueryConst {  // per-query splatted constants of the EXACT evaluation
    f32x2 a0, a1, a2, a3;
};

template <int FORM>
__device__ __forceinline__ QueryConst make_query(float x, float y, float z) {
    QueryConst q;
    if (FORM == B200PC_FORM_DIRECT) {
        q.a0 = splat2(-x); q.a1 = splat2(-y); q.a2 = splat2(-z); q.a3 = splat2(torch_sq_norm(x, y, z));   // a3: filter only
    } else {
        // -2*(s.d) == s.(-2d) exactly: scaling by a power of two commutes with every rounding
        q.a0 = splat2(-2.0f * x); q.a1 = splat2(-2.0f * y); q.a2 = splat2(-2.0f * z);
        q.a3 = splat2(torch_sq_norm(x, y, z));
    }
    return q;
}

// exact distances of the two refs of a pair, bit for bit what the reference computes
template <int FORM>
__device__ __forceinline__ f32x2 pair_dist(const float4 &A, const float4 &Bv, const QueryConst &q) {
    f32x2 X = pack2(A.x, A.y), Y = pack2(A.z, A.w), Z = pack2(Bv.x, Bv.y);
    if (FORM == B200PC_FORM_DIRECT) {
        // pytorch3d: d = fma(dz,dz, fma(dy,dy, dx*dx)); (r-q)^2 == (q-r)^2 bit for bit
        f32x2 dx = add2(X, q.a0), dy = add2(Y, q.a1), dz = add2(Z, q.a2);
        f32x2 t = mul2(dx, dx);
        t = fma2(dy, dy, t);
        return fma2(dz, dz, t);
    }
    // torch CPU (MKL sgemm, K=3): dot = fma(z,z', fma(y,y', x*x')); then two separate adds.  |r|^2 is rebuilt with
    // torch's rounding, (xx + yy) + zz unfused -- the record's norm word is the deflated filter copy.  Scalar
    // __fmul_rn/__fadd_rn on purpose: ptxas 12.9 CONTRACTS mul.rn.f32x2 feeding add.rn.f32x2 into FFMA2 (seen in
    // the SASS, and in 32 failing parity tests), which the scalar .rn forms are guaranteed never to be.
    const f32x2 W = pack2(torch_sq_norm(A.x, A.z, Bv.x), torch_sq_norm(A.y, A.w, Bv.y));
    f32x2 t = mul2(X, q.a0);
    t = fma2(Y, q.a1, t);
    t = fma2(Z, q.a2, t);
    if (FORM == B200PC_FORM_REF_NORM_FIRST) {
        t = add2(t, W);         // dist += |src|^2   (src = refs at the kNN call site)
        return add2(t, q.a3);   // dist += |dst|^2
    } else {
        t = add2(t, q.a3);      // src = queries (ball query, three-NN)
        return add2(t, W);
    }
}

// Filter value of the two refs of a pair: u ~= |r|^2 - 2 q.r, three packed FMAs (b0..b2 = -2q splatted).
__device__ __forceinline__ f32x2 pair_u(const float4 &A, const float4 &Bv, f32x2 b0, f32x2 b1, f32x2 b2) {
    f32x2 t = fma2(pack2(A.x, A.y), b0, pack2(Bv.z, Bv.w));
    t = fma2(pack2(A.z, A.w), b1, t);
    return fma2(pack2(Bv.x, Bv.y), b2, t);
}
__device__ __forceinline__ float half_chunk_umin(const float4 (&H)[4], f32x2 b0, f32x2 b1, f32x2 b2) {
    float d0, d1, d2, d3;
    unpack2(pair_u(H[0], H[1], b0, b1, b2), d0, d1);
    unpack2(pair_u(H[2], H[3], b0, b1, b2), d2, d3);
    return fminf(min3(d0, d1, d2), d3);      // FMNMX returns the non-NaN operand: a NaN (padding) never wins
}
__device__ __forceinline__ float chunk_umin(const float4 (&R)[REC], f32x2 b0, f32x2 b1, f32x2 b2) {
    float d[8];
#pragma unroll
    for (int p = 0; p < 4; ++p) unpack2(pair_u(R[2 * p], R[2 * p + 1], b0, b1, b2), d[2 * p], d[2 * p + 1]);
    return min3(min3(d[0], d[1], d[2]), min3(d[3], d[4], d[5]), fminf(d[6], d[7]));
}

// Threshold of the filter.  Claim: for every ref,  dist_ref(q, r) < tau  (or <=)  implies  u < thr  (or <=), where
// dist_ref is the reference's rounded distance in any of the three forms and u is pair_u's value on the packed record.
//   eps = 2^-24, nq = fl|q|^2, w = fl|r|^2, w' = filter_norm(w) <= w (1 - 18.9 eps), a = -2q,
//   U = x a0 + y a1 + z a2 + w (real arithmetic),  M = |x a0| + |y a1| + |z a2| + w <= 2|q||r| + w <= 1.001 nq + 2.001 w.
//   * u is a 3-rounding evaluation of U - (w - w'):                                u <= U - (w - w') + 3.01 eps M
//   * forms 0/1 are 5-rounding evaluations of U + nq:                       |dist_ref - (U + nq)| <= 5.01 eps (M + nq)
//   * form 2 is a 5-rounding evaluation of |r - q|^2 (positive terms only) and |r - q|^2 differs from U + nq by the
//     rounding of the two norms:                             |dist_ref - (U + nq)| <= 5.01 eps |tau| + 4.01 eps (nq + w)
//   so dist_ref < tau  =>  u < (tau - nq) + 5.01 eps |tau| + 8.02 eps M + 5.01 eps nq - (w - w')
//                            <= (tau - nq) + 5.01 eps |tau| + 13.1 eps nq + (16.1 - 18.9) eps w.
//   * fl(tau - nq) and the final addition add at most eps (|tau| + nq) each.
//   Query-side margin needed: 7.1 eps |tau| + 15.2 eps nq; used: 7.5 eps and 18.4 eps, plus an absolute 1e-35 for
//   products that underflow.  A non-finite margin (inf / NaN coordinates) opens the filter completely -- the drain's
//   exact test decides, as the reference's own arithmetic would.
__device__ __forceinline__ float filter_threshold(float tau, float nq) {
    const float margin = 4.5e-7f * fabsf(tau) + (1.1e-6f * nq + 1e-35f);
    if (tau == -CUDART_INF_F) return tau;
    return margin < CUDART_INF_F ? (tau - nq) + margin : CUDART_INF_F;
}

// exact distances of logical pair p (refs 2p, 2p+1) of chunk `chunk` whose records start at `cb`
template <int FORM>
__device__ __forceinline__ f32x2 chunk_pair_dist(const float4 *cb, int chunk, int p, const QueryConst &q) {
    const float4 *pp = cb + 2 * (p ^ (chunk & 3));       // un-swizzle: where pair p of this chunk lives
    return pair_dist<FORM>(pp[0], pp[1], q);
}

// ---------------------------------------------------------------------------------------------
// 3. the streaming search kernel
// ---------------------------------------------------------------------------------------------
struct SearchArgs {
    const float4 *packed;  // [B][n_pad/2][2]
    const float *qry;      // [B][S][3]
    const int64_t *ref_len, *qry_len;   // [B] valid refs / queries per item (ragged batches), or null: all valid
    int N, n_pad, S, k;
    int strided;           // 1: tile t holds refs t, t + n_tiles, ... (top-k); 0: natural order (ball query)
    float r2;              // ball radius^2 (fp32)
    int debug_nodrain;     // measurement only: start with tau = -inf so nothing ever hits
    int lane_filter;       // 1: refs in registers, queries broadcast (default); 0: queries in registers, refs broadcast
    int n_split, tiles_per_split;
    // grid path (section 1b) or null: queries in cell order {x, y, z, index}, their starting thresholds, tile slot -> ref index
    const float4 *qsorted; // [B][S]
    const float *seed;     // [B][S]
    const int *perm;       // [B][n_pad]
    int interleave;        // cell-ordered queries dealt to the CTAs warp by warp (1) or in contiguous blocks (0)
    int64_t *idx_out;      // [B][S][k]   (n_split == 1)
    int32_t *idx32_out;    // same rows as 32-bit indices (host-buffer callers: halves the read-back); either may be null
    float *dist_out;       // [B][S][k] or null
    float *part_d;         // [B][S][n_split][k]  (top-k partial lists)
    int *part_i;           // [B][S][n_split][k]
    int *part_cnt;         // [B][S][n_split]     (ball partial counts)
};

// Order-preserving map fp32 -> u32 (negative expanded-form distances included), so that a
// 64-bit key (map(d) << 32 | index) realises the total order (distance, index) with one compare.
__device__ __forceinline__ uint32_t order_key(float d) {
    const uint32_t b = __float_as_uint(d);
    return b ^ (static_cast<uint32_t>(static_cast<int32_t>(b) >> 31) | 0x80000000u);
}
__device__ __forceinline__ float key_to_float(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
}
constexpr unsigned long long HEAP_SENTINEL = 0xFF800000FFFFFFFFull;  // (+inf, max index)

__device__ __forceinline__ unsigned long long lds_u64(uint32_t a) {
    unsigned long long v;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_u64(uint32_t a, unsigned long long v) {
    asm volatile("st.shared.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory");
}

// max-heap of 64-bit keys in shared memory: element e of this query lives at byte address hb + e*SB.
// Put `nk` at the root of a heap holding nB/SB elements and sift it down (depth ceil(log2 n): every
// lane of a warp runs the same short loop).  PADDED = the element right after the heap is readable and
// holds key 0, so the right child needs no bounds check (true while streaming, false during heapsort).
template <bool PADDED>
__device__ __forceinline__ void heap_sift_root(uint32_t hb, uint32_t SB, uint32_t nB, unsigned long long nk) {
    uint32_t pos = 0;
    while (true) {
        const uint32_t l = 2 * pos + SB;
        if (l >= nB) break;
        unsigned long long kc = lds_u64(hb + l);
        uint32_t c = l;
        if (PADDED || l + SB < nB) {
            const unsigned long long kr = lds_u64(hb + l + SB);
            if (kr > kc) { kc = kr; c = l + SB; }
        }
        if (kc <= nk) break;
        sts_u64(hb + pos, kc);
        pos = c;
    }
    sts_u64(hb + pos, nk);
}

constexpr int CAND_CAP = 8;   // per-query buffer: one u16 entry (chunk << 8 | candidate mask) per hit chunk of a drain pass

// Exact distance of ONE ref of the tile (ref number `off`), scalar: the same IEEE operations in the same order as
// pair_dist (explicit .rn intrinsics, so nothing is contracted), a third of its instructions.  (ax, ay, az) is -2q for
// the expanded forms and -q for the direct form; nq = fl|q|^2.
template <int FORM>
__device__ __forceinline__ float ref_dist(const float4 *tp, int off, float ax, float ay, float az, float nq) {
    const int chunk = off >> 3;
    const float *rec = reinterpret_cast<const float *>(tp + chunk * REC + 2 * (((off >> 1) ^ chunk) & 3)) + (off & 1);
    const float x = rec[0], y = rec[2], z = rec[4];
    if (FORM == B200PC_FORM_DIRECT) {
        const float dx = __fadd_rn(x, ax), dy = __fadd_rn(y, ay), dz = __fadd_rn(z, az);
        return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
    }
    const float t = __fmaf_rn(z, az, __fmaf_rn(y, ay, __fmul_rn(x, ax)));
    const float w = torch_sq_norm(x, y, z);
    if (FORM == B200PC_FORM_REF_NORM_FIRST) return __fadd_rn(__fadd_rn(t, w), nq);
    return __fadd_rn(__fadd_rn(t, nq), w);
}

// 32 x 32 bit-matrix transpose across a warp: on return, bit i of lane l's word is bit l of lane i's input word
// (five butterfly stages; replaces 32 x (ballot + compare + select)).
__device__ __forceinline__ uint32_t warp_transpose32(uint32_t x, int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const uint32_t m = s == 16 ? 0x0000FFFFu : s == 8 ? 0x00FF00FFu : s == 4 ? 0x0F0F0F0Fu : s == 2 ? 0x33333333u : 0x55555555u;
        const uint32_t other = __shfl_xor_sync(0xffffffffu, x, s);
        x = (lane & s) == 0 ? ((x & m) | ((other << s) & ~m)) : ((x & ~m) | ((other >> s) & m));
    }
    return x;
}

constexpr int MAX_WARPS = 16;
constexpr int FILTER_UNROLL = 8;   // queries of the lane filter in flight per warp
constexpr int MAX_WARPS_Q1 = 14;   // Q=1 kernels are compiled for two resident CTAs of 14 warps (<= 72 registers)

// blockDim.x = warps * 32 is a RUNTIME value so that the planner can size the grid as whole waves of resident CTAs.
template <int FORM, int MODE, int Q>
__global__ void __launch_bounds__(Q == 1 ? MAX_WARPS_Q1 * 32 : MAX_WARPS * 32, Q == 1 ? 2 : 1) search_kernel(const SearchArgs P) {
    const int NCW = (int)(blockDim.x >> 5);       // warps
    const int NCT = NCW * 32;                     // threads
    const int QPB = NCT * Q;                      // queries per block
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(128) unsigned char smem[];
    const float4 *tiles = reinterpret_cast<const float4 *>(smem);
    const uint32_t bar_base = smem_u32(smem + STAGES * TILE_BYTES);   // full[s] at +8s, empty[s] at +8(STAGES+s)
    int *issued = reinterpret_cast<int *>(smem + STAGES * TILE_BYTES + 8 * 2 * STAGES);   // tiles issued so far
    int *item_nt = issued + 1;                    // tiles of this batch item (slot_to_ref in the drain; kept out of the registers)
    // query records [QPB] float4 {-2qx, -2qy, -2qz, filter threshold} (read by the lane filter), then
    // top-k: heap [k+1][QPB] u64 and candidate buffer [CAND_CAP][QPB] u16.   ball: list [k][QPB] u32
    float4 *qrec = reinterpret_cast<float4 *>(smem + STAGES * TILE_BYTES + BAR_BYTES);
    unsigned long long *heap_all = reinterpret_cast<unsigned long long *>(qrec + QPB);
    unsigned short *cand_all = reinterpret_cast<unsigned short *>(heap_all + (size_t)(P.k + 1) * QPB);
    int *list_all = reinterpret_cast<int *>(heap_all);

    const int lane = threadIdx.x & 31;
    const int b = blockIdx.y, split = blockIdx.z;
    // Ragged items: the tile loop stops at the item's own tiles, and a CTA that holds no valid query (its lowest query,
    // blockIdx.x * QPB or, dealt warp by warp, 32 * blockIdx.x, is past s_b) visits none.  A range without tiles of the
    // item still writes its partial list of every row: all sentinel keys, which the merge turns into -1 / +inf.
    const int tile0 = split * P.tiles_per_split;
    int ntiles, s_b = item_len(P.qry_len, b, P.S);
    {
        const int nt_b = item_tiles(item_len(P.ref_len, b, P.N));
        const int first_q = P.qsorted && P.interleave ? (int)blockIdx.x * 32 : (int)blockIdx.x * QPB;
        ntiles = min(tile0 + P.tiles_per_split, first_q < s_b ? nt_b : 0) - tile0;     // <= 0: no tile
        if (threadIdx.x == 0) *item_nt = nt_b;
    }
    const int k = P.k;
    const char *src = reinterpret_cast<const char *>(P.packed) + ((size_t)b * P.n_pad + (size_t)tile0 * TILE) * 16;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bar_base + 8 * s, 1);
            mbar_init(bar_base + 8 * (STAGES + s), NCW);
        }
        mbar_fence_init();
        const int pre = ntiles < STAGES ? ntiles : STAGES;
        for (int t = 0; t < pre; ++t) {
            mbar_expect_tx(bar_base + 8 * t, TILE_BYTES);
            bulk_g2s(smem_u32(smem + t * TILE_BYTES), src + (size_t)t * TILE_BYTES, TILE_BYTES, bar_base + 8 * t);
        }
        *issued = pre;
    }
    __syncthreads();

    const int ct = threadIdx.x;  // 0 .. NCT-1
    // Which query a thread owns.  Cell-ordered queries: contiguous blocks of the order by default (a CTA = a patch of space;
    // measured 1-4 % faster on the lidar-like clouds), or dealt out warp by warp (B200PC_INTERLEAVE=1: warp w of CTA x takes
    // the (w * gridDim.x + x)-th group of 32, so that no CTA holds all the sparse, loosely bounded regions).
    auto query_of = [&](int j) {
        return P.qsorted && P.interleave ? (((j * NCW + (ct >> 5)) * (int)gridDim.x + (int)blockIdx.x) << 5) + lane : (int)blockIdx.x * QPB + j * NCT + ct;
    };
    // Per-query state that stays in registers across the filter: tau (exact threshold) and the ball count.  Everything
    // else about a query is rebuilt from its 16-byte shared-memory record at the start of a drain.
    // A padded query of a ragged item (qi >= s_b) is not loaded and starts from tau = -inf: nothing ever hits, its row is
    // written from the sentinel heap (-1 / +inf), and a warp with no valid query skips the filters altogether.
    float tau[Q];
    int cnt[Q];
    bool live_any = false;
#pragma unroll
    for (int j = 0; j < Q; ++j) {
        const int qi = query_of(j);
        const bool live = qi < s_b;
        live_any = live_any || live;
        float x = 0.f, y = 0.f, z = 0.f;
        if (live) {
            if (P.qsorted) {
                const float4 qv = __ldg(P.qsorted + (size_t)b * P.S + qi);
                x = qv.x; y = qv.y; z = qv.z;
            } else {
                const float *qp = P.qry + ((size_t)b * P.S + qi) * 3;
                x = qp[0]; y = qp[1]; z = qp[2];
            }
        }
        cnt[j] = 0;
        if (MODE == MODE_TOPK) {
            tau[j] = P.debug_nodrain || !live ? -CUDART_INF_F : CUDART_INF_F;
            // warm start: an upper bound of the k-th distance from grid_seed_kernel
            if (P.seed && !P.debug_nodrain && live) tau[j] = __ldg(P.seed + (size_t)b * P.S + qi);
            for (int e = 0; e < k; ++e) heap_all[e * QPB + j * NCT + ct] = HEAP_SENTINEL;
            heap_all[k * QPB + j * NCT + ct] = 0ull;   // pad: the smallest key, never selected as a child
        } else {
            tau[j] = P.r2;
        }
        qrec[j * NCT + ct] = make_float4(-2.0f * x, -2.0f * y, -2.0f * z, filter_threshold(tau[j], torch_sq_norm(x, y, z)));
    }

    bool warp_cold = true;
    if (MODE == MODE_TOPK) {
        bool cold = false;
#pragma unroll
        for (int j = 0; j < Q; ++j) cold = cold || tau[j] == CUDART_INF_F;
        warp_cold = __any_sync(FULL, cold);
    }
    const bool warp_live = MODE == MODE_BALL || __any_sync(FULL, live_any);
    for (int t = 0; t < ntiles; ++t) {
        const int s = t % STAGES;
        mbar_wait(bar_base + 8 * s, (t / STAGES) & 1);
        const float4 *tp = tiles + (size_t)s * TILE;
        const int tile_ref0 = (tile0 + t) * TILE;

        // ---- filter A (broadcast): queries in registers, every lane walks the same nch <= 32 chunks from c ----
        auto filter_bcast = [&](const int c, const int nch, uint32_t (&mask)[Q][2]) {
            f32x2 b0[Q], b1[Q], b2[Q];
            float thr[Q];
#pragma unroll
            for (int j = 0; j < Q; ++j) {
                const float4 qv = qrec[j * NCT + ct];
                b0[j] = splat2(qv.x); b1[j] = splat2(qv.y); b2[j] = splat2(qv.z); thr[j] = qv.w;
                mask[j][0] = 0u; mask[j][1] = 0u;
            }
            // register double buffer: half a chunk is requested ahead of its use and a warp-level memory barrier
            // pins those loads above the math of the current group (ptxas would sink every LDS next to its use).
            const float4 *cp = tp + c * REC;
            float4 H[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) H[p] = cp[p];
            uint32_t bit = 1u;
            for (int cc = 0; cc < nch; ++cc, bit <<= 1) {
                float4 N1[4];
#pragma unroll
                for (int p = 0; p < 4; ++p) N1[p] = cp[4 + p];
                __syncwarp();
                float ma[Q];
#pragma unroll
                for (int j = 0; j < Q; ++j) ma[j] = half_chunk_umin(H, b0[j], b1[j], b2[j]);
                cp += REC;       // one chunk past the tile end is still inside the ring / barrier block: harmless
                float4 N2[4];
#pragma unroll
                for (int p = 0; p < 4; ++p) N2[p] = cp[p];
                __syncwarp();
#pragma unroll
                for (int j = 0; j < Q; ++j) {
                    const float m = fminf(ma[j], half_chunk_umin(N1, b0[j], b1[j], b2[j]));
                    const bool hit = MODE == MODE_TOPK ? (m < thr[j]) : (m <= thr[j]);
                    if (hit) mask[j][0] |= bit;
                }
#pragma unroll
                for (int p = 0; p < 4; ++p) H[p] = N2[p];
            }
        };

        // ---- filter B (lanes): lane l keeps chunk c0+32h+l (8 refs) in registers and the warp's 32*Q queries are
        // broadcast one at a time from their shared-memory records; the ballot of query i is exactly the 32-chunk
        // hit mask that lane i needs for its drain.
        auto filter_lanes = [&](const int c0, uint32_t (&mask)[Q][2]) {
#pragma unroll
            for (int j = 0; j < Q; ++j) { mask[j][0] = 0u; mask[j][1] = 0u; }
            __syncwarp();                                     // the owners' threshold updates are visible
#pragma unroll 1
            for (int h = 0; c0 + 32 * h < CHUNKS_PER_TILE; ++h) {
                float4 R[REC];
                {
                    // lane-distinct 16-byte loads: rotate the pair slot by the lane so that a quarter warp covers
                    // four different 32-byte slots (2-way instead of 32-way conflicts).  The pair ORDER inside a
                    // chunk does not matter to a min; the two records of a pair stay together.
                    const float4 *cb = tp + (c0 + 32 * h + lane) * REC;
                    const int rot = (lane & 3) << 1;
#pragma unroll
                    for (int p = 0; p < REC; ++p) R[p] = cb[p ^ rot];
                }
#pragma unroll
                for (int j = 0; j < Q; ++j) {
                    const int s0 = j * NCT + (ct & ~31);
                    uint32_t mine = 0u;                       // bit l: my chunk holds a candidate of the warp's l-th query
#pragma unroll FILTER_UNROLL
                    for (int l = 0; l < 32; ++l) {
                        const float4 qv = qrec[s0 + l];
                        const float m = chunk_umin(R, splat2(qv.x), splat2(qv.y), splat2(qv.z));
                        const bool hit = MODE == MODE_TOPK ? (m < qv.w) : (m <= qv.w);
                        if (hit) mine |= 1u << l;
                    }
                    mine = warp_transpose32(mine, lane);      // bit i: chunk c0+32h+i holds a candidate of MY query
                    if (h == 0) mask[j][0] = mine; else mask[j][1] = mine;
                }
            }
        };

        // ---- drain, warp-synchronous so that the lanes' slow work overlaps instead of serialising ----
        auto drain = [&](const int c, uint32_t (&mask)[Q][2]) {
#pragma unroll
            for (int j = 0; j < Q; ++j) {
                uint32_t m0 = mask[j][0], m1 = mask[j][1];
                const int slot = j * NCT + ct;
                const float4 qv = qrec[slot];
                // x = -0.5 * (-2x) exactly, so these are the constants the coordinates themselves would give
                const float nq = torch_sq_norm(0.5f * qv.x, 0.5f * qv.y, 0.5f * qv.z);
                if (MODE == MODE_TOPK) {
                    const float ex = FORM == B200PC_FORM_DIRECT ? 0.5f * qv.x : qv.x, ey = FORM == B200PC_FORM_DIRECT ? 0.5f * qv.y : qv.y,
                                ez = FORM == B200PC_FORM_DIRECT ? 0.5f * qv.z : qv.z;
                    const uint32_t hb = smem_u32(heap_all + slot), SB = (uint32_t)QPB * 8u;
                    unsigned short *cand = cand_all + slot;
                    const f32x2 b0 = splat2(qv.x), b1 = splat2(qv.y), b2 = splat2(qv.z);
                    float thr = qv.w;
                    while (__any_sync(FULL, (m0 | m1) != 0u)) {
                        // phase 1: every lane revisits its r-th hit chunk; the refs that pass the filter test on their
                        // own are only recorded, as ONE entry (chunk << 8 | 8-bit mask), at most CAND_CAP per pass.
                        int nc = 0;
                        while (__any_sync(FULL, (m0 | m1) != 0u && nc < CAND_CAP)) {
                            if ((m0 | m1) != 0u && nc < CAND_CAP) {
                                int cc;
                                if (m0 != 0u) { cc = __ffs(m0) - 1; m0 &= m0 - 1; }
                                else { cc = 32 + __ffs(m1) - 1; m1 &= m1 - 1; }
                                B200PC_DEV_ASSERT(c + cc >= 0 && c + cc < CHUNKS_PER_TILE && nc < CAND_CAP);
                                const float4 *dp = tp + (c + cc) * REC;
                                // logical pair p lives in pair slot p ^ (chunk & 3): lanes on different chunks spread over the banks
                                const float4 *dq = dp + 2 * ((c + cc) & 3);
                                float u[8];
#pragma unroll
                                for (int p = 0; p < 4; ++p) {
                                    const float4 *pp = reinterpret_cast<const float4 *>(reinterpret_cast<uintptr_t>(dq) ^ (uintptr_t)(p * 32));
                                    unpack2(pair_u(pp[0], pp[1], b0, b1, b2), u[2 * p], u[2 * p + 1]);
                                }
                                uint32_t cm = 0u;
#pragma unroll
                                for (int i = 0; i < 8; ++i) cm |= (u[i] < thr) ? (1u << i) : 0u;
                                if (cm != 0u) { cand[nc * QPB] = (unsigned short)((cc << 8) | cm); ++nc; }
                            }
                        }
                        // phase 2: all lanes insert their next candidate together (index order is preserved)
                        uint32_t cur = 0u;
                        int e = 0, base = 0;
                        while (true) {
                            if (cur == 0u && e < nc) {
                                const uint32_t v = cand[e * QPB];
                                ++e;
                                cur = v & 0xffu;
                                base = (c + (int)(v >> 8)) * CHUNK;
                            }
                            if (!__any_sync(FULL, cur != 0u)) break;
                            if (cur != 0u) {
                                const int off = base + __ffs(cur) - 1;
                                B200PC_DEV_ASSERT(off >= 0 && off < TILE && tile_ref0 + off < P.n_pad);
                                cur &= cur - 1;
                                const float d = ref_dist<FORM>(tp, off, ex, ey, ez, nq);
                                // only a finite distance is a candidate: while the heap still holds its (+inf, 0xffffffff)
                                // sentinels tau is +inf, and a +inf distance that the filter let through (a query such
                                // as (+inf, 0, 0), whose filter value is -inf for refs with x > 0) would enter with a
                                // real index.  NaN fails d <= tau, and no form yields -inf.
                                if (d <= tau[j] && d < CUDART_INF_F) {
                                    // the refs are not visited in index order: an EQUAL distance still wins with a lower index
                                    // than the root's (rare; only then is the root read)
                                    const uint32_t ri = P.perm ? (uint32_t)__ldg(P.perm + (size_t)b * P.n_pad + tile_ref0 + off)
                                                               : (uint32_t)slot_to_ref(tile_ref0 + off, P.strided, *item_nt);
                                    B200PC_DEV_ASSERT(ri < (uint32_t)P.n_pad);
                                    if (d < tau[j] || ri < (uint32_t)lds_u64(hb)) {
                                        heap_sift_root<true>(hb, SB, (uint32_t)k * SB, ((unsigned long long)order_key(d) << 32) | ri);
                                        // never above the starting bound: the root is still the +inf sentinel until k refs are in
                                        tau[j] = fminf(tau[j], key_to_float((uint32_t)(lds_u64(hb) >> 32)));
                                    }
                                }
                            }
                        }
                        thr = filter_threshold(tau[j], nq);   // the next pass of this drain filters with the tightened threshold
                    }
                    // publish the tightened threshold to the filters
                    reinterpret_cast<float *>(qrec + slot)[3] = filter_threshold(tau[j], nq);
                } else {
                    const QueryConst qcj = make_query<FORM>(-0.5f * qv.x, -0.5f * qv.y, -0.5f * qv.z);
                    int *list = list_all + slot;
                    while (__any_sync(FULL, (m0 | m1) != 0u)) {
                        if ((m0 | m1) != 0u) {
                            int cc;
                            if (m0 != 0u) { cc = __ffs(m0) - 1; m0 &= m0 - 1; }
                            else { cc = 32 + __ffs(m1) - 1; m1 &= m1 - 1; }
                            const int off0 = (c + cc) * CHUNK;
                            B200PC_DEV_ASSERT(c + cc >= 0 && c + cc < CHUNKS_PER_TILE);
                            const float4 *dp = tp + (c + cc) * REC;
                            float d[8];
#pragma unroll
                            for (int p = 0; p < 4; ++p) unpack2(chunk_pair_dist<FORM>(dp, c + cc, p, qcj), d[2 * p], d[2 * p + 1]);
#pragma unroll
                            for (int i = 0; i < 8; ++i)
                                if (d[i] <= tau[j] && cnt[j] < k) {
                                    B200PC_DEV_ASSERT(tile_ref0 + off0 + i < P.N);      // a padding record never passes the exact test
                                    list[cnt[j] * QPB] = tile_ref0 + off0 + i; ++cnt[j];
                                }
                            if (cnt[j] == k) {   // this query is complete: nothing can hit any more
                                tau[j] = -CUDART_INF_F; m0 = 0u; m1 = 0u;
                                reinterpret_cast<float *>(qrec + slot)[3] = -CUDART_INF_F;
                            }
                        }
                    }
                }
            }
        };

        // Schedule.  First tile of a split (top-k only): the broadcast filter with a drain after 2,2,4,8,16 chunks so
        // that tau tightens quickly, then the lane filter on the second half.  Every other tile: the lane filter on
        // both halves (two 32-bit hit masks per query) and ONE drain.
        uint32_t mask[Q][2];
        // the warm-up schedule of the first tile is only needed by warps that hold a query starting from tau = +inf
        const bool warm = MODE == MODE_TOPK && t == 0 && warp_cold;
        int c = warp_live ? 0 : CHUNKS_PER_TILE;         // a warp without a valid query only releases the stages
        if (MODE == MODE_BALL) {
            // a ball is "the first nsample refs by index": once every query of the warp has its nsample refs, no later ref
            // can change anything -- the warp only keeps releasing stages so that the other warps' tiles keep coming
            bool full = true;
#pragma unroll
            for (int j = 0; j < Q; ++j) full = full && cnt[j] == k;
            if (__all_sync(FULL, full)) c = CHUNKS_PER_TILE;
        }
        while (c < CHUNKS_PER_TILE) {
            int nch = CHUNKS_PER_TILE - c;
            if (P.lane_filter && !(warm && c < 32)) {
                filter_lanes(c, mask);
            } else {
                nch = warm ? (c < 2 ? 2 : c) : 32;
                if (nch > 32) nch = 32;
                filter_bcast(c, nch, mask);
            }
            drain(c, mask);
            c += nch;
        }

        // ---- release the stage; the warp that completes the release refills it ----
        __syncwarp();
        if (lane == 0) {
            const uint32_t ebar = bar_base + 8 * (STAGES + s);
            mbar_arrive(ebar);
            const int nxt = t + STAGES;                 // the tile that will reuse this stage
            if (nxt < ntiles && mbar_test(ebar, (t / STAGES) & 1)) {
                if (atomicCAS(issued, nxt, nxt + 1) == nxt) {
                    mbar_expect_tx(bar_base + 8 * s, TILE_BYTES);
                    bulk_g2s(smem_u32(smem + s * TILE_BYTES), src + (size_t)nxt * TILE_BYTES, TILE_BYTES, bar_base + 8 * s);
                }
            }
        }
    }

    // ---------------- results ----------------
    s_b = item_len(P.qry_len, b, P.S);
#pragma unroll
    for (int j = 0; j < Q; ++j) {
        const int qi = query_of(j);
        const int slot = j * NCT + ct;
        if (MODE == MODE_TOPK) {
            // in-place heapsort: ascending (distance, index) order
            const uint32_t hb = smem_u32(heap_all + slot), SB = (uint32_t)QPB * 8u;
            for (int n = k; n > 1; --n) {
                const unsigned long long top = lds_u64(hb);
                const unsigned long long last = lds_u64(hb + (uint32_t)(n - 1) * SB);
                heap_sift_root<false>(hb, SB, (uint32_t)(n - 1) * SB, last);
                sts_u64(hb + (uint32_t)(n - 1) * SB, top);
            }
        }
        if (qi >= P.S) continue;
        // cell-ordered queries: the result goes to the caller's row.  Only the s_b valid queries are in the sorted copy, so
        // the sorted positions s_b .. S-1 are free and take the padded rows s_b .. S-1 one to one.
        const size_t row = (size_t)b * P.S + (P.qsorted && qi < s_b ? __float_as_int(__ldg(&P.qsorted[(size_t)b * P.S + qi].w)) : qi);
        B200PC_DEV_ASSERT(row >= (size_t)b * P.S && row < (size_t)(b + 1) * P.S);
        if (P.n_split == 1) {
            int64_t *io = P.idx_out ? P.idx_out + row * k : nullptr;
            int32_t *io32 = P.idx32_out ? P.idx32_out + row * k : nullptr;
            if (MODE == MODE_TOPK) {
                float *dout = P.dist_out ? P.dist_out + row * k : nullptr;
                for (int e = 0; e < k; ++e) {
                    const unsigned long long key = heap_all[e * QPB + slot];
                    if (io) io[e] = (int64_t)(int32_t)(uint32_t)key;     // unfilled slot (fewer than k candidates): -1, distance +inf
                    if (io32) io32[e] = (int32_t)(uint32_t)key;
                    if (dout) dout[e] = key_to_float((uint32_t)(key >> 32));
                }
            } else {
                const int *list = list_all + slot;
                const int first = cnt[j] > 0 ? list[0] : P.N;
                for (int e = 0; e < k; ++e) {
                    const int v = e < cnt[j] ? list[e * QPB] : first;
                    if (io) io[e] = v;
                    if (io32) io32[e] = v;
                }
            }
        } else {
            const size_t prow = (row * P.n_split + split) * k;
            if (MODE == MODE_TOPK) {
                for (int e = 0; e < k; ++e) {
                    const unsigned long long key = heap_all[e * QPB + slot];
                    P.part_d[prow + e] = key_to_float((uint32_t)(key >> 32));
                    P.part_i[prow + e] = (int)(uint32_t)key;
                }
            } else {
                const int *list = list_all + slot;
                P.part_cnt[row * P.n_split + split] = cnt[j];
                for (int e = 0; e < cnt[j]; ++e) P.part_i[prow + e] = list[e * QPB];
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// 4. merge of partial lists (only when the ref range was split)
// ---------------------------------------------------------------------------------------------
// One WARP per query row: lane s holds the head of partial list s (n_split <= 32) as a 64-bit key (order(d) << 32 | index),
// k rounds of warp arg-min (two REDUX + a ballot), the winner advances.  Round 1 used a thread per row walking all heads:
// 43 us for the 16 384 x 8 x 16 lists of a B=1 fusion search, on the critical path of the PointINet frame; this takes ~10 us.
// The splits interleave the index ranges (strided tiles), so ties are broken on the index by the key itself.
constexpr unsigned long long MERGE_DONE = ~0ull;     // an exhausted list: larger than the sentinel key (+inf, 0xffffffff)

__global__ void __launch_bounds__(256) merge_topk_kernel(const float *__restrict__ part_d, const int *__restrict__ part_i, int rows,
                                                         int n_split, int k, int64_t *__restrict__ idx_out,
                                                         int32_t *__restrict__ idx32_out, float *__restrict__ dist_out) {
    const int lane = threadIdx.x & 31;
    const int row = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (row >= rows) return;
    const float *pd = part_d + ((size_t)row * n_split + lane) * k;
    const int *pi = part_i + ((size_t)row * n_split + lane) * k;
    int h = 0;
    unsigned long long key = lane < n_split ? (((unsigned long long)order_key(pd[0]) << 32) | (unsigned)pi[0]) : MERGE_DONE;
    unsigned int out_i = 0u, out_d = 0u;
    for (int o = 0; o < k; ++o) {
        const unsigned int hi = (unsigned int)(key >> 32), lo = (unsigned int)key;
        const unsigned int mh = __reduce_min_sync(0xffffffffu, hi);
        const unsigned int ml = __reduce_min_sync(0xffffffffu, hi == mh ? lo : 0xffffffffu);
        const int win = __ffs(__ballot_sync(0xffffffffu, hi == mh && lo == ml)) - 1;
        if ((o & 31) == lane) { out_i = ml; out_d = mh; }
        if (lane == win) {
            ++h;
            key = h < k ? (((unsigned long long)order_key(pd[h]) << 32) | (unsigned)pi[h]) : MERGE_DONE;
        }
        if ((o & 31) == 31 || o == k - 1) {                            // flush up to 32 results with coalesced stores
            const int oo = (o & ~31) + lane;
            if (oo <= o) {
                if (idx_out) idx_out[(size_t)row * k + oo] = (int64_t)(int32_t)out_i;
                if (idx32_out) idx32_out[(size_t)row * k + oo] = (int32_t)out_i;
                if (dist_out) dist_out[(size_t)row * k + oo] = key_to_float(out_d);
            }
        }
    }
}

// One warp per query row: lane s owns split s; an exclusive prefix sum of the counts places every split's hits.
__global__ void __launch_bounds__(256) merge_ball_kernel(const int *__restrict__ part_i, const int *__restrict__ part_cnt, int rows,
                                                         int n_split, int k, int N, int64_t *__restrict__ idx_out,
                                                         int32_t *__restrict__ idx32_out) {
    const int lane = threadIdx.x & 31;
    const int row = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (row >= rows) return;
    const int c = lane < n_split ? part_cnt[(size_t)row * n_split + lane] : 0;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += up;
    }
    const int off = incl - c;
    const int *pi = part_i + ((size_t)row * n_split + lane) * k;
    const unsigned nonempty = __ballot_sync(0xffffffffu, c > 0);
    const int first_lane = __ffs(nonempty) - 1;
    int first = N;                                                        // empty ball: the reference's sentinel
    if (first_lane >= 0) first = __shfl_sync(0xffffffffu, c > 0 ? pi[0] : 0, first_lane);
    int total = __shfl_sync(0xffffffffu, incl, 31);
    total = total < k ? total : k;
    int64_t *o = idx_out ? idx_out + (size_t)row * k : nullptr;
    int32_t *o32 = idx32_out ? idx32_out + (size_t)row * k : nullptr;
    for (int e = 0; e < c && off + e < k; ++e) {
        const int v = pi[e];
        if (o) o[off + e] = v;
        if (o32) o32[off + e] = v;
    }
    for (int e = total + lane; e < k; e += 32) {
        if (o) o[e] = first;
        if (o32) o32[e] = first;
    }
}

// ---------------------------------------------------------------------------------------------
// 5. planning + launch
// ---------------------------------------------------------------------------------------------
// per-query shared-memory bytes: 16-byte query record, then  top-k: u64 heap [k] + u16 candidate buffer [CAND_CAP];  ball: u32 list [nsample]
static size_t query_bytes(int k, int mode) { return 16 + (mode == MODE_TOPK ? (size_t)(k + 1) * 8 + (size_t)CAND_CAP * 2 : (size_t)k * 4); }
static const size_t kMaxSmem = 227 * 1024;
static const size_t kFixedSmem = (size_t)STAGES * TILE_BYTES + BAR_BYTES;

// Choose {queries per thread, consumer warps, ref split} so that the grid is (close to) a whole
// number of waves of resident CTAs: CTA count = B * ceil(S / q_per_block) * n_split against
// slots = SMs * CTAs-per-SM.  Among the candidates the one with the best wave efficiency wins;
// ties go to more resident warps.
// warm start only where it pays: the grid costs a memset, a bounding-box kernel and one atomic per ref
// 0: no grid; 1: counts + starting thresholds only (4 small launches); 2: refs and queries sorted by cell as well (7 launches)
static int grid_mode(int B, int N, int S, int k) {
    const int g = tuning().grid;
    if (g <= 0) return 0;
    if (g == 2 || g == 3) return g - 1;                        // forced: 2 = thresholds only, 3 = sorted
    // measured (tools/grid_probe.py): a nearest-neighbour search (k = 1) inserts too little to pay for any of it; the sorted
    // variant wins where the drain is a large part of a long search (C2: -12 %, k = 64: -28 %) and loses its three extra
    // launches on the short ones (fusion search of one frame pair, three-NN)
    if (k < 3 || N < 2048 || (long)B * N * S < GRID_MIN_PAIRS) return 0;
    return k >= 8 && (long)B * N * S >= GRID_SORT_MIN_PAIRS ? 2 : 1;
}

bool plan_search(int B, int N, int S, int k, int mode, SearchPlan *pl) {
    const int sms = sm_count();
    const size_t qb = query_bytes(k, mode);
    if (kFixedSmem + 32 * qb > kMaxSmem) return false;   // not even one warp of queries fits
    pl->n_pad = (int)align_up((size_t)N, TILE);
    pl->n_tiles = pl->n_pad / TILE;

    const Tuning &tn = tuning();                      // tuning / debugging overrides (cached; not part of the ABI)
    const int force_q = tn.force_q, force_w = tn.force_warps > 0 ? tn.force_warps : 0;
    // A forced split is evaluated as the only candidate (not filtered out of the 1, 2, 3, 4, 8, ... sequence below, which
    // would leave no candidate for 5 or for a tile count outside it), clamped to the tile count and to the 32 lists one
    // merge warp holds.
    int force_split = tn.force_split > 0 ? tn.force_split : 0;
    if (force_split > pl->n_tiles) force_split = pl->n_tiles;
    if (force_split > MAX_SPLIT) force_split = MAX_SPLIT;

    double best_score = -1.0;
    int best_q = 1, best_w = 1, best_split = 1;
    const double lnk = 1.0 + log(fmax(1.0, (double)N / k));
    for (int q = 1; q <= 2; ++q) {
        // With the lane filter the queries per thread only matter to the drain, where two queries per lane drain one
        // after the other with half the resident warps: measured 20-40 % slower on every shape, so Q=2 is kept for
        // A/B measurements (B200PC_FORCE_Q=2) only.
        if (force_q ? q != force_q : q != 1) continue;
        // A forced warp count is clamped once, to what one resident CTA can hold, and then only candidates that can run
        // exactly that many warps compete: a smaller count at more CTAs per SM must not replace it unannounced.  One CTA
        // per SM always passes the register check below.
        int wforce = force_w;
        if (wforce) {
            const int cap = q == 1 ? MAX_WARPS_Q1 : MAX_WARPS;
            const size_t budget1 = kMaxSmem - 1024;
            const int fit1 = budget1 > kFixedSmem ? (int)((budget1 - kFixedSmem) / (32 * q * qb)) : 0;
            if (wforce > cap) wforce = cap;
            if (wforce > fit1) wforce = fit1 > 1 ? fit1 : 1;
        }
        for (int c = 1; c <= 8; ++c) {                       // target CTAs per SM
            const size_t budget = kMaxSmem / c - 1024;          // ~1 KB per resident CTA is reserved by the system
            if (budget <= kFixedSmem + 32 * q * qb) continue;
            int wmax = (int)((budget - kFixedSmem) / (32 * q * qb));
            if (wmax > (q == 1 ? MAX_WARPS_Q1 : MAX_WARPS)) wmax = q == 1 ? MAX_WARPS_Q1 : MAX_WARPS;
            const long slots = (long)sms * c;
            for (int split = force_split ? force_split : 1; split <= MAX_SPLIT && split <= pl->n_tiles;
                 split = force_split ? MAX_SPLIT + 1 : split < 4 ? split + 1 : split * 2) {
                // queries per CTA if the work items (query block x ref split) of each batch item fill the slots
                long ipb = slots / ((long)B * split);           // query blocks per batch item, one wave
                if (ipb < 1) ipb = 1;
                int w = (int)((((long)S + ipb - 1) / ipb + 32 * q - 1) / (32 * q));
                if (w < 1) w = 1;
                if (w > wmax) w = wmax;
                if (wforce) {
                    if (wforce > wmax) continue;
                    w = wforce;
                }
                // register file: 64K registers per SM, <= 128 (Q=2) / <= 72 (Q=1) per thread
                if ((long)w * 32 * c * (q == 2 ? 128 : 72) > 65536) continue;
                const long items = (long)B * (((long)S + 32L * q * w - 1) / (32L * q * w));
                const int tps = (pl->n_tiles + split - 1) / split;
                const int real_split = (pl->n_tiles + tps - 1) / tps;
                const long ctas = items * real_split;
                const long waves = (ctas + slots - 1) / slots;
                const double wave_eff = (double)ctas / (double)(waves * slots);
                const double pad_eff = (double)B * S / ((double)items * 32 * q * w);
                // resident warps per SM: below ~16 the SM cannot hide the drain's latency (and below 4 it idles)
                const double resident = fmin((double)c, (double)ctas / sms) * w;
                const double occ = pow(fmin(1.0, resident / 16.0), 0.8);
                // A split repeats the warm-up of the k-best list in every ref range: ~k(1+ln(n/k)) inserts each, and one
                // insert costs about as much as filtering 130 refs (calibrated at C2, where the blind drain is half the
                // kernel).  For k = 1 the inserts are noise next to the filter, so splitting to fill the SMs is nearly free
                // (k=1, 65536 queries x 65536 refs: 0.97 -> 0.86 ms with 4 ranges; the former model, which weighed the
                // drain as half the work whatever k, kept it in one range on 147 CTAs of 14 warps).
                const double ins = 130.0 * k;
                const double work = ((double)N + ins * real_split * (1.0 + log(fmax(1.0, (double)N / real_split / k)))) / ((double)N + ins * lnk) +
                                    (mode == MODE_TOPK ? 0.05 * (real_split - 1) : real_split > 1 ? 0.05 : 0.0);   // merge + one more k-best warm-up per range
                const double score = wave_eff * pad_eff * occ / work + 1e-5 * resident;
                if (score > best_score) { best_score = score; best_q = q; best_w = w; best_split = real_split; }
            }
        }
    }
    // No candidate: the one-warp plan below, which the check at the top allows -- unless Q = 2 was forced (or a Q that does
    // not exist), which must not quietly run as Q = 1.
    if (best_score < 0.0 && force_q > 1) return false;
    pl->q_per_thread = best_q;
    pl->consumer_warps = best_w;
    pl->q_per_block = best_q * best_w * 32;
    pl->tiles_per_split = (pl->n_tiles + best_split - 1) / best_split;
    pl->n_split = (pl->n_tiles + pl->tiles_per_split - 1) / pl->tiles_per_split;
    pl->smem_bytes = kFixedSmem + (size_t)pl->q_per_block * qb;
    pl->packed_bytes = align_up((size_t)B * pl->n_pad * 16, 256);
    pl->part_bytes = 0;
    if (pl->n_split > 1) {
        const size_t rows = (size_t)B * S * pl->n_split;
        pl->part_bytes = align_up(rows * k * 4, 256) * (mode == MODE_TOPK ? 2 : 1) + align_up(rows * 4, 256);
    }
    // grid path of a top-k search (section 1b): counters, cell-sorted copies of refs and queries, one starting threshold per query
    pl->grid_bytes = 0;
    pl->grid_sorted = 0;
    if (mode == MODE_TOPK && grid_mode(B, N, S, k)) {
        pl->grid_bytes = grid_layout(B, N, S, pl->n_pad, nullptr, nullptr);
        pl->grid_sorted = grid_mode(B, N, S, k) == 2;
    }
    pl->total_bytes = pl->packed_bytes + pl->part_bytes + pl->grid_bytes;
    return true;
}

template <int FORM, int MODE, int Q>
static int launch_one(const SearchArgs &a, const SearchPlan &pl, int B, cudaStream_t st) {
    auto kern = search_kernel<FORM, MODE, Q>;
    B200PC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem_bytes));
    dim3 grid((a.S + pl.q_per_block - 1) / pl.q_per_block, B, pl.n_split);
    kern<<<grid, pl.consumer_warps * 32, pl.smem_bytes, st>>>(a);
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}

template <int FORM, int MODE>
static int launch_shape(const SearchArgs &a, const SearchPlan &pl, int B, cudaStream_t st) {
    if (pl.q_per_thread == 2) return launch_one<FORM, MODE, 2>(a, pl, B, st);
    return launch_one<FORM, MODE, 1>(a, pl, B, st);
}

// ref_len / qry_len: [B] device lengths of a ragged batch (top-k only), or null.  The plan and the workspace are those of
// the padded shape.
static int run_search(const float *ref, const float *qry, const int64_t *ref_len, const int64_t *qry_len, int B, int N, int S, int k,
                      int form, int mode, float r2, int64_t *idx, int32_t *idx32, float *dist, void *ws, size_t ws_bytes, cudaStream_t st) {
    B200PC_REQUIRE(B >= 0 && N >= 1 && S >= 0 && k >= 1, "search: bad sizes B=%d N=%d S=%d k=%d", B, N, S, k);
    if (B == 0 || S == 0) return B200PC_OK;             // empty work: nothing to validate, empty tensors have null pointers
    B200PC_REQUIRE(ref && qry, "search: null input pointer");
    B200PC_REQUIRE(idx || idx32 || dist, "search: no output requested");
    if (!idx32) {   // small reference sets: warp-per-query kernel, one launch, no workspace (small_search.cu)
        const int rc_small = run_small(ref, qry, ref_len, qry_len, B, N, S, k, form, mode, r2, idx, dist, st);
        if (rc_small != -100) return rc_small;
    }
    SearchPlan pl;
    if (!plan_search(B, N, S, k, mode, &pl)) {
        set_error("search: list length k=%d does not fit in shared memory%s", k,
                  tuning().force_q > 1 ? " at the forced queries per thread (B200PC_FORCE_Q)" : "");
        return B200PC_EINVAL;
    }
    if (!ws || ws_bytes < pl.total_bytes) {
        set_error("search: workspace too small (%zu < %zu bytes)", ws_bytes, pl.total_bytes);
        return B200PC_EWORKSPACE;
    }
    B200PC_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 15) == 0, "search: workspace must be 16-byte aligned");

    char *w = static_cast<char *>(ws);
    float4 *packed = reinterpret_cast<float4 *>(w);
    // top-k: refs dealt out to the tiles in a strided order (see slot_to_ref).  Not for form 1: its only caller is three-NN
    // feature propagation, whose reference points are FPS picks -- an order that is already ideal for a running k-best
    // (every prefix is a well-spread sample; measured 0.32 ms natural vs 0.36 ms strided on C3).
    const Tuning &tn = tuning();
    const int strided = mode == MODE_TOPK && (tn.natural_order >= 0 ? tn.natural_order == 0 : form != B200PC_FORM_QRY_NORM_FIRST);
    GridBufs gb{};
    int strided_eff = strided;
    if (pl.grid_bytes) {
        grid_layout(B, N, S, pl.n_pad, w + pl.packed_bytes + pl.part_bytes, &gb);
        const size_t zero_bytes = pl.grid_sorted ? reinterpret_cast<char *>(gb.cend) - reinterpret_cast<char *>(gb.counts)
                                                 : (size_t)B * GRID_STRIDE * sizeof(unsigned);
        B200PC_CUDA(cudaMemsetAsync(gb.counts, 0, zero_bytes, st));
        grid_bbox_kernel<<<B, 1024, 0, st>>>(ref, ref_len, N, gb.desc);
        B200PC_LAUNCH_CHECK();
    }
    if (pl.grid_bytes && pl.grid_sorted) {
        // count -> pyramid + segment sums -> scan -> scatter (sorted copies, packed tiles, slot table) -> starting thresholds
        grid_count_kernel<<<dim3((N + S + 255) / 256, B), 256, 0, st>>>(ref, ref_len, N, qry, qry_len, S, gb.desc, gb.counts, gb.qcend);
        B200PC_LAUNCH_CHECK();
        grid_pyramid_kernel<<<dim3(GRID_SEGS, B, 2), 256, 0, st>>>(gb.desc, gb.counts, gb.seg, gb.qcend, gb.qseg);
        B200PC_LAUNCH_CHECK();
        grid_scan_kernel<<<dim3(GRID_SEGS, B, 2), 256, 0, st>>>(gb.desc, gb.counts, gb.seg, gb.cend, gb.qcend, gb.qseg);
        B200PC_LAUNCH_CHECK();
        grid_scatter_kernel<<<dim3((pl.n_pad + S + 255) / 256, B), 256, 0, st>>>(ref, ref_len, N, pl.n_pad, pl.tiles_per_split, qry, qry_len, S,
                                                                                  gb.desc, gb, packed, tn.seed > 0 ? 0 : k);
        B200PC_LAUNCH_CHECK();
        if (tn.seed > 0) {                               // thresholds from the refs inside the boxes (A/B: B200PC_SEED=n); else the scatter wrote them
            grid_seed_kernel<<<dim3((S + SEED_THREADS - 1) / SEED_THREADS, B), SEED_THREADS, 0, st>>>(gb.qsorted, nullptr, qry_len, S, N, k, gb.desc, gb.counts,
                                                                                                gb.cend, gb.sorted, gb.seed, tn.seed);
            B200PC_LAUNCH_CHECK();
        }
        strided_eff = 0;                                  // the slot order is sorted_slot's
    } else {
        dim3 grid((pl.n_pad / 2 + 255) / 256, B);
        pack_refs_kernel<<<grid, 256, 0, st>>>(ref, ref_len, N, pl.n_pad, strided, packed, pl.grid_bytes ? gb.desc : nullptr, gb.counts);
        B200PC_LAUNCH_CHECK();
        if (pl.grid_bytes) {                              // thresholds only: the caller's order of refs and queries stays
            grid_pyramid_kernel<<<dim3(GRID_SEGS, B, 1), 256, 0, st>>>(gb.desc, gb.counts, gb.seg, gb.qcend, gb.qseg);
            B200PC_LAUNCH_CHECK();
            grid_seed_kernel<<<dim3((S + SEED_THREADS - 1) / SEED_THREADS, B), SEED_THREADS, 0, st>>>(nullptr, qry, qry_len, S, N, k, gb.desc, gb.counts, gb.cend,
                                                                                                gb.sorted, gb.seed, 0);
            B200PC_LAUNCH_CHECK();
            gb.qsorted = nullptr; gb.perm = nullptr;
        }
    }

    SearchArgs a;
    a.packed = packed; a.strided = strided_eff; a.qry = qry; a.ref_len = ref_len; a.qry_len = qry_len; a.N = N; a.n_pad = pl.n_pad; a.S = S; a.k = k; a.r2 = r2;
    a.n_split = pl.n_split; a.tiles_per_split = pl.tiles_per_split;
    a.debug_nodrain = tn.nodrain;
    a.lane_filter = tn.filter >= 0 ? tn.filter != 0 : 1;                          // 0: A/B measurement only
    a.qsorted = gb.qsorted; a.seed = gb.seed; a.perm = gb.perm; a.interleave = tn.interleave == 1;
    a.idx_out = idx; a.idx32_out = idx32; a.dist_out = dist; a.part_d = nullptr; a.part_i = nullptr; a.part_cnt = nullptr;
    if (pl.n_split > 1) {
        const size_t rows = (size_t)B * S * pl.n_split;
        char *p = w + pl.packed_bytes;
        a.part_i = reinterpret_cast<int *>(p); p += align_up(rows * k * 4, 256);
        if (mode == MODE_TOPK) { a.part_d = reinterpret_cast<float *>(p); p += align_up(rows * k * 4, 256); }
        a.part_cnt = reinterpret_cast<int *>(p);
    }
    if (tn.debug_plan)   // order: the ref order inside the tiles (strided: slot_to_ref; cell: sorted_slot)
        fprintf(stderr, "b200pc plan: B=%d N=%d S=%d k=%d mode=%d -> %d warps/CTA, %d queries/CTA, ref split %d (%d tiles each), grid %s, "
                "filter %s, order %s, %zu B smem\n", B, N, S, k, mode, pl.consumer_warps, pl.q_per_block, pl.n_split, pl.tiles_per_split,
                pl.grid_bytes ? (pl.grid_sorted ? "sorted" : "thresholds") : "off", a.lane_filter ? "lane" : "broadcast",
                pl.grid_sorted ? "cell" : strided_eff ? "strided" : "natural", pl.smem_bytes);
    int rc;
    if (mode == MODE_BALL) rc = launch_shape<B200PC_FORM_QRY_NORM_FIRST, MODE_BALL>(a, pl, B, st);
    else if (form == B200PC_FORM_REF_NORM_FIRST) rc = launch_shape<B200PC_FORM_REF_NORM_FIRST, MODE_TOPK>(a, pl, B, st);
    else if (form == B200PC_FORM_QRY_NORM_FIRST) rc = launch_shape<B200PC_FORM_QRY_NORM_FIRST, MODE_TOPK>(a, pl, B, st);
    else rc = launch_shape<B200PC_FORM_DIRECT, MODE_TOPK>(a, pl, B, st);
    if (rc != B200PC_OK) return rc;

    if (pl.n_split > 1) {
        const int rows = B * S;
        if (mode == MODE_TOPK)
            merge_topk_kernel<<<(rows + 7) / 8, 256, 0, st>>>(a.part_d, a.part_i, rows, pl.n_split, k, idx, idx32, dist);
        else
            merge_ball_kernel<<<(rows + 7) / 8, 256, 0, st>>>(a.part_i, a.part_cnt, rows, pl.n_split, k, N, idx, idx32);
        B200PC_LAUNCH_CHECK();
    }
    return B200PC_OK;
}

int run_topk(const float *ref, const float *qry, int B, int N, int S, int k, int form, int64_t *idx, float *dist,
             void *ws, size_t ws_bytes, cudaStream_t st, const int64_t *ref_len, const int64_t *qry_len) {
    B200PC_REQUIRE(form >= 0 && form <= 2, "knn: unknown distance form %d", form);
    B200PC_REQUIRE(k <= N, "knn: k=%d exceeds the number of reference points N=%d", k, N);
    return run_search(ref, qry, ref_len, qry_len, B, N, S, k, form, MODE_TOPK, 0.f, idx, nullptr, dist, ws, ws_bytes, st);
}

int run_topk_i32(const float *ref, const float *qry, int B, int N, int S, int k, int form, int32_t *idx32, float *dist,
                 void *ws, size_t ws_bytes, cudaStream_t st) {
    B200PC_REQUIRE(form >= 0 && form <= 2, "knn: unknown distance form %d", form);
    B200PC_REQUIRE(k <= N, "knn: k=%d exceeds the number of reference points N=%d", k, N);
    return run_search(ref, qry, nullptr, nullptr, B, N, S, k, form, MODE_TOPK, 0.f, nullptr, idx32, dist, ws, ws_bytes, st);
}

int run_ball(const float *ref, const float *qry, int B, int N, int S, float r2, int nsample, int64_t *idx,
             void *ws, size_t ws_bytes, cudaStream_t st) {
    B200PC_REQUIRE(idx || B == 0 || S == 0, "ball_query: null output pointer");
    return run_search(ref, qry, nullptr, nullptr, B, N, S, nsample, B200PC_FORM_QRY_NORM_FIRST, MODE_BALL, r2, idx, nullptr, nullptr, ws,
                      ws_bytes, st);
}

}  // namespace b200pc

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
using namespace b200pc;

extern "C" size_t b200pc_search_workspace_bytes(int B, int N, int S, int k) {
    if (B <= 0 || N <= 0 || S <= 0 || k <= 0) return 256;
    SearchPlan a, c;
    size_t need = 256;
    if (plan_search(B, N, S, k, MODE_TOPK, &a)) need = a.total_bytes > need ? a.total_bytes : need;
    if (plan_search(B, N, S, k, MODE_BALL, &c)) need = c.total_bytes > need ? c.total_bytes : need;
    return need;
}

extern "C" int b200pc_knn(const float *ref, const float *qry, int B, int N, int S, int k, int form, int64_t *idx,
                          float *dist, void *workspace, size_t workspace_bytes, b200pc_stream_t stream) {
    return run_topk(ref, qry, B, N, S, k, form, idx, dist, workspace, workspace_bytes, as_stream(stream));
}

extern "C" int b200pc_knn_ragged(const float *ref, const float *qry, const int64_t *ref_len, const int64_t *qry_len, int B, int N,
                                 int S, int k, int form, int64_t *idx, float *dist, void *workspace, size_t workspace_bytes,
                                 b200pc_stream_t stream) {
    return run_topk(ref, qry, B, N, S, k, form, idx, dist, workspace, workspace_bytes, as_stream(stream), ref_len, qry_len);
}

extern "C" int b200pc_knn_i32(const float *ref, const float *qry, int B, int N, int S, int k, int form, int32_t *idx,
                              float *dist, void *workspace, size_t workspace_bytes, b200pc_stream_t stream) {
    return run_topk_i32(ref, qry, B, N, S, k, form, idx, dist, workspace, workspace_bytes, as_stream(stream));
}

extern "C" int b200pc_ball_query(const float *xyz, const float *new_xyz, int B, int N, int S, float r2, int nsample,
                                 int64_t *idx, void *workspace, size_t workspace_bytes, b200pc_stream_t stream) {
    B200PC_REQUIRE(nsample >= 1, "ball_query: nsample must be >= 1");
    return run_ball(xyz, new_xyz, B, N, S, r2, nsample, idx, workspace, workspace_bytes, as_stream(stream));
}
