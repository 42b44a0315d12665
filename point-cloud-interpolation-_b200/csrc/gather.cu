// gather.cu -- HBM-bound row movers (sm_100a):
//   index_points        Utils/Pointnet2Utils.py:44-61      (also pytorch3d knn_gather, Utils/Layers.py:396,434)
//   three_nn weights    Utils/Layers.py:183-186 (variant 0), Utils/Pointnet2Utils.py:301-303 (variant 1)
//   three_interpolate   Utils/Layers.py:187-188, Utils/Pointnet2Utils.py:304
// and their gradients.  Rows are moved as 16-byte vectors whenever the channel count and the base
// addresses allow it, one warp per row with several rows in flight; streamed data bypasses L1
// allocation.  Grids are capped at 16 CTAs per SM and grid-stride over the rows.
#include <stdlib.h>

#include "common.cuh"
#include "search.cuh"

namespace b200pc {

static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int wave_grid(long work_items, int threads, int per_thread) {
    const int sms = sm_count();
    long blocks = (work_items + (long)threads * per_thread - 1) / ((long)threads * per_thread);
    const long cap = (long)sms * 16;  // enough CTAs in flight to saturate HBM, then grid-stride
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

// ------------------------------------------------------------------------------------------
// index_points
// ------------------------------------------------------------------------------------------
// One WARP per output row, ROWS rows in flight per warp: the index of a row is read once (lanes < ROWS,
// then shuffled), so there is no per-vector division and no redundant index traffic, and every lane has
// ROWS independent 16-byte loads outstanding before the first store (memory-level parallelism is what
// bounds a 20-70 us gather).  Lanes stride over the row when C4 > 32.
template <int ROWS>
__global__ void __launch_bounds__(256) gather_rows_kernel(const float4 *__restrict__ points, const int64_t *__restrict__ idx,
                                                          int N, int C4, long R, long rows_total, float4 *__restrict__ out,
                                                          int *__restrict__ oob) {
    const int lane = threadIdx.x & 31;
    const long warp = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long nwarps = ((long)gridDim.x * blockDim.x) >> 5;
    for (long r0 = warp * ROWS; r0 < rows_total; r0 += nwarps * ROWS) {
        long src = -1;                                   // lane l < ROWS owns row r0 + l
        if (lane < ROWS && r0 + lane < rows_total) {
            const long row = r0 + lane;
            long i = idx[row];
            if (i < 0) i += N;
            if (i < 0 || i >= N) { if (oob) *oob = 1; }
            else src = ((row / R) * N + i) * C4;
            B200PC_DEV_ASSERT(src < 0 || (src >= 0 && i >= 0 && i < N));
        }
        long so[ROWS];                                   // every lane takes part in the shuffles
#pragma unroll
        for (int u = 0; u < ROWS; ++u) so[u] = __shfl_sync(0xffffffffu, src, u);
        for (int col = lane; col < C4; col += 32) {
            float4 v[ROWS];
#pragma unroll
            for (int u = 0; u < ROWS; ++u)
                v[u] = so[u] >= 0 ? ldg_stream(points + so[u] + col) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < ROWS; ++u)
                if (r0 + u < rows_total) stg_stream(out + (r0 + u) * C4 + col, v[u]);
        }
    }
}

// Flat variant: one thread per 16-byte output vector, no loop and no shuffles -- the C4 threads of a row read the same
// index (one broadcast transaction) and the whole grid's loads are in flight at once.  Used for rows narrower than a
// warp (C < 128: 0.015 vs 0.025 ms at C=64, C3 size); wider rows keep the warp-per-row kernel (B200PC_GATHER_FLAT=0|1 forces).
__global__ void __launch_bounds__(256) gather_flat_kernel(const float4 *__restrict__ points, const int64_t *__restrict__ idx,
                                                          int N, int C4, long R, long total, float4 *__restrict__ out,
                                                          int *__restrict__ oob) {
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const long row = t / C4;
    const int col = (int)(t - row * C4);
    long i = __ldg(idx + row);
    if (i < 0) i += N;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < 0 || i >= N) { if (oob) *oob = 1; }
    else v = ldg_stream(points + ((row / R) * N + i) * C4 + col);
    stg_stream(out + t, v);
}

__global__ void __launch_bounds__(256) gather_scalar_kernel(const float *__restrict__ points, const int64_t *__restrict__ idx,
                                                            int N, int C, long R, long total, float *__restrict__ out,
                                                            int *__restrict__ oob) {
    const long stride = (long)gridDim.x * blockDim.x;
    for (long v = (long)blockIdx.x * blockDim.x + threadIdx.x; v < total; v += stride) {
        const long row = v / C;
        const int col = (int)(v - row * C);
        const long b = row / R;
        long i = idx[row];
        if (i < 0) i += N;
        float r = 0.f;
        if (i < 0 || i >= N) { if (oob) *oob = 1; }
        else r = __ldg(points + ((b * N + i) * C + col));
        out[v] = r;
    }
}

// gradient: gpoints[b, idx[b,r], :] += gout[b,r,:]
__global__ void __launch_bounds__(256) scatter_add_vec4_kernel(const float4 *__restrict__ gout, const int64_t *__restrict__ idx,
                                                               int N, int C4, long R, long total, float *__restrict__ gpoints) {
    const long stride = (long)gridDim.x * blockDim.x;
    for (long v = (long)blockIdx.x * blockDim.x + threadIdx.x; v < total; v += stride) {
        const long row = v / C4;
        const int col = (int)(v - row * C4);
        const long b = row / R;
        long i = idx[row];
        if (i < 0) i += N;
        if (i < 0 || i >= N) continue;
        red_add_v4(gpoints + ((b * N + i) * C4 + col) * 4, ldg_stream(gout + v));
    }
}

__global__ void __launch_bounds__(256) scatter_add_scalar_kernel(const float *__restrict__ gout, const int64_t *__restrict__ idx,
                                                                 int N, int C, long R, long total, float *__restrict__ gpoints) {
    const long stride = (long)gridDim.x * blockDim.x;
    for (long v = (long)blockIdx.x * blockDim.x + threadIdx.x; v < total; v += stride) {
        const long row = v / C;
        const int col = (int)(v - row * C);
        const long b = row / R;
        long i = idx[row];
        if (i < 0) i += N;
        if (i < 0 || i >= N) continue;
        atomicAdd(gpoints + ((b * N + i) * C + col), gout[v]);
    }
}

// ------------------------------------------------------------------------------------------
// three-NN weights
// ------------------------------------------------------------------------------------------
__global__ void three_weights_kernel(const float *__restrict__ dist, long rows, int variant, float *__restrict__ w) {
    const long r = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    float inv[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        float d = dist[r * 3 + j];
        if (variant == 0) {
            if (d < 1e-10f) d = 1e-10f;        // dists[dists < 1e-10] = 1e-10
            inv[j] = __fdiv_rn(1.0f, d);
        } else {
            inv[j] = __fdiv_rn(1.0f, __fadd_rn(d, 1e-8f));
        }
    }
    const float norm = __fadd_rn(__fadd_rn(inv[0], inv[1]), inv[2]);
#pragma unroll
    for (int j = 0; j < 3; ++j) w[r * 3 + j] = __fdiv_rn(inv[j], norm);
}

// ------------------------------------------------------------------------------------------
// three_interpolate: out[b,n,:] = (f[i0]*w0 + f[i1]*w1) + f[i2]*w2   (separate mul / add)
// ------------------------------------------------------------------------------------------
// index hygiene of the interpolation kernels: negative indices wrap once (torch indexing); an index that is still out
// of range contributes nothing (row 0 with weight 0) instead of reading outside the table -- the reference raises there.
__device__ __forceinline__ void clean_neighbour(long &i, float &w, int S) {
    if ((unsigned long long)i >= (unsigned long long)S) {      // one compare on the common path
        if (i < 0) i += S;
        if (i < 0 || i >= S) { i = 0; w = 0.0f; }
    }
}

__device__ __forceinline__ float mix3(float a, float wa, float b, float wb, float c, float wc) {
    return __fadd_rn(__fadd_rn(__fmul_rn(a, wa), __fmul_rn(b, wb)), __fmul_rn(c, wc));
}

// warp per dense row, ROWS rows in flight: lanes < 3*ROWS read the row's three (index, weight) pairs once
// and shuffle them; every lane then has 3*ROWS independent 16-byte gathers outstanding.  Row offsets are kept
// as 32-bit vector indices (the launcher checks B*S*C4 < 2^31) and the register budget is capped so that at
// least 3 CTAs stay resident: the kernel is a latency chain (idx -> gather -> store), occupancy is what feeds it.
// resident CTAs asked of ptxas: 2 rows in flight fit 62 registers without spills = 4 CTAs = 32 warps instead of 24 (the
// kernel is a latency chain: 59.7 -> 51.3 us at C3); 1 row fits 6 CTAs
constexpr int interp_min_blocks(int rows) { return rows == 1 ? 6 : rows == 2 ? 4 : 2; }
template <int ROWS>
__global__ void __launch_bounds__(256, interp_min_blocks(ROWS)) interp_rows_kernel(const float4 *__restrict__ feat, const int64_t *__restrict__ idx,
                                                             const float *__restrict__ w, int S, int C4, long N, long rows_total,
                                                             float4 *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long warp = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long nwarps = ((long)gridDim.x * blockDim.x) >> 5;
    // (index, weight) of the NEXT group of rows are requested before the current group is gathered
    long i_next = 0;
    float w_next = 0.f;
    {
        const long row = warp * ROWS + lane / 3;
        if (lane < 3 * ROWS && row < rows_total) { i_next = idx[row * 3 + lane % 3]; w_next = w[row * 3 + lane % 3]; }
    }
    for (long r0 = warp * ROWS; r0 < rows_total; r0 += nwarps * ROWS) {
        int src = 0;
        float wt = w_next;
        long i_cur = i_next;
        clean_neighbour(i_cur, wt, S);                   // at the point of use: the prefetch below stays in flight
        {
            const long rn = r0 + nwarps * ROWS + lane / 3;
            if (lane < 3 * ROWS && rn < rows_total) { i_next = idx[rn * 3 + lane % 3]; w_next = w[rn * 3 + lane % 3]; }
        }
        if (lane < 3 * ROWS) {                          // lane = 3*u + j  ->  neighbour j of row r0+u
            const long row = r0 + lane / 3;
            B200PC_DEV_ASSERT(i_cur >= 0 && i_cur < S);
            if (row < rows_total) src = (int)(((row / N) * S + i_cur) * C4);
        }
        int so[ROWS][3];                                 // every lane takes part in the shuffles
        float ww[ROWS][3];
#pragma unroll
        for (int u = 0; u < ROWS; ++u)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                so[u][j] = __shfl_sync(0xffffffffu, src, 3 * u + j);
                ww[u][j] = __shfl_sync(0xffffffffu, wt, 3 * u + j);
            }
        for (int col = lane; col < C4; col += 32) {
            float4 f[ROWS][3];
#pragma unroll
            for (int u = 0; u < ROWS; ++u)
#pragma unroll
                for (int j = 0; j < 3; ++j) f[u][j] = __ldg(feat + so[u][j] + col);   // sparse rows are re-read ~3N/S times: keep them cached
#pragma unroll
            for (int u = 0; u < ROWS; ++u) {
                if (r0 + u >= rows_total) continue;
                float4 o;
                o.x = mix3(f[u][0].x, ww[u][0], f[u][1].x, ww[u][1], f[u][2].x, ww[u][2]);
                o.y = mix3(f[u][0].y, ww[u][0], f[u][1].y, ww[u][1], f[u][2].y, ww[u][2]);
                o.z = mix3(f[u][0].z, ww[u][0], f[u][1].z, ww[u][1], f[u][2].z, ww[u][2]);
                o.w = mix3(f[u][0].w, ww[u][0], f[u][1].w, ww[u][1], f[u][2].w, ww[u][2]);
                stg_stream(out + (r0 + u) * C4 + col, o);
            }
        }
    }
}

// Flat variant: one thread per 16-byte output vector; default for C < 128 (0.035 vs 0.053 ms at C=64), B200PC_INTERP_FLAT=0|1 forces.
__global__ void __launch_bounds__(256) interp_flat_kernel(const float4 *__restrict__ feat, const int64_t *__restrict__ idx,
                                                          const float *__restrict__ w, int S, int C4, long N, long total,
                                                          float4 *__restrict__ out) {
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const long row = t / C4;
    const int col = (int)(t - row * C4);
    const long base = (row / N) * S;
    long i0 = __ldg(idx + row * 3), i1 = __ldg(idx + row * 3 + 1), i2 = __ldg(idx + row * 3 + 2);
    float w0 = __ldg(w + row * 3), w1 = __ldg(w + row * 3 + 1), w2 = __ldg(w + row * 3 + 2);
    clean_neighbour(i0, w0, S); clean_neighbour(i1, w1, S); clean_neighbour(i2, w2, S);
    const float4 a = __ldg(feat + (base + i0) * C4 + col), b = __ldg(feat + (base + i1) * C4 + col), c = __ldg(feat + (base + i2) * C4 + col);
    float4 o;
    o.x = mix3(a.x, w0, b.x, w1, c.x, w2); o.y = mix3(a.y, w0, b.y, w1, c.y, w2);
    o.z = mix3(a.z, w0, b.z, w1, c.z, w2); o.w = mix3(a.w, w0, b.w, w1, c.w, w2);
    stg_stream(out + t, o);
}

__global__ void __launch_bounds__(256) interp_scalar_kernel(const float *__restrict__ feat, const int64_t *__restrict__ idx,
                                                            const float *__restrict__ w, int S, int C, long N, long total,
                                                            float *__restrict__ out) {
    const long stride = (long)gridDim.x * blockDim.x;
    for (long v = (long)blockIdx.x * blockDim.x + threadIdx.x; v < total; v += stride) {
        const long row = v / C;
        const int col = (int)(v - row * C);
        const long b = row / N;
        long i0 = idx[row * 3], i1 = idx[row * 3 + 1], i2 = idx[row * 3 + 2];
        float w0 = w[row * 3], w1 = w[row * 3 + 1], w2 = w[row * 3 + 2];
        clean_neighbour(i0, w0, S); clean_neighbour(i1, w1, S); clean_neighbour(i2, w2, S);
        out[v] = mix3(__ldg(feat + (b * S + i0) * C + col), w0, __ldg(feat + (b * S + i1) * C + col), w1,
                      __ldg(feat + (b * S + i2) * C + col), w2);
    }
}

// gradient: one warp per dense row.  gfeat[b,i_j,:] += gout*w_j ; gweight[b,n,j] = <gout, feat[i_j]>
// A neighbour the forward pass dropped (index out of range after one wrap) contributed nothing: it gets no gfeat add and
// gweight 0.
__global__ void __launch_bounds__(256) interp_bwd_kernel(const float *__restrict__ gout, const float *__restrict__ feat,
                                                         const int64_t *__restrict__ idx, const float *__restrict__ w, int S,
                                                         int C, long N, long rows, float *__restrict__ gfeat,
                                                         float *__restrict__ gweight) {
    const int lane = threadIdx.x & 31;
    const long warp_global = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long nwarps = ((long)gridDim.x * blockDim.x) >> 5;
    for (long row = warp_global; row < rows; row += nwarps) {
        const long b = row / N;
        long id[3];
        float ww[3], acc[3] = {0.f, 0.f, 0.f};
        bool ok[3];                                      // warp-uniform: the whole warp works on one row
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            long i = idx[row * 3 + j];
            if (i < 0) i += S;
            ok[j] = i >= 0 && i < S;
            id[j] = ok[j] ? i : 0;
            ww[j] = w[row * 3 + j];
        }
        for (int c = lane; c < C; c += 32) {
            const float g = gout[row * C + c];
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                if (!ok[j]) continue;
                const long o = (b * S + id[j]) * C + c;
                B200PC_DEV_ASSERT(id[j] >= 0 && id[j] < S);
                atomicAdd(gfeat + o, g * ww[j]);
                if (gweight) acc[j] += g * feat[o];
            }
        }
        if (gweight) {
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                float a = acc[j];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
                if (lane == 0) gweight[row * 3 + j] = ok[j] ? a : 0.0f;
            }
        }
    }
}

}  // namespace b200pc

using namespace b200pc;

extern "C" int b200pc_gather(const float *points, const int64_t *idx, int B, int N, int C, int64_t R, float *out,
                             int *oob_flag, b200pc_stream_t stream) {
    B200PC_REQUIRE(B >= 0 && N >= 1 && C >= 1 && R >= 0, "gather: bad sizes");
    if (B == 0 || R == 0) return B200PC_OK;
    B200PC_REQUIRE(points && idx && out, "gather: null pointer");
    cudaStream_t st = as_stream(stream);
    if (C % 4 == 0 && aligned16(points) && aligned16(out)) {
        const long rows = (long)B * R;
        const Tuning &tn = tuning();                        // cached knobs (not part of the ABI)
        const int rw = tn.gather_rows > 0 ? tn.gather_rows : 8;
        if (tn.gather_flat >= 0 ? tn.gather_flat != 0 : C / 4 < 32) {   // default: flat for narrow rows (a warp per row idles lanes when C < 128)
            const long total = rows * (C / 4);
            gather_flat_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(reinterpret_cast<const float4 *>(points), idx, N, C / 4,
                                                                               (long)R, total, reinterpret_cast<float4 *>(out), oob_flag);
        } else if (rw == 8)
            gather_rows_kernel<8><<<wave_grid(rows * 32 / 8, 256, 1), 256, 0, st>>>(
                reinterpret_cast<const float4 *>(points), idx, N, C / 4, (long)R, rows, reinterpret_cast<float4 *>(out), oob_flag);
        else if (rw == 2)
            gather_rows_kernel<2><<<wave_grid(rows * 32 / 2, 256, 1), 256, 0, st>>>(
                reinterpret_cast<const float4 *>(points), idx, N, C / 4, (long)R, rows, reinterpret_cast<float4 *>(out), oob_flag);
        else
            gather_rows_kernel<4><<<wave_grid(rows * 32 / 4, 256, 1), 256, 0, st>>>(
                reinterpret_cast<const float4 *>(points), idx, N, C / 4, (long)R, rows, reinterpret_cast<float4 *>(out), oob_flag);
    } else {
        const long total = (long)B * R * C;
        gather_scalar_kernel<<<wave_grid(total, 256, 1), 256, 0, st>>>(points, idx, N, C, (long)R, total, out, oob_flag);
    }
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}

extern "C" int b200pc_gather_bwd(const float *gout, const int64_t *idx, int B, int N, int C, int64_t R, float *gpoints,
                                 b200pc_stream_t stream) {
    if (B == 0 || R == 0) return B200PC_OK;
    B200PC_REQUIRE(gout && idx && gpoints, "gather_bwd: null pointer");
    cudaStream_t st = as_stream(stream);
    if (C % 4 == 0 && aligned16(gout) && aligned16(gpoints)) {
        const long total = (long)B * R * (C / 4);
        scatter_add_vec4_kernel<<<wave_grid(total, 256, 1), 256, 0, st>>>(reinterpret_cast<const float4 *>(gout), idx, N,
                                                                          C / 4, (long)R, total, gpoints);
    } else {
        const long total = (long)B * R * C;
        scatter_add_scalar_kernel<<<wave_grid(total, 256, 1), 256, 0, st>>>(gout, idx, N, C, (long)R, total, gpoints);
    }
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}

extern "C" int b200pc_three_nn(const float *unknown, const float *known, int B, int N, int S, int variant, float *dist,
                               int64_t *idx, float *weight, void *workspace, size_t workspace_bytes,
                               b200pc_stream_t stream) {
    B200PC_REQUIRE(dist && idx, "three_nn: dist and idx outputs are required");
    B200PC_REQUIRE(S >= 3, "three_nn: needs at least 3 known points, got S=%d", S);
    B200PC_REQUIRE(variant == 0 || variant == 1, "three_nn: unknown weight variant %d", variant);
    cudaStream_t st = as_stream(stream);
    // refs = known (sparse), queries = unknown (dense); the dense cloud is `src` of square_distance
    int rc = run_topk(known, unknown, B, S, N, 3, B200PC_FORM_QRY_NORM_FIRST, idx, dist, workspace, workspace_bytes, st);
    if (rc != B200PC_OK) return rc;
    if (weight && B > 0 && N > 0) {
        const long rows = (long)B * N;
        three_weights_kernel<<<(int)((rows + 255) / 256), 256, 0, st>>>(dist, rows, variant, weight);
        B200PC_LAUNCH_CHECK();
    }
    return B200PC_OK;
}

extern "C" int b200pc_three_interpolate(const float *feat, const int64_t *idx, const float *weight, int B, int S, int N,
                                        int C, float *out, b200pc_stream_t stream) {
    if (B == 0 || N == 0) return B200PC_OK;
    B200PC_REQUIRE(feat && idx && weight && out, "three_interpolate: null pointer");
    cudaStream_t st = as_stream(stream);
    if (C % 4 == 0 && aligned16(feat) && aligned16(out) && (long)B * S * (C / 4) < (1L << 31)) {
        const long rows = (long)B * N;
        const Tuning &tn = tuning();                        // cached knobs (not part of the ABI)
        const int rw = tn.interp_rows > 0 ? tn.interp_rows : 2;
        const float4 *f4 = reinterpret_cast<const float4 *>(feat);
        float4 *o4 = reinterpret_cast<float4 *>(out);
        if (tn.interp_flat >= 0 ? tn.interp_flat != 0 : C / 4 < 32) {   // default: flat for narrow rows (C < 128)
            const long total = rows * (C / 4);
            interp_flat_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(f4, idx, weight, S, C / 4, (long)N, total, o4);
        } else if (rw == 1) interp_rows_kernel<1><<<wave_grid(rows * 32, 256, 1), 256, 0, st>>>(f4, idx, weight, S, C / 4, (long)N, rows, o4);
        else if (rw == 8) interp_rows_kernel<8><<<wave_grid(rows * 32 / 8, 256, 1), 256, 0, st>>>(f4, idx, weight, S, C / 4, (long)N, rows, o4);
        else if (rw == 2) interp_rows_kernel<2><<<wave_grid(rows * 32 / 2, 256, 1), 256, 0, st>>>(f4, idx, weight, S, C / 4, (long)N, rows, o4);
        else interp_rows_kernel<4><<<wave_grid(rows * 32 / 4, 256, 1), 256, 0, st>>>(f4, idx, weight, S, C / 4, (long)N, rows, o4);
    } else {
        const long total = (long)B * N * C;
        interp_scalar_kernel<<<wave_grid(total, 256, 1), 256, 0, st>>>(feat, idx, weight, S, C, (long)N, total, out);
    }
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}

extern "C" int b200pc_three_interpolate_bwd(const float *gout, const float *feat, const int64_t *idx, const float *weight,
                                            int B, int S, int N, int C, float *gfeat, float *gweight,
                                            b200pc_stream_t stream) {
    if (B == 0 || N == 0) return B200PC_OK;
    B200PC_REQUIRE(gout && feat && idx && weight && gfeat, "three_interpolate_bwd: null pointer");
    const long rows = (long)B * N;
    interp_bwd_kernel<<<wave_grid(rows * 32, 256, 1), 256, 0, as_stream(stream)>>>(gout, feat, idx, weight, S, C, (long)N,
                                                                                  rows, gfeat, gweight);
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}


// a5 in one call: FeaturePropagation.forward's interpolation (Utils/Layers.py:180-188) / PointNetFeaturePropagation's
// (Utils/Pointnet2Utils.py:297-304): three-NN search -> inverse-distance weights -> weighted mix of the three rows.
// The distances never leave the workspace; idx and weight are returned because the backward pass needs them.
extern "C" size_t b200pc_feature_propagation_workspace_bytes(int B, int N, int S) {
    if (B <= 0 || N <= 0 || S <= 0) return 256;
    return align_up(b200pc_search_workspace_bytes(B, S, N, 3), 256) + align_up((size_t)B * N * 3 * sizeof(float), 256);
}

extern "C" int b200pc_feature_propagation(const float *unknown, const float *known, const float *feat, int B, int N, int S,
                                          int C, int variant, float *out, int64_t *idx, float *weight, void *workspace,
                                          size_t workspace_bytes, b200pc_stream_t stream) {
    B200PC_REQUIRE(B >= 0 && N >= 0 && S >= 3 && C >= 1, "feature_propagation: bad sizes B=%d N=%d S=%d C=%d (needs S >= 3)", B, N, S, C);
    if (B == 0 || N == 0) return B200PC_OK;
    B200PC_REQUIRE(unknown && known && feat && out && idx && weight, "feature_propagation: null pointer");
    const size_t search_bytes = align_up(b200pc_search_workspace_bytes(B, S, N, 3), 256);
    if (!workspace || workspace_bytes < b200pc_feature_propagation_workspace_bytes(B, N, S)) {
        set_error("feature_propagation: workspace too small (%zu < %zu bytes)", workspace_bytes,
                  b200pc_feature_propagation_workspace_bytes(B, N, S));
        return B200PC_EWORKSPACE;
    }
    float *dist = reinterpret_cast<float *>(static_cast<char *>(workspace) + search_bytes);
    int rc = b200pc_three_nn(unknown, known, B, N, S, variant, dist, idx, weight, workspace, search_bytes, stream);
    if (rc != B200PC_OK) return rc;
    return b200pc_three_interpolate(feat, idx, weight, B, S, N, C, out, stream);
}
