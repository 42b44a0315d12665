// small_search.cu -- warp-per-query search for SMALL reference sets (N <= 1024), one launch, raw xyz.
//
// The streaming kernel (search.cu) gives one thread per query; with a few hundred queries against a few
// hundred refs (FlowNet3D's inner layers: kNN k=64 on 256x256, k=8 on 64x16 / 256x64 / 1024x256, ball
// queries 256x1024 / 64x256 / 16x64 -- Models.py:31-38 in the reference) that is a handful of warps whose
// serial list maintenance is pure latency (0.31 ms for 256x256, k=64).  Here a WARP owns a query: each
// lane evaluates N/32 refs (same fp32 rounding sequences as search.cu, scalar instead of packed), then
//   * top-k: k rounds of warp arg-min over 64-bit keys (order(d) << 32 | index) -- two REDUX per round,
//     only the winning lane rescans its N/32 values;  ties go to the lower index by construction;
//   * ball : refs are visited 32 at a time in index order, a ballot + popc prefix appends the hits, and the
//     warp stops as soon as nsample are found.
// Results are bit-identical to the streaming kernel (tests/test_gpu_search.py runs both).
#include <math_constants.h>
#include <stdlib.h>

#include "search.cuh"

namespace b200pc {

constexpr int SMALL_MAX_N = 1024;
constexpr int SMALL_WARPS = 4;

__device__ __forceinline__ float sq_norm_torch(float x, float y, float z) {
    return __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
}
__device__ __forceinline__ uint32_t okey(float d) {
    const uint32_t b = __float_as_uint(d);
    return b ^ (static_cast<uint32_t>(static_cast<int32_t>(b) >> 31) | 0x80000000u);
}
__device__ __forceinline__ float okey_inv(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k); }

template <int FORM>
__device__ __forceinline__ float dist_scalar(float rx, float ry, float rz, float rn, float qx, float qy, float qz, float qn) {
    if (FORM == B200PC_FORM_DIRECT) {
        const float dx = __fadd_rn(rx, -qx), dy = __fadd_rn(ry, -qy), dz = __fadd_rn(rz, -qz);
        return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
    }
    float t = __fmul_rn(rx, -2.0f * qx);
    t = __fmaf_rn(ry, -2.0f * qy, t);
    t = __fmaf_rn(rz, -2.0f * qz, t);
    if (FORM == B200PC_FORM_REF_NORM_FIRST) return __fadd_rn(__fadd_rn(t, rn), qn);
    return __fadd_rn(__fadd_rn(t, qn), rn);
}

// NI = refs per lane (N <= 32*NI)
template <int FORM, int MODE, int NI>
__global__ void __launch_bounds__(SMALL_WARPS * 32) small_search_kernel(const float *__restrict__ ref, const float *__restrict__ qry,
                                                                        int N, int S, int k, float r2, int64_t *__restrict__ idx_out,
                                                                        float *__restrict__ dist_out) {
    __shared__ float sx[SMALL_MAX_N], sy[SMALL_MAX_N], sz[SMALL_MAX_N], sn[SMALL_MAX_N];
    const int b = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float *rb = ref + (size_t)b * N * 3;
    for (int i = threadIdx.x; i < 32 * NI; i += blockDim.x) {
        float x = 0.f, y = 0.f, z = 0.f;
        if (i < N) { x = rb[i * 3]; y = rb[i * 3 + 1]; z = rb[i * 3 + 2]; }
        sx[i] = x; sy[i] = y; sz[i] = z;
        sn[i] = FORM == B200PC_FORM_DIRECT ? 0.f : sq_norm_torch(x, y, z);
    }
    __syncthreads();
    for (int q = blockIdx.x * SMALL_WARPS + warp; q < S; q += gridDim.x * SMALL_WARPS) {
        const float *qp = qry + ((size_t)b * S + q) * 3;
        const float qx = qp[0], qy = qp[1], qz = qp[2];
        const float qn = FORM == B200PC_FORM_DIRECT ? 0.f : sq_norm_torch(qx, qy, qz);
        const size_t row = (size_t)b * S + q;
        if (MODE == MODE_BALL) {
            int cnt = 0;
            int64_t first = N;
            int64_t *o = idx_out + row * k;
#pragma unroll 1
            for (int i = 0; i < NI && cnt < k; ++i) {
                const int r = i * 32 + lane;
                const float d = dist_scalar<FORM>(sx[r], sy[r], sz[r], sn[r], qx, qy, qz, qn);
                const bool hit = r < N && d <= r2;        // same predicate as the streaming kernel: a NaN distance is never a hit
                const unsigned m = __ballot_sync(0xffffffffu, hit);
                if (m) {
                    if (cnt == 0) first = i * 32 + (__ffs(m) - 1);
                    const int pos = cnt + __popc(m & ((1u << lane) - 1u));
                    if (hit && pos < k) o[pos] = r;
                    cnt += __popc(m);
                }
            }
            for (int e = (cnt < k ? cnt : k) + lane; e < k; e += 32) o[e] = first;
        } else {
            unsigned long long key[NI];
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int r = i * 32 + lane;
                const float d = dist_scalar<FORM>(sx[r], sy[r], sz[r], sn[r], qx, qy, qz, qn);
                // only a finite distance is a candidate (NaN and +inf get the empty key; no form yields -inf)
                key[i] = r < N && d < CUDART_INF_F ? (((unsigned long long)okey(d) << 32) | (unsigned)r) : ~0ull;
            }
            unsigned long long best = ~0ull;
#pragma unroll
            for (int i = 0; i < NI; ++i) best = key[i] < best ? key[i] : best;
            for (int e = 0; e < k; ++e) {
                const unsigned hi = (unsigned)(best >> 32);
                const unsigned whi = __reduce_min_sync(0xffffffffu, hi);
                const unsigned wlo = __reduce_min_sync(0xffffffffu, hi == whi ? (unsigned)best : 0xffffffffu);
                if (lane == 0) {      // the empty key: fewer than k candidates, -1 with distance +inf
                    const bool empty = whi == 0xffffffffu;
                    if (idx_out) idx_out[row * k + e] = empty ? -1 : (int64_t)wlo;
                    if (dist_out) dist_out[row * k + e] = empty ? CUDART_INF_F : okey_inv(whi);
                }
                if (hi == whi && (unsigned)best == wlo) {     // the winning lane retires that ref and rescans
                    unsigned long long nb = ~0ull;
#pragma unroll
                    for (int i = 0; i < NI; ++i) {
                        if (key[i] == best) key[i] = ~0ull;
                        nb = key[i] < nb ? key[i] : nb;
                    }
                    best = nb;
                }
            }
        }
    }
}

template <int FORM, int MODE>
static int launch_small(const float *ref, const float *qry, int B, int N, int S, int k, float r2, int64_t *idx, float *dist,
                        cudaStream_t st) {
    const int ni = (N + 31) / 32;
    int blocks = (S + SMALL_WARPS - 1) / SMALL_WARPS;
    const int cap = sm_count() * 8;
    if (blocks > cap) blocks = cap;
    dim3 grid(blocks, B);
#define B200PC_SMALL(NI_) small_search_kernel<FORM, MODE, NI_><<<grid, SMALL_WARPS * 32, 0, st>>>(ref, qry, N, S, k, r2, idx, dist)
    if (ni <= 1) B200PC_SMALL(1);
    else if (ni <= 2) B200PC_SMALL(2);
    else if (ni <= 4) B200PC_SMALL(4);
    else if (ni <= 8) B200PC_SMALL(8);
    else if (ni <= 16) B200PC_SMALL(16);
    else B200PC_SMALL(32);
#undef B200PC_SMALL
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}

// decides whether the warp-per-query path serves this problem; returns -100 if not (caller streams instead)
int run_small(const float *ref, const float *qry, int B, int N, int S, int k, int form, int mode, float r2, int64_t *idx,
              float *dist, cudaStream_t st) {
    if (N > SMALL_MAX_N) return -100;
    const int forced = tuning().small_path;             // cached knob (-1: decide by size)
    if (forced >= 0) { if (forced == 0) return -100; }
    else {
        // per query: ~N/32*6 instructions of distances + k*(N/32*3+20) of selection per WARP, against
        // ~N*6/32 + k(1+ln(N/k))*100/32 per warp-lane in the streaming kernel: worth it for few queries or big k
        const long queries = (long)B * S;
        if (!(queries <= 4096 || (mode == MODE_TOPK && k * 4 >= N))) return -100;
    }
    if (mode == MODE_BALL) return launch_small<B200PC_FORM_QRY_NORM_FIRST, MODE_BALL>(ref, qry, B, N, S, k, r2, idx, nullptr, st);
    if (form == B200PC_FORM_REF_NORM_FIRST) return launch_small<B200PC_FORM_REF_NORM_FIRST, MODE_TOPK>(ref, qry, B, N, S, k, 0.f, idx, dist, st);
    if (form == B200PC_FORM_QRY_NORM_FIRST) return launch_small<B200PC_FORM_QRY_NORM_FIRST, MODE_TOPK>(ref, qry, B, N, S, k, 0.f, idx, dist, st);
    return launch_small<B200PC_FORM_DIRECT, MODE_TOPK>(ref, qry, B, N, S, k, 0.f, idx, dist, st);
}

}  // namespace b200pc
