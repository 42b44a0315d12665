// fps.cu -- farthest_point_sample (Utils/Pointnet2Utils.py:64-85 in the reference), sm_100a.
//
// npoint strictly sequential rounds; each round updates a running min-distance for every point
// and picks the FIRST arg-max.  The reference spends ~8 ATen launches per round; here one
// thread-block CLUSTER owns one cloud for the whole loop:
//   * every thread keeps P points (x,y,z,min-dist) in REGISTERS for all rounds; 512 threads x
//     P<=16 = 8192 points per CTA, up to 16 CTAs per cluster (131072 points);
//   * larger clouds, up to 262144 points, run the wide tier (fps_wide_kernel): every CTA holds up to
//     8192 more points in shared memory, their running minima still in registers;
//   * the update is packed fp32x2 math in the reference's exact rounding order
//     d = ((dx*dx + dy*dy) + dz*dz), dx = x - cx, every product rounded on its own (SURVEY Appendix A.5);
//   * arg-max: min-dists are >= +0, so their bit patterns order like unsigned ints:
//     the pair (bits, ~index) is reduced as one key: two REDUX per warp, ONE __syncthreads per round,
//     two REDUX over the warp keys (lowest index wins ties);
//   * across CTAs: each CTA pushes {max bits, index, centroid xyz} into every peer's shared memory with
//     st.async (DSMEM); the bytes complete on the receiver's mbarrier, so a round costs one DSMEM latency
//     and no cluster-wide barrier or membar; every thread then picks the winner locally.
// HBM traffic is N*12 bytes in and npoint*8 bytes out per cloud; the kernel is bound by the
// barrier latency of a round, reported by bench.py as microseconds per round.
#include <cooperative_groups.h>
#include <limits.h>
#include <stdlib.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace b200pc {

constexpr int FPS_T = 512;        // threads per CTA
constexpr int FPS_WARPS = FPS_T / 32;
constexpr int FPS_MAX_CLUSTER = 16;

struct __align__(16) FpsRecord {  // what a CTA tells its peers each round
    unsigned int bits;  // float bits of the CTA-wide max of min-dist
    int idx;            // lowest point index attaining it
    float x, y, z;      // its coordinates
    int pad[3];
};

// ---- round steps shared by the FPS kernels ----

// running-min update of P points against the last pick, reference rounding order, two points per instruction; returns the
// largest running minimum of the P points
template <int P>
__device__ __forceinline__ float fps_update(const float (&x)[P], const float (&y)[P], const float (&z)[P], float (&mind)[P],
                                            float cx, float cy, float cz) {
    float lmax = 0.f;
    if (P >= 2) {
        const f32x2 ncx = splat2(-cx), ncy = splat2(-cy), ncz = splat2(-cz);
#pragma unroll
        for (int p = 0; p < P; p += 2) {
            const f32x2 dx = add2(pack2(x[p], x[p + 1]), ncx);
            const f32x2 dy = add2(pack2(y[p], y[p + 1]), ncy);
            const f32x2 dz = add2(pack2(z[p], z[p + 1]), ncz);
            // Only the subtractions stay packed.  ptxas 12.9 contracts mul.rn.f32x2 feeding add.rn.f32x2 into FFMA2 (it even
            // folds fma(d, d, -0.0) back to a product first), which would turn the reference's (dx*dx + dy*dy) + dz*dz into
            // fma(dz,dz,fma(dy,dy,dx*dx)) and flip near-tied arg-max picks.  The scalar .rn intrinsics are never
            // contracted (tests/test_abi.py and tests/test_gpu_fps_large.py check the SASS of every FPS kernel: no FFMA2, no
            // FMUL2, no FFMA).
            float ax, bx, ay, by, az, bz;
            unpack2(dx, ax, bx); unpack2(dy, ay, by); unpack2(dz, az, bz);
            const float d0 = __fadd_rn(__fadd_rn(__fmul_rn(ax, ax), __fmul_rn(ay, ay)), __fmul_rn(az, az));
            const float d1 = __fadd_rn(__fadd_rn(__fmul_rn(bx, bx), __fmul_rn(by, by)), __fmul_rn(bz, bz));
            mind[p] = fminf(mind[p], d0);
            mind[p + 1] = fminf(mind[p + 1], d1);
            lmax = fmaxf(lmax, fmaxf(mind[p], mind[p + 1]));
        }
    } else {
        const float dx = __fadd_rn(x[0], -cx), dy = __fadd_rn(y[0], -cy), dz = __fadd_rn(z[0], -cz);
        const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
        mind[0] = fminf(mind[0], d);
        lmax = mind[0];
    }
    return lmax;
}

// cluster arg-max: all-to-all of one 32-byte record through DSMEM.  Each record is pushed with st.async, which completes
// bytes on the RECEIVER's mbarrier: no cluster-wide barrier and no membar per round, only the DSMEM latency.  rec / bar are
// this round's slots (they alternate with round parity, `phase` = (round >> 1) & 1).  Every warp then picks the winner among
// the C records in parallel: lane r holds record r, two REDUX give (max bits, lowest index), one ballot finds the lane that
// owns it.  This CTA's candidate is point ci, local slot cl of the lookup copy sx / sy / sz.  -> the winner's index; its
// coordinates in cx, cy, cz
__device__ __forceinline__ int fps_cluster_argmax(FpsRecord *rec, unsigned long long *bar, uint32_t phase, int C, int rank, int t,
                                                  int lane, unsigned int cbits, int ci, const float *sx, const float *sy,
                                                  const float *sz, int cl, float &cx, float &cy, float &cz) {
    const uint32_t my_bar = smem_u32(bar);
    if (t == 0) mbar_expect_tx(my_bar, (uint32_t)(C * sizeof(FpsRecord)));   // C records will land here
    if (t < C) {
        const uint32_t dst = map_to_rank(smem_u32(&rec[rank]), (uint32_t)t);
        const uint32_t rbar = map_to_rank(my_bar, (uint32_t)t);
        st_async_v4(dst, cbits, (uint32_t)ci, __float_as_uint(sx[cl]), __float_as_uint(sy[cl]), rbar);
        st_async_v4(dst + 16, __float_as_uint(sz[cl]), 0u, 0u, 0u, rbar);
    }
    mbar_wait_cluster(my_bar, phase);
    const FpsRecord mine = rec[lane < C ? lane : 0];
    const unsigned int vb = lane < C ? mine.bits : 0u;
    const unsigned int bb = __reduce_max_sync(0xffffffffu, vb);
    const unsigned int vinv = (lane < C && vb == bb) ? 0xffffffffu - (unsigned int)mine.idx : 0u;
    const unsigned int binv = __reduce_max_sync(0xffffffffu, vinv);
    const int src = __ffs(__ballot_sync(0xffffffffu, lane < C && vb == bb && vinv == binv)) - 1;
    cx = __shfl_sync(0xffffffffu, mine.x, src);
    cy = __shfl_sync(0xffffffffu, mine.y, src);
    cz = __shfl_sync(0xffffffffu, mine.z, src);
    return (int)(0xffffffffu - binv);
}

template <int P>
__global__ void __launch_bounds__(FPS_T) fps_kernel(const float *__restrict__ xyz, int N, int npoint,
                                                    const int64_t *__restrict__ start, int64_t *__restrict__ out) {
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    const int b = blockIdx.y;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int cta_base = rank * (FPS_T * P);

    extern __shared__ __align__(16) float fps_smem[];
    float *sx = fps_smem, *sy = sx + FPS_T * P, *sz = sy + FPS_T * P;
    __shared__ uint2 warp_key[2][FPS_WARPS];   // per-warp (max bits, ~index), double-buffered by round parity
    __shared__ FpsRecord rec[2][FPS_MAX_CLUSTER];
    __shared__ __align__(8) unsigned long long xbar[2];   // receive barriers of the record exchange

    const float *cloud = xyz + (size_t)b * N * 3;
    float x[P], y[P], z[P], mind[P];
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const int i = cta_base + p * FPS_T + t;
        if (i < N) {
            x[p] = cloud[i * 3 + 0]; y[p] = cloud[i * 3 + 1]; z[p] = cloud[i * 3 + 2];
            mind[p] = 1e10f;
        } else {  // padding: min-dist 0 loses every tie because its index is larger than any real one
            x[p] = 0.f; y[p] = 0.f; z[p] = 0.f; mind[p] = 0.f;
        }
        sx[p * FPS_T + t] = x[p]; sy[p * FPS_T + t] = y[p]; sz[p * FPS_T + t] = z[p];
    }
    if (t == 0) {
        mbar_init(smem_u32(&xbar[0]), 1); mbar_init(smem_u32(&xbar[1]), 1);
        mbar_fence_init();
    }
    int far = (int)start[b];
    far = far < 0 ? 0 : (far >= N ? N - 1 : far);      // a bad start index must not read outside the cloud
    float cx = cloud[far * 3 + 0], cy = cloud[far * 3 + 1], cz = cloud[far * 3 + 2];
    if (C > 1) cluster.sync(); else __syncthreads();

#ifdef B200PC_FPS_TIMING
    long long acc[5] = {0, 0, 0, 0, 0}, t0 = 0;
#define TICK(i) { const long long now = clock64(); acc[i] += now - t0; t0 = now; }
#else
#define TICK(i)
#endif
    for (int it = 0; it < npoint; ++it) {
#ifdef B200PC_FPS_TIMING
        t0 = clock64();
#endif
        B200PC_DEV_ASSERT(far >= 0 && far < N);
        if (rank == 0 && t == 0) out[(size_t)b * npoint + it] = far;
        if (it == npoint - 1) break;  // the last pick needs no further update

        // ---- running-min update, reference rounding order, two points per instruction ----
        const float lmax = fps_update<P>(x, y, z, mind, cx, cy, cz);

        TICK(0)
        // ---- block arg-max (first index) with ONE barrier: the pair (max bits, ~index) is reduced as a
        // 64-bit key -- two REDUX per warp, one shared write per warp, one __syncthreads, two REDUX again.
        int lp = 0;
#pragma unroll
        for (int p = P - 1; p >= 0; --p)
            if (mind[p] == lmax) lp = p;                       // first local point attaining the local max
        const unsigned int lbits = __float_as_uint(lmax);
        const unsigned int linv = 0xffffffffu - (unsigned int)(cta_base + lp * FPS_T + t);   // larger = lower index
        unsigned int wbits = __reduce_max_sync(0xffffffffu, lbits);
        unsigned int winv = __reduce_max_sync(0xffffffffu, lbits == wbits ? linv : 0u);
        TICK(1)
        if (lane == 0) warp_key[it & 1][warp] = make_uint2(wbits, winv);
        __syncthreads();
        TICK(2)
        const uint2 wk = warp_key[it & 1][lane & (FPS_WARPS - 1)];
        const unsigned int cbits = __reduce_max_sync(0xffffffffu, wk.x);
        const unsigned int cinv = __reduce_max_sync(0xffffffffu, wk.x == cbits ? wk.y : 0u);
        const int ci = (int)(0xffffffffu - cinv);
        const int cl = ci - cta_base;
        TICK(3)

        if (C == 1) {
            far = ci;
            cx = sx[cl]; cy = sy[cl]; cz = sz[cl];
        } else {
            const int par = it & 1;
            far = fps_cluster_argmax(rec[par], &xbar[par], (uint32_t)((it >> 1) & 1), C, rank, t, lane, cbits, ci, sx, sy, sz, cl,
                                     cx, cy, cz);
        }
        TICK(4)
    }
#ifdef B200PC_FPS_TIMING
    if (rank == 0 && t == 0 && b == 0)
        printf("fps timing (cycles/round, C=%d P=%d): update %lld | warp redux %lld | sts+bar %lld | block redux %lld | exchange %lld\n", C, P,
               acc[0] / npoint, acc[1] / npoint, acc[2] / npoint, acc[3] / npoint, acc[4] / npoint);
#endif
    if (C > 1) cluster.sync();  // nobody exits while a peer may still write into its shared memory
}

// ------------------------------------------------------------------------------------------------------------------
// Flat variant (round 2).  The two-level arg-max above costs, per round, a block barrier plus a second exchange stage:
// ~340 cycles of block reduction and 600-750 of record exchange on top of an ~100-cycle update.  Here every WARP sends its
// 8-byte key (max bits << 32 | ~index) straight to all CTAs of the cluster with st.async (one lane per destination); the
// bytes complete on each receiver's mbarrier, every warp then reduces the C*16 keys itself (4 per lane + two REDUX), and the
// winner's coordinates come from a copy of the WHOLE cloud that every CTA keeps in shared memory (N <= 16 384; larger
// clouds read them from global memory).  No __syncthreads in the loop, one cluster-wide dependency per round.
// It did NOT turn out uniformly faster: the st.async -> mbarrier -> wake path costs ~700 cycles even inside one CTA, so
// the launcher uses it only for 4-CTA clusters (see b200pc_fps).
// Arithmetic, tie rule and padding are those of fps_kernel: the picks are identical.
// ------------------------------------------------------------------------------------------------------------------
constexpr int FPS_FULL_COPY_MAX = 16384;      // points whose xyz fit beside the keys in one CTA's shared memory (196 608 bytes)

template <int P>
__global__ void __launch_bounds__(FPS_T) fps_flat_kernel(const float *__restrict__ xyz, int N, int npoint,
                                                         const int64_t *__restrict__ start, int64_t *__restrict__ out, int full_copy) {
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    const int b = blockIdx.y;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int cta_base = rank * (FPS_T * P);
    const int W = C * FPS_WARPS;                                       // warps of the cluster = keys per round
    const int gwid = rank * FPS_WARPS + warp;

    extern __shared__ __align__(16) float fps_smem[];                 // full_copy: xyz of the whole cloud, [N][3]
    __shared__ __align__(8) unsigned long long keys[2][FPS_MAX_CLUSTER * FPS_WARPS];   // per parity: one key per warp of the cluster
    __shared__ __align__(8) unsigned long long xbar[2];

    const float *cloud = xyz + (size_t)b * N * 3;
    float x[P], y[P], z[P], mind[P];
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const int i = cta_base + p * FPS_T + t;
        if (i < N) {
            x[p] = cloud[i * 3 + 0]; y[p] = cloud[i * 3 + 1]; z[p] = cloud[i * 3 + 2];
            mind[p] = 1e10f;
        } else {  // padding: min-dist 0 loses every tie because its index is larger than any real one
            x[p] = 0.f; y[p] = 0.f; z[p] = 0.f; mind[p] = 0.f;
        }
    }
    if (full_copy)
        for (int i = t; i < N * 3; i += FPS_T) fps_smem[i] = cloud[i];
    if (t == 0) {
        mbar_init(smem_u32(&xbar[0]), 1); mbar_init(smem_u32(&xbar[1]), 1);
        mbar_fence_init();
    }
    int far = (int)start[b];
    far = far < 0 ? 0 : (far >= N ? N - 1 : far);      // a bad start index must not read outside the cloud
    float cx = cloud[far * 3 + 0], cy = cloud[far * 3 + 1], cz = cloud[far * 3 + 2];
    cluster.sync();                                     // barriers initialised and copies visible everywhere

    for (int it = 0; it < npoint; ++it) {
        B200PC_DEV_ASSERT(far >= 0 && far < N);
        if (rank == 0 && t == 0) out[(size_t)b * npoint + it] = far;
        if (it == npoint - 1) break;  // the last pick needs no further update

        // ---- running-min update, reference rounding order (every product rounded on its own: see fps_update) ----
        const float lmax = fps_update<P>(x, y, z, mind, cx, cy, cz);
        int lp = 0;
#pragma unroll
        for (int p = P - 1; p >= 0; --p)
            if (mind[p] == lmax) lp = p;                       // first local point attaining the local max
        const unsigned int lbits = __float_as_uint(lmax);      // min-dists are >= +0: their bits order like unsigned ints
        const unsigned int linv = 0xffffffffu - (unsigned int)(cta_base + lp * FPS_T + t);   // larger = lower index
        const unsigned int wbits = __reduce_max_sync(0xffffffffu, lbits);
        const unsigned int winv = __reduce_max_sync(0xffffffffu, lbits == wbits ? linv : 0u);

        // ---- flat exchange: this warp's key goes to every CTA of the cluster; bytes complete on the receiver's barrier ----
        const int par = it & 1;
        const uint32_t my_bar = smem_u32(&xbar[par]);
        if (t == 0) mbar_expect_tx(my_bar, (uint32_t)(W * 8));             // W keys of 8 bytes will land here this round
        if (lane < C)
            st_async_b64(map_to_rank(smem_u32(&keys[par][gwid]), (uint32_t)lane), ((unsigned long long)wbits << 32) | winv,
                         map_to_rank(my_bar, (uint32_t)lane));
        mbar_wait_cluster(my_bar, (uint32_t)((it >> 1) & 1));
        unsigned int kb = 0u, ki = 0u;
        for (int j = lane; j < W; j += 32) {
            const unsigned long long k = keys[par][j];
            const unsigned int hb = (unsigned int)(k >> 32), lo = (unsigned int)k;
            if (hb > kb || (hb == kb && lo > ki)) { kb = hb; ki = lo; }
        }
        const unsigned int bb = __reduce_max_sync(0xffffffffu, kb);
        const unsigned int bi = __reduce_max_sync(0xffffffffu, kb == bb ? ki : 0u);
        far = (int)(0xffffffffu - bi);
        if (full_copy) { cx = fps_smem[far * 3 + 0]; cy = fps_smem[far * 3 + 1]; cz = fps_smem[far * 3 + 2]; }
        else { cx = __ldg(cloud + far * 3 + 0); cy = __ldg(cloud + far * 3 + 1); cz = __ldg(cloud + far * 3 + 2); }
    }
    cluster.sync();  // nobody exits while a peer may still write into its shared memory
}

template <int P>
static int launch_fps_flat(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *idx, int C,
                           cudaStream_t st) {
    auto kern = fps_flat_kernel<P>;
    const int full_copy = N <= FPS_FULL_COPY_MAX;
    const size_t smem = full_copy ? (size_t)N * 3 * sizeof(float) : 16;
    B200PC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (C > 8) B200PC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C, B, 1);
    cfg.blockDim = dim3(FPS_T, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    B200PC_CUDA(cudaLaunchKernelEx(&cfg, kern, xyz, N, npoint, start, idx, full_copy));
    return B200PC_OK;
}

template <int P>
static int launch_fps(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *idx, int C,
                      cudaStream_t st) {
    auto kern = fps_kernel<P>;
    const size_t smem = (size_t)3 * FPS_T * P * sizeof(float);
    B200PC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (C > 8) B200PC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C, B, 1);
    cfg.blockDim = dim3(FPS_T, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    B200PC_CUDA(cudaLaunchKernelEx(&cfg, kern, xyz, N, npoint, start, idx));
    return B200PC_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Wide tier: clouds the registers of one cluster cannot hold (131 073 .. 262 144 points by default), still one cluster of
// C CTAs per cloud, all state on chip and no workspace.  Every CTA owns a contiguous slice of S = ceil(N / C) points: the
// first 8 192 live in registers as in fps_kernel<16>, the other S - 8 192 (at most 8 192, Q per thread) in shared memory.
// Their coordinates are the tail of the x/y/z lookup copy every CTA keeps anyway (3 * 512 * (16 + Q) floats, 196 608 bytes
// at Q = 16); their running minima stay in registers, Q more per thread.  Balancing the slices keeps the shared part small
// for clouds just above the register capacity: a 133 312-point sweep puts 140 points per CTA there (Q = 1).
// Slot s of thread t (s < 16: register point s, s >= 16: shared point s - 16) is point base + s * 512 + t of the cloud, so
// a thread's slots are in index order and its first local arg-max is the lowest index.  Slots at or past the slice's end are
// padding with min-dist 0: they tie only when every real point has min-dist 0, and then point 0 of the cloud wins.
// Arithmetic (fps_update), tie rule and the two-level exchange are those of fps_kernel: the picks are identical.
// ------------------------------------------------------------------------------------------------------------------
constexpr int FPS_WIDE_P = 16;                          // register points per thread
constexpr int FPS_WIDE_MAX_Q = 16;                      // shared-memory points per thread
constexpr int FPS_MAX_N = FPS_MAX_CLUSTER * FPS_T * (FPS_WIDE_P + FPS_WIDE_MAX_Q);   // 262 144

template <int Q>
__global__ void __launch_bounds__(FPS_T) fps_wide_kernel(const float *__restrict__ xyz, int N, int npoint,
                                                         const int64_t *__restrict__ start, int64_t *__restrict__ out) {
    constexpr int P = FPS_WIDE_P, L = FPS_T * (P + Q);  // L: slots per CTA
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    const int b = blockIdx.y;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int S = (N + C - 1) / C;
    const int base = rank * S;                          // first point of this CTA's slice
    const int len = min(S, N - base);                   // points in the slice; slots from len on are padding
    B200PC_DEV_ASSERT(len > 0 && len <= L);

    extern __shared__ __align__(16) float fps_smem[];
    float *sx = fps_smem, *sy = sx + L, *sz = sy + L;
    __shared__ uint2 warp_key[2][FPS_WARPS];
    __shared__ FpsRecord rec[2][FPS_MAX_CLUSTER];
    __shared__ __align__(8) unsigned long long xbar[2];

    const float *cloud = xyz + (size_t)b * N * 3;
    float x[P], y[P], z[P], mind[P], qmind[Q];
#pragma unroll
    for (int s = 0; s < P + Q; ++s) {
        const int l = s * FPS_T + t;
        float px = 0.f, py = 0.f, pz = 0.f, m = 0.f;
        if (l < len) {
            const int i = base + l;
            B200PC_DEV_ASSERT(i < N);
            px = cloud[i * 3 + 0]; py = cloud[i * 3 + 1]; pz = cloud[i * 3 + 2];
            m = 1e10f;
        }
        sx[l] = px; sy[l] = py; sz[l] = pz;
        if (s < P) { x[s] = px; y[s] = py; z[s] = pz; mind[s] = m; }
        else qmind[s - P] = m;
    }
    if (t == 0) {
        mbar_init(smem_u32(&xbar[0]), 1); mbar_init(smem_u32(&xbar[1]), 1);
        mbar_fence_init();
    }
    int far = (int)start[b];
    far = far < 0 ? 0 : (far >= N ? N - 1 : far);      // a bad start index must not read outside the cloud
    float cx = cloud[far * 3 + 0], cy = cloud[far * 3 + 1], cz = cloud[far * 3 + 2];
    if (C > 1) cluster.sync(); else __syncthreads();   // barriers initialised, shared points stored

    for (int it = 0; it < npoint; ++it) {
        B200PC_DEV_ASSERT(far >= 0 && far < N);
        if (rank == 0 && t == 0) out[(size_t)b * npoint + it] = far;
        if (it == npoint - 1) break;  // the last pick needs no further update

        // ---- running-min update of the register points, then of the shared-memory points ----
        float qx[Q], qy[Q], qz[Q];
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            const int l = (P + q) * FPS_T + t;
            qx[q] = sx[l]; qy[q] = sy[l]; qz[q] = sz[l];
        }
        const float lmax = fmaxf(fps_update<P>(x, y, z, mind, cx, cy, cz), fps_update<Q>(qx, qy, qz, qmind, cx, cy, cz));

        // ---- block arg-max over the global index (as in fps_kernel): shared slots follow the register slots of a thread ----
        int ls = 0;
#pragma unroll
        for (int q = Q - 1; q >= 0; --q)
            if (qmind[q] == lmax) ls = P + q;
#pragma unroll
        for (int p = P - 1; p >= 0; --p)
            if (mind[p] == lmax) ls = p;                       // first local slot attaining the local max
        const unsigned int lbits = __float_as_uint(lmax);
        const unsigned int linv = 0xffffffffu - (unsigned int)(base + ls * FPS_T + t);   // larger = lower index
        const unsigned int wbits = __reduce_max_sync(0xffffffffu, lbits);
        const unsigned int winv = __reduce_max_sync(0xffffffffu, lbits == wbits ? linv : 0u);
        if (lane == 0) warp_key[it & 1][warp] = make_uint2(wbits, winv);
        __syncthreads();
        const uint2 wk = warp_key[it & 1][lane & (FPS_WARPS - 1)];
        const unsigned int cbits = __reduce_max_sync(0xffffffffu, wk.x);
        const unsigned int cinv = __reduce_max_sync(0xffffffffu, wk.x == cbits ? wk.y : 0u);
        const int ci = (int)(0xffffffffu - cinv);
        const int cl = ci - base;
        B200PC_DEV_ASSERT(cl >= 0 && cl < len);

        if (C == 1) {
            far = ci;
            cx = sx[cl]; cy = sy[cl]; cz = sz[cl];
        } else {
            const int par = it & 1;
            far = fps_cluster_argmax(rec[par], &xbar[par], (uint32_t)((it >> 1) & 1), C, rank, t, lane, cbits, ci, sx, sy, sz, cl,
                                     cx, cy, cz);
        }
    }
    if (C > 1) cluster.sync();  // nobody exits while a peer may still write into its shared memory
}

template <int Q>
static int launch_fps_wide(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *idx, int C,
                           cudaStream_t st) {
    auto kern = fps_wide_kernel<Q>;
    const size_t smem = (size_t)3 * FPS_T * (FPS_WIDE_P + Q) * sizeof(float);
    B200PC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (C > 8) B200PC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C, B, 1);
    cfg.blockDim = dim3(FPS_T, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    // one CTA per SM at this much shared memory: a device (or a partition of one) without C such SMs in one GPC cannot run
    // the cluster at all, so ask before launching instead of failing at launch
    int clusters = 0;
    B200PC_CUDA(cudaOccupancyMaxActiveClusters(&clusters, kern, &cfg));
    if (clusters < 1) {
        set_error("fps: N=%d needs a cluster of %d CTAs with %zu bytes of dynamic shared memory each, which this device cannot "
                  "schedule", N, C, smem);
        return B200PC_ECUDA;
    }
    if (tuning().debug_plan)
        fprintf(stderr, "b200pc fps wide tier: at most %d clusters of %d CTAs co-resident, %zu bytes of dynamic shared memory per CTA\n",
                clusters, C, smem);
    B200PC_CUDA(cudaLaunchKernelEx(&cfg, kern, xyz, N, npoint, start, idx));
    return B200PC_OK;
}

// cluster size C, register points per thread P and shared-memory points per thread Q (0: fps_kernel / fps_flat_kernel,
// >= 1: fps_wide_kernel) for a cloud of N points in a batch of B
static void fps_shape(int B, int N, int *C_out, int *P_out, int *Q_out) {
    const int sms = sm_count();
    // Measured (tools/fps_timing_probe.py, tools/fps_time.py): a single CTA needs ~560 cycles per round plus ~12 per
    // point held by a thread; a cluster adds ~600-750 cycles of DSMEM exchange.  So one CTA whenever the cloud fits
    // its registers (8192 points); otherwise spread to ~4 points per thread while the grid stays within half of the
    // SMs (16384 points: 0.61 us/round at C=8 for B<=8, 0.70 at C=4 for B=16, against 0.88 at C=2).
    int C = 1;
    while (C < FPS_MAX_CLUSTER && (long)C * FPS_T * 16 < N) C *= 2;
    if (C > 1)
        while (C < 8 && (long)B * C * 4 <= sms && (long)C * FPS_T * 4 < N) C *= 2;
    {   // tuning override (cached; not part of the ABI); a cluster too small for the cloud in registers runs the wide tier
        const int f = tuning().fps_cluster;
        if (f >= 1 && f <= FPS_MAX_CLUSTER && (long)f * FPS_T * (FPS_WIDE_P + FPS_WIDE_MAX_Q) >= N) C = f;
    }
    int P = 1, Q = 0;
    if ((long)C * FPS_T * FPS_WIDE_P < N) {             // wide tier: 16 register points per thread, the rest of a slice shared
        const int shared_points = (N + C - 1) / C - FPS_T * FPS_WIDE_P;
        P = FPS_WIDE_P; Q = 1;
        while (FPS_T * Q < shared_points) Q *= 2;
    } else {
        while ((long)C * FPS_T * P < N) P *= 2;
    }
    *C_out = C; *P_out = P; *Q_out = Q;
}

}  // namespace b200pc

using namespace b200pc;

extern "C" size_t b200pc_fps_workspace_bytes(int, int) { return 256; }

extern "C" int b200pc_fps(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *idx, void *,
                          size_t, b200pc_stream_t stream) {
    B200PC_REQUIRE(B >= 0 && N >= 1 && npoint >= 0, "fps: bad sizes B=%d N=%d npoint=%d", B, N, npoint);
    B200PC_REQUIRE(N <= FPS_MAX_N, "fps: N=%d exceeds the %d points one cluster can hold", N, FPS_MAX_N);
    if (B == 0 || npoint == 0) return B200PC_OK;
    B200PC_REQUIRE(xyz && start && idx, "fps: null pointer");
    int C, P, Q;
    fps_shape(B, N, &C, &P, &Q);
    cudaStream_t st = as_stream(stream);
    // Measured at 16 384 points (tools/fps_sweep.py, us per round, two-level / flat): C=2 0.98 / 1.05, C=4 0.75 / 0.67,
    // C=8 0.62 / 0.68, C=16 0.63 / 0.94; one CTA 0.29 / 0.50.  The flat exchange wins exactly where the cluster is 4 CTAs
    // (batches of >= 10 clouds, e.g. C3: 3.05 -> 2.70 ms); everywhere else the two-level kernel stays.  The wide tier
    // always exchanges in two levels.
    const int flat = tuning().fps_flat;
    const bool use_flat = Q == 0 && (flat > 0 || (flat < 0 && C == 4));
    if (tuning().debug_plan) {
        if (Q == 0)
            fprintf(stderr, "b200pc fps plan: B=%d N=%d npoint=%d -> cluster %d, %d points/thread, exchange %s\n", B, N, npoint, C,
                    P, use_flat ? "flat" : "two-level");
        else
            fprintf(stderr, "b200pc fps plan: B=%d N=%d npoint=%d -> cluster %d, %d points/thread, exchange two-level, shared %d "
                    "points/thread\n", B, N, npoint, C, P, Q);
    }
    if (Q > 0) {
        switch (Q) {
            case 1: return launch_fps_wide<1>(xyz, B, N, npoint, start, idx, C, st);
            case 2: return launch_fps_wide<2>(xyz, B, N, npoint, start, idx, C, st);
            case 4: return launch_fps_wide<4>(xyz, B, N, npoint, start, idx, C, st);
            case 8: return launch_fps_wide<8>(xyz, B, N, npoint, start, idx, C, st);
            default: return launch_fps_wide<16>(xyz, B, N, npoint, start, idx, C, st);
        }
    }
    if (use_flat) {
        switch (P) {
            case 1: return launch_fps_flat<1>(xyz, B, N, npoint, start, idx, C, st);
            case 2: return launch_fps_flat<2>(xyz, B, N, npoint, start, idx, C, st);
            case 4: return launch_fps_flat<4>(xyz, B, N, npoint, start, idx, C, st);
            case 8: return launch_fps_flat<8>(xyz, B, N, npoint, start, idx, C, st);
            default: return launch_fps_flat<16>(xyz, B, N, npoint, start, idx, C, st);
        }
    }
    switch (P) {
        case 1: return launch_fps<1>(xyz, B, N, npoint, start, idx, C, st);
        case 2: return launch_fps<2>(xyz, B, N, npoint, start, idx, C, st);
        case 4: return launch_fps<4>(xyz, B, N, npoint, start, idx, C, st);
        case 8: return launch_fps<8>(xyz, B, N, npoint, start, idx, C, st);
        default: return launch_fps<16>(xyz, B, N, npoint, start, idx, C, st);
    }
}

// a7: Sample.forward (Utils/Layers.py:23-27) = farthest_point_sample + index_points(points, ind) behind one entry point.
// Two launches on purpose: writing the picks' coordinates from inside the round loop of fps_kernel cost 3.7 % per call
// (0.652 vs 0.629 ms for 16 384 -> 1 024 on the same box), the separate 3-channel gather 0.6 % (0.630 ms).
extern "C" int b200pc_gather(const float *points, const int64_t *idx, int B, int N, int C, int64_t R, float *out, int *oob_flag,
                             b200pc_stream_t stream);

extern "C" int b200pc_fps_sample(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *idx,
                                 float *new_xyz, b200pc_stream_t stream) {
    B200PC_REQUIRE(new_xyz || B == 0 || npoint == 0, "fps_sample: null output pointer");
    const int rc = b200pc_fps(xyz, B, N, npoint, start, idx, nullptr, 0, stream);
    if (rc != B200PC_OK || B == 0 || npoint == 0) return rc;
    return b200pc_gather(xyz, idx, B, N, 3, npoint, new_xyz, nullptr, stream);
}
