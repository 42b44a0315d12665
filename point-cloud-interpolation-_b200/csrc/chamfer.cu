// chamfer.cu -- chamfer_loss (Utils/Utils.py:39-48 -> pytorch3d.loss.chamfer_distance defaults).
//   loss = mean_b [ mean_i min_j |x_i - y_j|^2 + mean_j min_i |x_i - y_j|^2 ]
// Forward = two K=1 direct-form searches (search.cu, no [N,M] matrix) + one deterministic
// reduction; the per-point minima / arg-minima are kept for the backward pass, which is a pair of
// scatter kernels (the nearest-neighbour assignment is piecewise constant, so the gradient is
// 2*(x_i - y_nn(i)) through both directions).
#include "common.cuh"
#include "search.cuh"

namespace b200pc {

// single CTA, double accumulation in a fixed order: deterministic, and exact enough that the
// scalar agrees with a float64 host sum to ~1e-7 relative.
__global__ void __launch_bounds__(1024) chamfer_reduce_kernel(const float *__restrict__ dx, const float *__restrict__ dy,
                                                              int B, int N, int M, float *__restrict__ loss) {
    __shared__ double part[32];
    double acc = 0.0;
    const double wx = 1.0 / ((double)N * B), wy = 1.0 / ((double)M * B);
    for (long i = threadIdx.x; i < (long)B * N; i += blockDim.x) acc += (double)dx[i] * wx;
    for (long i = threadIdx.x; i < (long)B * M; i += blockDim.x) acc += (double)dy[i] * wy;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) loss[0] = (float)v;
    }
}

// for every a_i with nearest b_j:  g = scale * 2 * (a_i - b_j);  ga[i] += g;  gb[j] -= g
__global__ void __launch_bounds__(256) chamfer_bwd_kernel(const float *__restrict__ a, const float *__restrict__ bpts,
                                                          const int64_t *__restrict__ nn, const float *__restrict__ gloss,
                                                          int Na, int Nb, long rows, float scale, float *__restrict__ ga,
                                                          float *__restrict__ gb) {
    const long r = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const long b = r / Na;
    const long j = nn[r];
    if (j < 0 || j >= Nb) return;          // a point without a finite distance (non-finite coordinates) has index -1: no gradient
    const float s = 2.0f * scale * gloss[0];
    const float *pa = a + r * 3;
    const float *pb = bpts + (b * Nb + j) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float g = s * (pa[c] - pb[c]);
        atomicAdd(ga + r * 3 + c, g);
        atomicAdd(gb + (b * Nb + j) * 3 + c, -g);
    }
}

}  // namespace b200pc

using namespace b200pc;

extern "C" int b200pc_chamfer_fwd(const float *x, const float *y, int B, int N, int M, float *dx, int64_t *ix, float *dy,
                                  int64_t *iy, float *loss, void *workspace, size_t workspace_bytes,
                                  b200pc_stream_t stream) {
    B200PC_REQUIRE(x && y && dx && ix && dy && iy && loss, "chamfer_fwd: null pointer");
    B200PC_REQUIRE(B >= 1 && N >= 1 && M >= 1, "chamfer_fwd: empty clouds are not supported");
    cudaStream_t st = as_stream(stream);
    int rc = run_topk(y, x, B, M, N, 1, B200PC_FORM_DIRECT, ix, dx, workspace, workspace_bytes, st);
    if (rc != B200PC_OK) return rc;
    rc = run_topk(x, y, B, N, M, 1, B200PC_FORM_DIRECT, iy, dy, workspace, workspace_bytes, st);
    if (rc != B200PC_OK) return rc;
    chamfer_reduce_kernel<<<1, 1024, 0, st>>>(dx, dy, B, N, M, loss);
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}

extern "C" int b200pc_chamfer_bwd(const float *x, const float *y, const int64_t *ix, const int64_t *iy, const float *gloss,
                                  int B, int N, int M, float *gx, float *gy, b200pc_stream_t stream) {
    B200PC_REQUIRE(x && y && ix && iy && gloss && gx && gy, "chamfer_bwd: null pointer");
    cudaStream_t st = as_stream(stream);
    B200PC_CUDA(cudaMemsetAsync(gx, 0, (size_t)B * N * 3 * sizeof(float), st));
    B200PC_CUDA(cudaMemsetAsync(gy, 0, (size_t)B * M * 3 * sizeof(float), st));
    const long rx = (long)B * N, ry = (long)B * M;
    chamfer_bwd_kernel<<<(int)((rx + 255) / 256), 256, 0, st>>>(x, y, ix, gloss, N, M, rx, 1.0f / ((float)N * B), gx, gy);
    B200PC_LAUNCH_CHECK();
    chamfer_bwd_kernel<<<(int)((ry + 255) / 256), 256, 0, st>>>(y, x, iy, gloss, M, N, ry, 1.0f / ((float)M * B), gy, gx);
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}
