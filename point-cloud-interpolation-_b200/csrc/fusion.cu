// fusion.cu -- points-fusion grouping in one C call (SURVEY 8a row a8 / 8f rank 2).
//
// Replaces the body of PointsFusion.knn_group (Utils/Layers.py:207-226; upstream PointINet20230424/models/layers.py:346-368),
// knn_group_withI (Utils/Layers.py:384-402) and the neighbour part of TransformerLayer.forward (Utils/Layers.py:430-434):
//     _, nn_idx, nn = knn_points(points1, points2, K=k, return_nn=True)
//     points_resi  = nn - points1.unsqueeze(2).repeat(1, 1, k, 1)
//     grouped_dist = torch.norm(points_resi, dim=-1, keepdim=True)
//     new_features = torch.cat([points_resi, grouped_dist], dim=-1).permute(0, 3, 1, 2).contiguous()     [B,4,S,k]
//     nn.permute(0, 3, 1, 2).contiguous()                                                               [B,3,S,k]
//     knn_gather(features2, nn_idx).permute(0, 3, 1, 2).contiguous()                                    [B,Cf,S,k]
// which the reference runs as a search, two gathers and seven element-wise / copy kernels.  Here: the direct-form
// top-k search (search.cu, form 2) followed by ONE kernel that reads each neighbour once and writes the three
// Conv2d-layout tensors; thread e = (s, j) with j fastest, so every store instruction of a warp is 128 contiguous bytes
// of one channel plane.  |resi| is sqrt((rx*rx + ry*ry) + rz*rz), every step rounded on its own like torch's
// pow/sum/sqrt composition; values within 1e-5 relative of torch.norm (its accumulation order is not part of its contract).
#include <math_constants.h>

#include "common.cuh"
#include "search.cuh"

namespace b200pc {

__global__ void __launch_bounds__(256) fusion_features_kernel(const float *__restrict__ qry, const float *__restrict__ ref,
                                                              const float *__restrict__ feat, const int64_t *__restrict__ idx,
                                                              int N, int S, int K, int Cf, long total, float *__restrict__ resi,
                                                              float *__restrict__ nn, float *__restrict__ gfeat) {
    const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;      // e = (b*S + s)*K + j : the layout of idx and of every output plane
    if (e >= total) return;
    const long bs = e / K;
    const long b = bs / S;
    const long plane = (long)S * K, o = e - b * plane;               // offset inside one [S,K] plane
    const long i = idx[e];
    const bool ok = i >= 0 && i < N;                                 // -1: no candidate in this slot -> NaN features, like gathering nothing
    const float *q = qry + bs * 3;
    const float *r = ref + (b * N + (ok ? i : 0)) * 3;
    const float qn = __int_as_float(0x7fc00000);
    const float rx = ok ? __ldg(r + 0) : qn, ry = ok ? __ldg(r + 1) : qn, rz = ok ? __ldg(r + 2) : qn;
    const float dx = __fsub_rn(rx, __ldg(q + 0)), dy = __fsub_rn(ry, __ldg(q + 1)), dz = __fsub_rn(rz, __ldg(q + 2));
    const float n2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    B200PC_DEV_ASSERT(o >= 0 && o < plane && (!ok || (i >= 0 && i < N)));
    float *ro = resi + b * 4 * plane + o;
    __stcs(ro, dx); __stcs(ro + plane, dy); __stcs(ro + 2 * plane, dz); __stcs(ro + 3 * plane, __fsqrt_rn(n2));
    float *no = nn + b * 3 * plane + o;
    __stcs(no, rx); __stcs(no + plane, ry); __stcs(no + 2 * plane, rz);
    if (Cf > 0) {
        const float *fr = feat + (b * N + (ok ? i : 0)) * Cf;
        float *go = gfeat + b * Cf * plane + o;
        for (int c = 0; c < Cf; ++c) __stcs(go + c * plane, ok ? __ldg(fr + c) : qn);
    }
}

// PolyPCI.rebuild (PolyPCI/Models/Models_V1.py:102-114) for a query shard: nearest neighbour + its coordinates as ONE
// 16-byte record {index bits, x, y, z} per query, stored s-major ([S_total, B, 4]) so that the shards of the ranks are
// contiguous slabs.  The same thread stores the record into the local buffer and into every peer's buffer (peer-mapped
// symmetric memory: plain st.global over NVLink), i.e. the all-gather of the shard outputs happens from inside the
// producing kernel -- no separate collective launch; the ranks only meet at a barrier afterwards.
// PointsFusion.forward scores every (point, neighbour) slot by the MAXIMUM over the channels of its point-wise MLP
// (`torch.max(new_features, dim=1)`, Utils/Layers.py:276, upstream PointINet20230424/models/layers.py:416).  With the MLP run
// as GEMMs over channels-last rows that is a max over each contiguous row of C floats: one warp per row, 16-byte loads,
// five shuffles.  HBM bound (268 MB at C1); ATen's reduction takes 244 us for it, this 50 us.
__global__ void __launch_bounds__(256) channel_max_kernel(const float4 *__restrict__ x, long rows, int C4, float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long warp = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long)gridDim.x * blockDim.x) >> 5;
    for (long r = warp; r < rows; r += nwarps) {
        float m = -CUDART_INF_F;
        bool nan = false;
        for (int c = lane; c < C4; c += 32) {
            const float4 v = ldg_stream(x + r * C4 + c);
            nan = nan || v.x != v.x || v.y != v.y || v.z != v.z || v.w != v.w;
            m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        nan = __any_sync(0xffffffffu, nan);
        if (lane == 0) out[r] = nan ? __int_as_float(0x7fc00000) : m;       // torch.max propagates NaN
    }
}

constexpr int MAX_PEERS = 8;
struct PeerPtrs { float4 *p[MAX_PEERS]; };

__global__ void __launch_bounds__(256) rebuild_pack_kernel(const float *__restrict__ ref, const int32_t *__restrict__ idx, int B, int N,
                                                           int S_local, int s_offset, float4 *__restrict__ local_out,
                                                           PeerPtrs peers, int n_peers) {
    const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;      // e = s * B + b : the record's position inside the shard slab
    if (e >= (long)S_local * B) return;
    const int s = (int)(e / B), b = (int)(e - (long)s * B);
    const int i = idx[(size_t)b * S_local + s];
    float4 rec;
    rec.x = __int_as_float(i);
    if (i >= 0 && i < N) {
        const float *r = ref + ((size_t)b * N + i) * 3;
        rec.y = __ldg(r + 0); rec.z = __ldg(r + 1); rec.w = __ldg(r + 2);
    } else {
        rec.y = rec.z = rec.w = __int_as_float(0x7fc00000);
    }
    if (local_out) local_out[e] = rec;
    const size_t g = (size_t)s_offset * B + e;
#pragma unroll
    for (int p = 0; p < MAX_PEERS; ++p)
        if (p < n_peers) peers.p[p][g] = rec;
}

}  // namespace b200pc

using namespace b200pc;

namespace b200pc {
int run_topk_i32(const float *ref, const float *qry, int B, int N, int S, int k, int form, int32_t *idx32, float *dist,
                 void *ws, size_t ws_bytes, cudaStream_t st);
}

extern "C" int b200pc_channel_max(const float *x, int64_t rows, int C, float *out, b200pc_stream_t stream) {
    B200PC_REQUIRE(rows >= 0 && C >= 4 && C % 4 == 0, "channel_max: C=%d must be a positive multiple of 4", C);
    if (rows == 0) return B200PC_OK;
    B200PC_REQUIRE(x && out && (reinterpret_cast<uintptr_t>(x) & 15) == 0, "channel_max: null or misaligned pointer");
    long blocks = (rows + 7) / 8;
    const long cap = (long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    channel_max_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(reinterpret_cast<const float4 *>(x), (long)rows, C / 4, out);
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}

extern "C" size_t b200pc_rebuild_pack_workspace_bytes(int B, int N, int S_local) {
    if (B <= 0 || N <= 0 || S_local <= 0) return 256;
    return align_up(b200pc_search_workspace_bytes(B, N, S_local, 1), 256) + align_up((size_t)B * S_local * sizeof(int32_t), 256);
}

extern "C" int b200pc_rebuild_pack(const float *ref, const float *qry, int B, int N, int S_local, int s_offset, float *local_out,
                                   void *const *peer_out, int n_peers, void *workspace, size_t workspace_bytes,
                                   b200pc_stream_t stream) {
    B200PC_REQUIRE(B >= 0 && N >= 1 && S_local >= 0 && s_offset >= 0, "rebuild_pack: bad sizes");
    B200PC_REQUIRE(n_peers >= 0 && n_peers <= MAX_PEERS, "rebuild_pack: at most %d peer buffers", MAX_PEERS);
    if (B == 0 || S_local == 0) return B200PC_OK;
    B200PC_REQUIRE(ref && qry && (local_out || n_peers > 0), "rebuild_pack: null pointer");
    B200PC_REQUIRE(n_peers == 0 || peer_out, "rebuild_pack: n_peers=%d but no pointer array", n_peers);
    // the records are stored as float4: every destination must be 16-byte aligned (checked before anything is launched)
    B200PC_REQUIRE((reinterpret_cast<uintptr_t>(local_out) & 15) == 0, "rebuild_pack: local_out must be 16-byte aligned");
    for (int p = 0; p < n_peers; ++p)
        B200PC_REQUIRE(peer_out[p] && (reinterpret_cast<uintptr_t>(peer_out[p]) & 15) == 0,
                       "rebuild_pack: peer_out[%d] must be a non-null, 16-byte aligned pointer", p);
    if (!workspace || workspace_bytes < b200pc_rebuild_pack_workspace_bytes(B, N, S_local)) {
        set_error("rebuild_pack: workspace too small (%zu < %zu bytes)", workspace_bytes, b200pc_rebuild_pack_workspace_bytes(B, N, S_local));
        return B200PC_EWORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    const size_t search_bytes = align_up(b200pc_search_workspace_bytes(B, N, S_local, 1), 256);
    int32_t *idx = reinterpret_cast<int32_t *>(static_cast<char *>(workspace) + search_bytes);
    const int rc = run_topk_i32(ref, qry, B, N, S_local, 1, B200PC_FORM_DIRECT, idx, nullptr, workspace, search_bytes, st);
    if (rc != B200PC_OK) return rc;
    PeerPtrs pp;
    for (int p = 0; p < MAX_PEERS; ++p) pp.p[p] = p < n_peers ? static_cast<float4 *>(peer_out[p]) : nullptr;
    const long total = (long)S_local * B;
    rebuild_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(ref, idx, B, N, S_local, s_offset,
                                                                         reinterpret_cast<float4 *>(local_out), pp, n_peers);
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}

extern "C" int b200pc_fusion_group(const float *qry, const float *ref, const float *feat, int B, int N, int S, int k, int Cf,
                                   float *resi, float *nn, float *gfeat, int64_t *idx, void *workspace, size_t workspace_bytes,
                                   b200pc_stream_t stream) {
    B200PC_REQUIRE(B >= 0 && N >= 1 && S >= 0 && k >= 1 && Cf >= 0, "fusion_group: bad sizes B=%d N=%d S=%d k=%d Cf=%d", B, N, S, k, Cf);
    if (B == 0 || S == 0) return B200PC_OK;
    B200PC_REQUIRE(qry && ref && resi && nn && idx, "fusion_group: null pointer");
    B200PC_REQUIRE(Cf == 0 || (feat && gfeat), "fusion_group: Cf=%d feature channels but no feature pointers", Cf);
    cudaStream_t st = as_stream(stream);
    const int rc = run_topk(ref, qry, B, N, S, k, B200PC_FORM_DIRECT, idx, nullptr, workspace, workspace_bytes, st);
    if (rc != B200PC_OK) return rc;
    const long total = (long)B * S * k;
    B200PC_REQUIRE((total + 255) / 256 < (1L << 31), "fusion_group: problem too large for one launch");
    fusion_features_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(qry, ref, Cf ? feat : nullptr, idx, N, S, k, Cf, total, resi,
                                                                           nn, Cf ? gfeat : nullptr);
    B200PC_LAUNCH_CHECK();
    return B200PC_OK;
}
