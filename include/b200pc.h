/*
 * b200pc.h -- C ABI of libb200pc.so: the B200-native (sm_100a) geometric hot path behind
 * PointINet / PolyPCI / FlowNet3D-style models of jlx-dxl/Point-Cloud-Interpolation-.
 *
 * The reference has NO native interface: its hot path is plain Python functions imported by
 * name (Utils/Layers.py:8-10, Utils/Utils.py:9, PolyPCI/Models/Models_V1.py:12).  Each entry
 * point below states which reference function (file:line, relative to the reference root) it
 * replaces; the Python facade `b200pc` binds them 1:1 under the reference's own names
 * (see INTEGRATION.md for the binding a maintainer adds).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the function name ends in _host;
 *  - fp32 tensors are C-contiguous, point-major: xyz [B,N,3], features [B,N,C];
 *  - indices are int64 (torch.long), exactly as the reference produces/consumes them;
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work is
 *    stream-ordered, nothing synchronises, no global mutable state, re-entrant;
 *  - `workspace` is caller-owned device scratch of at least *_workspace_bytes(), 16-byte aligned (a search that needs
 *    it returns B200PC_EINVAL otherwise); its contents on entry do not matter, and it may be reused by the next call on the same
 *    stream;
 *  - every other buffer needs only its element's natural alignment (4 bytes for fp32 / int32, 8 for int64) unless its
 *    entry says otherwise; kernels that move 16-byte vectors check the alignment and take a scalar path without it;
 *  - return value: 0 on success, a negative B200PC_E* code on failure; the message is
 *    available from b200pc_last_error() (thread-local).  Nothing throws across this ABI.
 *  - there is NO CPU fallback: without a CUDA device every compute entry returns
 *    B200PC_ECUDA.
 *
 * Non-finite coordinates (NaN, +-inf: e.g. invalid LiDAR returns)
 *  - Top-k (knn, knn_i32, three_nn, feature_propagation, fusion_group, chamfer, rebuild_pack): a (query, ref) pair is a
 *    candidate only if its distance, in the call site's rounding, is finite.  Each row holds its candidates in ascending
 *    (distance, index) order, then index -1 with distance +inf in the remaining slots -- on every kernel path and for both
 *    index widths.  This departs from the reference's torch.topk, which ranks NaN distances last but still returns them.
 *  - Domain: for finite coordinates with |c| < 2^62 every distance in every form is finite (|r|^2, |q|^2 <= 3*2^124,
 *    |2q.r| <= 6*2^124, the expanded sum and |q-r|^2 <= 12*2^124 ~ 2.6e38 < FLT_MAX), so every finite pair is a candidate;
 *    a pair with a NaN or +-inf coordinate always has a non-finite distance.  Finite coordinates beyond 2^62 are outside
 *    the contract: indices stay in [-1, N) and nothing faults, but the results are not specified.
 *  - Ball query: a NaN distance is never a hit (see b200pc_ball_query).
 *  - Chamfer: a point without a candidate gets index -1 and minimum +inf, makes the loss +inf, and neither receives nor
 *    gives gradient.
 *  - FPS: a NaN or +inf distance never lowers a running minimum (the reference's `dist < distance` mask).
 *  - Consumers of indices (gather, group_points, three_interpolate) wrap -1 once to the last row, as Python indexing does.
 */
#ifndef B200PC_H
#define B200PC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200PC_OK        0
#define B200PC_EINVAL   -1 /* bad argument (k > N, null pointer, ...) */
#define B200PC_ECUDA    -2 /* CUDA runtime error (launch failure, no device, ...) */
#define B200PC_EWORKSPACE -3 /* workspace too small */

/* distance arithmetic ("form"): which fp32 rounding sequence a search reproduces */
#define B200PC_FORM_REF_NORM_FIRST 0 /* square_distance(refs, queries): kNN site Utils/Layers.py:51 */
#define B200PC_FORM_QRY_NORM_FIRST 1 /* square_distance(queries, refs): Utils/Pointnet2Utils.py:102, Utils/Layers.py:180 */
#define B200PC_FORM_DIRECT         2 /* sum((q-r)^2) with FMA accumulation: pytorch3d.ops.knn_points */

typedef void *b200pc_stream_t;

const char *b200pc_last_error(void);
int b200pc_version(void);
/* number of SMs of the current device, or a negative error code */
int b200pc_device_sm_count(void);
/* The B200PC_* tuning / debugging environment variables are read once, at the first launch, and cached (a launch never
 * calls getenv); this re-reads them.  For tests and A/B probes only -- the variables are not part of the ABI. */
void b200pc_tuning_reload(void);

/* ---- scratch sizing -------------------------------------------------------------------- */
/* scratch for any neighbour search (knn / ball_query / three_nn / chamfer) of S queries
 * against N refs per batch item with lists of length k (k = nsample for the ball query): the packed reference
 * records, the partial lists of a split search and, for the large top-k searches, the occupancy grid with the
 * cell-ordered copies of references and queries (csrc/search.cu section 1b; ~1.8 MB per batch item). */
size_t b200pc_search_workspace_bytes(int B, int N, int S, int k);
/* FPS keeps a cloud in the registers of one thread-block cluster and needs NO scratch: this query returns a token 256 and
 * b200pc_fps ignores its workspace arguments (both kept so that every compute entry has the same calling shape). */
size_t b200pc_fps_workspace_bytes(int B, int N);

/* ---- a1: square_distance(src, dst)  Utils/Pointnet2Utils.py:20-41 ---------------------- */
/* out[b,n,m] = ((-2*dot(src_n,dst_m)) + |src_n|^2) + |dst_m|^2, bit-identical to torch CPU. */
int b200pc_square_distance(const float *src, const float *dst, int B, int N, int M, float *out,
                           b200pc_stream_t stream);

/* ---- a4 / a8: k nearest refs for each query --------------------------------------------- */
/* form 0  -> Group.forward kNN branch, Utils/Layers.py:50-53 (exposed as knn_point)
 * form 2  -> pytorch3d.ops.knn_points(p1=qry, p2=ref, K=k) as called at Utils/Layers.py:220,
 *            311,393,430; PolyPCI/Models/Models_V1.py:113; PointINet20230424/models/layers.py:360
 * idx [B,S,k] int64 ascending by (distance, index), -1 / +inf where fewer than k refs have a finite distance (see
 * "Non-finite coordinates" above); dist [B,S,k] may be NULL.
 * k <= N (EINVAL otherwise, like torch.topk); the k-best lists live in shared memory: k up to ~780.  Empty work
 * (B == 0 or S == 0) returns OK without looking at the pointers.                                       */
int b200pc_knn(const float *ref, const float *qry, int B, int N, int S, int k, int form, int64_t *idx,
               float *dist, void *workspace, size_t workspace_bytes, b200pc_stream_t stream);

/* Ragged batches: pytorch3d.ops.knn_points(p1=qry, p2=ref, lengths1=qry_len, lengths2=ref_len, K=k) for clouds of
 * different sizes padded to [B,N,3] / [B,S,3] (LiDAR sweeps: the number of valid returns changes from frame to frame).
 * ref_len, qry_len: DEVICE int64 [B] (torch.long, as in pytorch3d); either may be NULL = every item full.  With
 * n_b = clamp(ref_len[b], 0, N) and s_b = clamp(qry_len[b], 0, S) -- clamped on the device, nothing is read back:
 *   rows q <  s_b: bit-identical (indices and distances) to b200pc_knn of qry[b,q] against ref[b, :n_b] -- same form, same
 *                  (distance, index) order, same non-finite rule; k > n_b (n_b == 0 included) ends the row in -1 / +inf;
 *   rows q >= s_b: every slot -1 / +inf.
 * No output depends on the contents of the padded rows (ref[b, n_b:], qry[b, s_b:]).  The work follows the lengths: an
 * item's refs fill ceil(n_b / 512) tiles, padded queries are not searched.  k <= N (EINVAL otherwise, like b200pc_knn);
 * workspace: b200pc_search_workspace_bytes(B, N, S, k) of the padded shape.  pytorch3d's zero padding of the empty slots
 * is the facade's business (b200pc.pytorch3d_shim); this entry keeps -1 / +inf.                                     */
int b200pc_knn_ragged(const float *ref, const float *qry, const int64_t *ref_len, const int64_t *qry_len, int B, int N,
                      int S, int k, int form, int64_t *idx, float *dist, void *workspace, size_t workspace_bytes,
                      b200pc_stream_t stream);

/* The same search with 32-bit indices (N < 2^31 always holds): for host-buffer callers that read the result back over
 * PCIe -- half the bytes of the int64 form the reference's tensors use.  Same order, same ties, -1 for unfilled slots. */
int b200pc_knn_i32(const float *ref, const float *qry, int B, int N, int S, int k, int form, int32_t *idx, float *dist,
                   void *workspace, size_t workspace_bytes, b200pc_stream_t stream);

/* ---- a2: query_ball_point(radius, nsample, xyz, new_xyz)  Utils/Pointnet2Utils.py:88-108 -- */
/* r2 = (float)(radius*radius) computed in double by the caller.  idx [B,S,nsample] int64:
 * the nsample lowest-index refs with d <= r2, padded with the first; N if the ball is empty.  (For finite inputs this is
 * the reference's NOT(d > r2); a NaN distance -- non-finite coordinates -- is never a hit, on either kernel path.) */
int b200pc_ball_query(const float *xyz, const float *new_xyz, int B, int N, int S, float r2, int nsample,
                      int64_t *idx, void *workspace, size_t workspace_bytes, b200pc_stream_t stream);

/* ---- a5: three_nn + weights  Utils/Layers.py:180-186 / Utils/Pointnet2Utils.py:297-303 ---- */
/* unknown [B,N,3] dense queries, known [B,S,3] sparse refs (S >= 3).
 * dist [B,N,3] (ascending, raw expanded-form values), idx [B,N,3] int64, weight [B,N,3] or NULL.
 * variant 0: d<1e-10 -> 1e-10, w=(1/d)/sum ; variant 1: w = 1/(d+1e-8) normalised.            */
int b200pc_three_nn(const float *unknown, const float *known, int B, int N, int S, int variant, float *dist,
                    int64_t *idx, float *weight, void *workspace, size_t workspace_bytes,
                    b200pc_stream_t stream);

/* ---- a5: three_interpolate  Utils/Layers.py:187-188 / Utils/Pointnet2Utils.py:304 -------- */
/* feat [B,S,C], idx [B,N,3], weight [B,N,3] -> out [B,N,C] = (f0*w0 + f1*w1) + f2*w2         */
int b200pc_three_interpolate(const float *feat, const int64_t *idx, const float *weight, int B, int S, int N,
                             int C, float *out, b200pc_stream_t stream);
/* gradients: gfeat [B,S,C] must be zero-filled by the caller (atomic accumulation);
 * gweight [B,N,3] may be NULL.  A neighbour out of range after one wrap gets no gradient (gweight 0, nothing into gfeat). */
int b200pc_three_interpolate_bwd(const float *gout, const float *feat, const int64_t *idx, const float *weight,
                                 int B, int S, int N, int C, float *gfeat, float *gweight,
                                 b200pc_stream_t stream);

/* a5 in ONE call: three-NN search -> inverse-distance weights -> mix (FeaturePropagation.forward Utils/Layers.py:180-188,
 * PointNetFeaturePropagation.forward Utils/Pointnet2Utils.py:297-304).  unknown [B,N,3], known [B,S,3], feat [B,S,C]
 * -> out [B,N,C]; idx [B,N,3] and weight [B,N,3] are returned for the backward pass (b200pc_three_interpolate_bwd);
 * the distances stay in the workspace.                                                         */
size_t b200pc_feature_propagation_workspace_bytes(int B, int N, int S);
int b200pc_feature_propagation(const float *unknown, const float *known, const float *feat, int B, int N, int S, int C,
                               int variant, float *out, int64_t *idx, float *weight, void *workspace,
                               size_t workspace_bytes, b200pc_stream_t stream);

/* ---- a3: farthest_point_sample(xyz, npoint)  Utils/Pointnet2Utils.py:64-85 --------------- */
/* start [B] int64: the first centroid of each cloud (the facade draws it with torch.randint
 * on the CPU generator exactly as the reference does).  idx [B,npoint] int64.                */
int b200pc_fps(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *idx, void *workspace,
               size_t workspace_bytes, b200pc_stream_t stream);

/* a7: Sample.forward (Utils/Layers.py:23-27) = farthest_point_sample + index_points(points, ind) behind one call:
 * idx [B,npoint] and the picks' coordinates new_xyz [B,npoint,3] (the FPS kernel followed by the gather kernel).     */
int b200pc_fps_sample(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *idx, float *new_xyz,
                      b200pc_stream_t stream);

/* ---- a6: index_points(points, idx)  Utils/Pointnet2Utils.py:44-61 ------------------------ */
/* points [B,N,C]; idx flattened to [B,R] (R = prod(idx.shape[1:])); out [B,R,C].
 * Negative indices wrap once (python semantics).  If oob_flag != NULL, *oob_flag (device int,
 * zero-initialised by the caller) is set to 1 when an index is out of range; such rows are
 * written as zeros.  The facade turns the flag into IndexError like the reference.           */
int b200pc_gather(const float *points, const int64_t *idx, int B, int N, int C, int64_t R, float *out,
                  int *oob_flag, b200pc_stream_t stream);
/* gpoints [B,N,C] must be zero-filled by the caller: gpoints[b, idx[b,r], :] += gout[b,r,:]  */
int b200pc_gather_bwd(const float *gout, const int64_t *idx, int B, int N, int C, int64_t R, float *gpoints,
                      b200pc_stream_t stream);

/* ---- f1 (SURVEY 8f rank 1): fused grouping  Utils/Layers.py:57-66 (Group.forward tail), ----
 *      Utils/Pointnet2Utils.py:243-253 (PointNetSetAbstractionMsg.forward grouping)            */
/* xyz [B,N,3], new_xyz [B,S,3], feat [B,N,D] (NULL when D == 0), idx [B,S,K] from knn / ball query
 * (negative indices wrap once and out-of-range rows read as zeros, like b200pc_gather).  out [B,3+D,K,S] -- the Conv2d input the
 * reference builds with two index_points, a subtraction, a cat and a permute+contiguous:
 *   xyz_first != 0 (Layers.py Group):   out[b,c,k,s]   = xyz[b,idx,c] - new_xyz[b,s,c]  (c < 3)
 *                                       out[b,3+d,k,s] = feat[b,idx,d]
 *   xyz_first == 0 (SA-MSG):            features in channels [0,D), relative xyz in [D,D+3).
 * Bit-identical to the reference (data movement + one fp32 subtraction).                     */
int b200pc_group_points(const float *xyz, const float *new_xyz, const float *feat, const int64_t *idx, int B, int N,
                        int S, int K, int D, int xyz_first, float *out, b200pc_stream_t stream);
/* grad_feat [B,N,D] must be zero-filled by the caller:
 * grad_feat[b, idx[b,s,k], d] += grad_out[b, (xyz_first ? 3 : 0) + d, k, s]
 * Out-of-range slots (after one wrap) get no gradient.                                       */
int b200pc_group_points_bwd(const float *grad_out, const int64_t *idx, int B, int N, int S, int K, int D,
                            int xyz_first, float *grad_feat, b200pc_stream_t stream);

/* ---- a8 / f2: points-fusion grouping  Utils/Layers.py:207-226 (PointsFusion.knn_group), :384-402 (knn_group_withI), ----
 *      PointINet20230424/models/layers.py:346-368; neighbour part of TransformerLayer.forward Utils/Layers.py:430-434     */
/* qry [B,S,3] (points1), ref [B,N,3] (points2), feat [B,N,Cf] or NULL (Cf == 0).  One call = knn_points(qry, ref, K=k,
 * return_nn=True) + resi + norm + cat + the three permute/contiguous copies:
 *   resi  [B,4,S,k]  = (nn - q) in channels 0..2, |nn - q| in channel 3
 *   nn    [B,3,S,k]  = the neighbours' coordinates
 *   gfeat [B,Cf,S,k] = knn_gather(feat, idx) in Conv2d layout (NULL when Cf == 0)
 *   idx   [B,S,k] int64, ascending (distance, index) like b200pc_knn(form 2); k <= N.
 * workspace: b200pc_search_workspace_bytes(B, N, S, k).                                           */
int b200pc_fusion_group(const float *qry, const float *ref, const float *feat, int B, int N, int S, int k, int Cf,
                        float *resi, float *nn, float *gfeat, int64_t *idx, void *workspace, size_t workspace_bytes,
                        b200pc_stream_t stream);

/* The score PointsFusion.forward gives every (point, neighbour) slot: the maximum over the channels of its point-wise MLP
 * (`torch.max(new_features, dim=1)`, Utils/Layers.py:276; upstream PointINet20230424/models/layers.py:416) when that MLP runs over
 * channels-last rows: x [rows, C] fp32 (C % 4 == 0, 16-byte aligned) -> out [rows] = max over C; NaN propagates like torch.max. */
int b200pc_channel_max(const float *x, int64_t rows, int C, float *out, b200pc_stream_t stream);

/* ---- a8 at C5: PolyPCI.rebuild for a QUERY SHARD  PolyPCI/Models/Models_V1.py:102-114 ------------------------------- */
/* knn_points(qry, ref, K=1, return_nn=True) for the S_local queries of this rank (queries [s_offset, s_offset+S_local) of
 * S_total), packed as 16-byte records {bit pattern of the int32 index, x, y, z} in s-major order:
 *   local_out [S_local, B, 4] fp32 (may be NULL);
 *   peer_out[p] (p < n_peers <= 8): base of a [S_total, B, 4] buffer of rank p, mapped into this process (symmetric /
 *   peer memory); this rank's slab [s_offset, s_offset+S_local) is written into every one of them by the same kernel,
 *   so the all-gather of the shard outputs needs no separate collective -- the ranks meet at a barrier afterwards.
 * With n_peers == 0 the records stay local (single GPU, or an NCCL all_gather of local_out by the caller).
 * peer_out is a HOST array of device pointers.  The records are stored 16 bytes at a time: local_out and every peer_out[p]
 * must be 16-byte aligned (B200PC_EINVAL before anything is launched otherwise).
 * workspace: b200pc_rebuild_pack_workspace_bytes().                                                                  */
size_t b200pc_rebuild_pack_workspace_bytes(int B, int N, int S_local);
int b200pc_rebuild_pack(const float *ref, const float *qry, int B, int N, int S_local, int s_offset, float *local_out,
                        void *const *peer_out, int n_peers, void *workspace, size_t workspace_bytes,
                        b200pc_stream_t stream);

/* ---- f4 (SURVEY 8f rank 4): PolyPCI polynomial fit + evaluation  ---------------------------
 *      PolyPCI/Models/Models_V1.py:116-124 (fitting_and_predict), call site :191-219           */
/* frames: HOST array of F (<= 16) device pointers, each a [B,per_batch] fp32 tensor (per_batch = 3*N for [B,3,N]
 * frames, in the reference's stacking order: key, forward 0, backward 0, forward 1, ...);
 * weights: device [B,F] float64, the least-squares weights of each batch item (linear in the data:
 * value = sum_f w[f] * frame_f -- see b200pc.polypci.poly_weights);  out [B,per_batch] fp32 =
 * (float) sum_f weights[b,f] * (double) frames[f][b,:], accumulated in float64 like numpy.           */
int b200pc_poly_predict(const float *const *frames, const double *weights, int B, int F, int64_t per_batch, float *out,
                        b200pc_stream_t stream);

/* ---- a9: chamfer_loss  Utils/Utils.py:39-48 -> pytorch3d.loss.chamfer_distance defaults --- */
/* x [B,N,3], y [B,M,3].  Outputs: per-point nearest squared distance and index in both
 * directions (dx,ix: [B,N]; dy,iy: [B,M]) and the scalar loss[1] =
 * mean_b( mean_i dx + mean_j dy ).  loss is written (not accumulated).  A point without a finite distance to the
 * other cloud gets index -1 and minimum +inf (the loss is then +inf); chamfer_bwd gives it no gradient.        */
int b200pc_chamfer_fwd(const float *x, const float *y, int B, int N, int M, float *dx, int64_t *ix, float *dy,
                       int64_t *iy, float *loss, void *workspace, size_t workspace_bytes,
                       b200pc_stream_t stream);
/* gx [B,N,3], gy [B,M,3] are written (zero-filled internally); gloss is a device scalar.     */
int b200pc_chamfer_bwd(const float *x, const float *y, const int64_t *ix, const int64_t *iy, const float *gloss,
                       int B, int N, int M, float *gx, float *gy, b200pc_stream_t stream);

/* Ragged Chamfer: pytorch3d.loss.chamfer_distance(x, y, x_lengths=x_len, y_lengths=y_len) with any point / batch reduction,
 * e.g. per-sample scores (batch_reduction=None) of interpolated frames against full-resolution sweeps of other sizes.
 * x [B,N,3], y [B,M,3] padded; x_len, y_len: DEVICE int64 [B] or NULL (full), clamped to [0,N] / [0,M] on the device.
 * Per point, as b200pc_chamfer_fwd against the other cloud's valid points (the two searches of b200pc_knn_ragged, K = 1,
 * form 2); padded points get index -1 and minimum +inf.  sums [B,2] fp32 = { sum of dx[b,i] over i < x_len[b],
 * sum of dy[b,j] over j < y_len[b] }, accumulated in double in a fixed order (the same bits on every run).  The reductions
 * ("mean": divide by max(len, 1); "sum"; batch "mean" / "sum" / none) are left to the caller.  An empty item sums to 0.
 * workspace: max(b200pc_search_workspace_bytes(B, M, N, 1), b200pc_search_workspace_bytes(B, N, M, 1)).            */
int b200pc_chamfer_ragged_fwd(const float *x, const float *y, const int64_t *x_len, const int64_t *y_len, int B, int N,
                              int M, float *dx, int64_t *ix, float *dy, int64_t *iy, float *sums, void *workspace,
                              size_t workspace_bytes, b200pc_stream_t stream);
/* gsums [B,2] (device) = d loss / d sums.  gx [B,N,3], gy [B,M,3] are written (zero-filled internally):
 * 2 gsums[b,0] (x_i - y_ix) into x_i and its negative into y_ix, likewise for y with gsums[b,1].  A padded point, or one
 * with index -1, gives and receives no gradient.                                                                     */
int b200pc_chamfer_ragged_bwd(const float *x, const float *y, const int64_t *ix, const int64_t *iy, const int64_t *x_len,
                              const int64_t *y_len, const float *gsums, int B, int N, int M, float *gx, float *gy,
                              b200pc_stream_t stream);

/* ---- measurement helper: sustained FP32 FMA throughput of the current device ------------- */
/* runs a register-resident FFMA2 chain kernel for `iters` iterations; *tflops receives the
 * measured rate (2 FLOP per FMA).  Used by bench.py for the FP32 roofline denominator.       */
int b200pc_fma_peak(int iters, double *tflops, double *ms, b200pc_stream_t stream);

/* ---- host-buffer convenience wrappers (non-torch callers) -------------------------------- */
/* Same semantics as above with HOST pointers: allocate, copy in, run, copy out, synchronise -- a convenience for plain C /
 * numpy callers, deliberately simple (pageable copies, a cudaMalloc per call, nothing overlapped).  Callers that stream
 * many clouds should hold device buffers and pinned host buffers themselves and overlap the copies of consecutive calls
 * the way b200pc.hostio.KnnHostPipeline does (two streams; b200pc_knn_i32 halves the read-back). */
int b200pc_knn_host(const float *ref, const float *qry, int B, int N, int S, int k, int form, int64_t *idx,
                    float *dist);
int b200pc_ball_query_host(const float *xyz, const float *new_xyz, int B, int N, int S, float r2, int nsample,
                           int64_t *idx);
/* Asynchronous host-buffer kNN for callers that pipeline by themselves: the H2D of ref / qry, the search and the D2H of the
 * int32 indices (and distances, if `dist` is not null) are all enqueued on `stream`; nothing is allocated, freed or
 * synchronised.  `arena` = caller-owned DEVICE scratch of b200pc_knn_async_host_workspace_bytes(B, N, S, k) bytes, 256-byte
 * aligned, in use until the stream has passed the call.  With two streams and two arenas the read-back of call i overlaps
 * the upload and search of call i+1 (what b200pc.hostio.KnnHostPipeline does above torch; host buffers should be pinned). */
size_t b200pc_knn_async_host_workspace_bytes(int B, int N, int S, int k);
int b200pc_knn_async_host(const float *ref, const float *qry, int B, int N, int S, int k, int form, int32_t *idx, float *dist,
                          void *arena, size_t arena_bytes, b200pc_stream_t stream);
int b200pc_fps_host(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *idx);

#ifdef __cplusplus
}
#endif
#endif /* B200PC_H */
