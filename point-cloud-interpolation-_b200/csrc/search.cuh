// search.cuh -- internal C++ interface of the brute-force neighbour search (search.cu)
#pragma once
#include "common.cuh"

namespace b200pc {

enum SearchMode { MODE_TOPK = 0, MODE_BALL = 1 };

// Ragged batches (b200pc_knn_ragged, b200pc_chamfer_ragged_*): item b has clamp(len[b], 0, full) valid points; a null
// length array means every item is full.  The clamp happens here, on the device: nothing is read back to the host.
__device__ __forceinline__ int item_len(const int64_t *len, int b, int full) {
    if (!len) return full;
    const int64_t v = __ldg(len + b);
    return v < 0 ? 0 : (v > (int64_t)full ? full : (int)v);
}

// Geometry of one search launch, derived deterministically from the problem size so that the
// workspace-size query and the launcher always agree.
struct SearchPlan {
    int q_per_thread;     // queries owned by one thread
    int consumer_warps;   // warps per CTA (all of them consume tiles; there is no producer warp)
    int q_per_block;      // = q_per_thread * consumer_warps * 32
    int n_pad;            // refs padded to a multiple of the tile
    int n_tiles;
    int n_split;          // ref range split across gridDim.z (partial lists merged afterwards)
    int tiles_per_split;
    size_t smem_bytes;
    size_t packed_bytes;  // workspace: packed ref tiles
    size_t part_bytes;    // workspace: partial lists (n_split > 1)
    size_t grid_bytes;    // workspace: occupancy grid (counters, sorted copies, starting thresholds) of a warm-started top-k search, else 0
    int grid_sorted;      // 1: refs and queries are visited in cell order (search.cu section 1b)
    size_t total_bytes;
};

// k: list length (k for top-k, nsample for ball).  Returns false if k cannot be served.
bool plan_search(int B, int N, int S, int k, int mode, SearchPlan *plan);

// Top-k search: idx [B,S,k] int64 and/or dist [B,S,k] (either may be null, not both).  ref_len / qry_len: [B] device
// lengths of a ragged batch (b200pc_knn_ragged), null = every item full.
int run_topk(const float *ref, const float *qry, int B, int N, int S, int k, int form, int64_t *idx, float *dist,
             void *ws, size_t ws_bytes, cudaStream_t st, const int64_t *ref_len = nullptr, const int64_t *qry_len = nullptr);

int run_ball(const float *ref, const float *qry, int B, int N, int S, float r2, int nsample, int64_t *idx,
             void *ws, size_t ws_bytes, cudaStream_t st);

// warp-per-query path for N <= 1024 (small_search.cu); returns -100 when it declines the problem
int run_small(const float *ref, const float *qry, const int64_t *ref_len, const int64_t *qry_len, int B, int N, int S, int k, int form,
              int mode, float r2, int64_t *idx, float *dist, cudaStream_t st);

}  // namespace b200pc
