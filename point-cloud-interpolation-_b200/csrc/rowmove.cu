// rowmove.cu -- group_points on the asynchronous-copy path (sm_100a): the 32 feature rows of a tile travel global -> shared
// with warp-cooperative 16-byte cp.async (SASS LDGSTS: no register is held while a row is in flight, a 512-byte row is ONE
// instruction, every copy is coalesced), tiles complete through cp.async groups, and each lane then reads ITS row from
// shared memory and writes channel after channel of the Conv2d layout.
//
//   group_async_kernel    Group.forward tail      Utils/Layers.py:57-66, SA-MSG grouping Utils/Pointnet2Utils.py:243-253
//
// Why: in the register-path kernel (group.cu) every lane walks its OWN gathered row, i.e. one L1 wavefront per 32-byte sector
// of every row: 580 wavefront-cycles per 8 KB of output, l1tex 82 % busy (profiles/r02_ncu_rowmovers_shipped.txt).  Copying
// the rows cooperatively takes the gather off the LSU's per-sector path (l1tex 46 %).  The kernel is then bound by one
// warp's dependent chain (index -> copy -> shared load -> store), so it runs as many warps as shared memory allows with a
// one-stage ring: 16 warps at D <= 64, where it beats the register kernel (90.7 vs 102.7 us at C3); with 10 warps at
// D = 128 it loses (210 vs 183 us) and the register kernel keeps those shapes.
// Measured and removed (profiles/r02_notes.md section 3): one cp.async.bulk (TMA) PER ROW -- the TMA unit serves ~1 request
// per 46-60 cycles per SM whatever its size, 10 B/clk/SM for 512-byte rows (three_interpolate 60 -> 163 us, group_points
// 108 -> 167 us); asynchronous-copy versions of index_points (26 vs 19 us) and three_interpolate (150 vs 51 us: 185
// instructions per row against 93) -- the register kernels of gather.cu stay.
#include <type_traits>

#include "common.cuh"

namespace b200pc {

constexpr size_t RM_SMEM_BUDGET = 200 * 1024;     // per CTA (one CTA per SM), leaves room for the driver's reservation

__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void *src_gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ float4 lds_f4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}

// One row (row_bytes, a multiple of 16) global -> shared by the whole warp.
__device__ __forceinline__ void warp_copy_row(uint32_t dst, const char *src, uint32_t row_bytes, int lane) {
    for (uint32_t o = 16u * lane; o < row_bytes; o += 512u) cp_async16(dst + o, src + o);
}

// ---------------------------------------------------------------------------------------------
// All index arithmetic below is 32-bit (the launchers check rows, B*N and B*S against 2^31): a 64-bit division is a
// ~100-instruction subroutine call, and these kernels run 4-8 warps per SM -- they are bound by the instruction stream
// of a single warp per scheduler, not by a pipe (ncu of the first version: 258 instructions per interpolated row).
// ---------------------------------------------------------------------------------------------
// group_points: out[b, c, k, s] from rows gathered by idx[b, s, k]  (the Conv2d layout)
// A unit = 32 consecutive centres s x a range of slots k.  Per slot: the 32 feature rows are copied by the whole warp
// (coalesced) into a padded tile (row stride chosen so that 16-byte reads of 8 lanes hit 32 different banks); each lane
// then reads ITS row with 16-byte shared loads and writes channel after channel: every store instruction is 128
// contiguous bytes.  The unit's index block is read once, coalesced, into shared memory (as 32-bit row numbers b*N + i).
// xyz rows (12 bytes) are read through the LSU.
// ---------------------------------------------------------------------------------------------
constexpr int GR_MAX_WARPS = 16;        // warps per CTA are a launch parameter: as many as shared memory allows (the kernel is bound by
                                        // one warp's instruction latency, not by a pipe: ncu 12 % warps active, 25 % issue active at 8 warps)

template <int NST>
__global__ void __launch_bounds__(GR_MAX_WARPS * 32, 1) group_async_kernel(const float *__restrict__ xyz, const float *__restrict__ new_xyz,
                                                                       const char *__restrict__ feat, const int64_t *__restrict__ idx,
                                                                       int N, int S, int K, int D, int xyz_first, int ksplit,
                                                                       int units_total, float *__restrict__ out) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t row_bytes = (uint32_t)D * 4u;
    const uint32_t row_stride = row_bytes + (((D >> 2) & 1) ? 32u : 16u);     // (stride / 16) odd -> conflict-free 16-byte reads
    const uint32_t tile_bytes = 32u * row_stride;
    const int kper = (K + ksplit - 1) / ksplit;                       // slots per unit
    const uint32_t idx_stride = (uint32_t)(kper | 1) * 4u;            // odd number of words: column reads are conflict-free
    const uint32_t idx_bytes = (32u * idx_stride + 127u) & ~127u;
    const uint32_t warp_bytes = idx_bytes + NST * tile_bytes;
    const uint32_t ibuf = smem_u32(smem) + (uint32_t)warp * warp_bytes;
    const uint32_t data0 = ibuf + idx_bytes;
    const int nwarps = (int)(blockDim.x >> 5);
    const int gw = blockIdx.x * nwarps + warp, nw = gridDim.x * nwarps;
    const int s_tiles = (S + 31) / 32;
    const int C = D + 3, xoff = xyz_first ? 0 : D, foff = xyz_first ? 3 : 0, D4 = D >> 2;
    const size_t cstride = (size_t)K * S;
    // how the warp copies a tile: cpr 16-byte chunks per row; rpp rows per instruction when a row is < 512 bytes
    const int cpr = (int)(row_bytes >> 4);
    const int lanes_per_row = cpr >= 32 ? 32 : cpr;
    const int rpp = 32 / lanes_per_row;
    const int sub = lane / lanes_per_row, chunk = lane - sub * lanes_per_row;

    for (int unit = gw; unit < units_total; unit += nw) {
        const int bt = unit / ksplit, kpart = unit - bt * ksplit;
        const int b = bt / s_tiles, stile = bt - b * s_tiles;
        const int s0 = stile * 32, k0 = kpart * kper;
        const int nk = K - k0 < kper ? K - k0 : kper;
        const int s = s0 + lane;
        const bool live = s < S;
        // ---- the unit's index block idx[b, s0..s0+31, k0..k0+nk) -> shared as row numbers b*N + i (-1: none) ----
        __syncwarp();
        {
            // element e = sl * nk + kk of the block, 32 per pass (coalesced over (s, k)); all loads of the block are issued
            // before the first store so that they overlap (the block is the head of the unit's dependent chain)
            const int total = 32 * nk;
            for (int e0 = 0; e0 < total; e0 += 128) {
                long iv[4];
                int ee[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    ee[u] = e0 + 32 * u + lane;
                    const int sl = ee[u] / nk, kk = ee[u] - sl * nk;
                    iv[u] = (ee[u] < total && s0 + sl < S) ? idx[((size_t)b * S + s0 + sl) * K + k0 + kk] : (long)N;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (ee[u] >= total) continue;
                    const int sl = ee[u] / nk, kk = ee[u] - sl * nk;
                    long i = iv[u];
                    if (i < 0) i += N;
                    const int r = (i >= 0 && i < N) ? b * N + (int)i : -1;
                    B200PC_DEV_ASSERT(sl >= 0 && sl < 32 && kk >= 0 && kk < nk && r < (b + 1) * N);
                    asm volatile("st.shared.b32 [%0], %1;" ::"r"(ibuf + (uint32_t)sl * idx_stride + 4u * kk), "r"(r) : "memory");
                }
            }
        }
        __syncwarp();
        auto row_of = [&](int sl, int kk) -> int {
            int r;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(r) : "r"(ibuf + (uint32_t)sl * idx_stride + 4u * kk));
            return r;
        };
        auto issue = [&](int kk, int st) {                            // always commits one cp.async group (possibly empty)
            if (kk < nk) {
                const uint32_t tile = data0 + (uint32_t)st * tile_bytes;
                if (cpr >= 32) {
                    for (int sl = 0; sl < 32; ++sl) {
                        const int r = row_of(sl, kk);                 // broadcast read
                        if (r >= 0) warp_copy_row(tile + (uint32_t)sl * row_stride, feat + (size_t)r * row_bytes, row_bytes, lane);
                    }
                } else {
                    uint32_t dst = tile + (uint32_t)sub * row_stride + 16u * chunk;
                    for (int sl = sub; sl < 32; sl += rpp, dst += rpp * row_stride) {   // rpp rows per instruction
                        const int r = row_of(sl, kk);
                        if (r >= 0) cp_async16(dst, feat + (size_t)r * row_bytes + 16u * chunk);
                    }
                }
            }
            cp_async_commit();
        };
        float cx = 0.f, cy = 0.f, cz = 0.f;
        if (live) {
            const float *cr = new_xyz + ((size_t)b * S + s) * 3;
            cx = cr[0]; cy = cr[1]; cz = cr[2];
        }
#pragma unroll
        for (int p = 0; p < NST - 1; ++p) issue(p, p);
        int st = 0;
        B200PC_DEV_ASSERT(b >= 0 && stile < s_tiles && k0 >= 0 && k0 < K && nk >= 1 && k0 + nk <= K);
        float *o = out + ((size_t)b * C * K + k0) * S + s;
        for (int kk = 0; kk < nk; ++kk, o += S) {
            // the xyz row (12 bytes, through the LSU) is requested BEFORE the feature rows are issued: its latency hides behind
            // the copy loop instead of stalling the warp in front of it
            const int r = row_of(lane, kk);
            const bool ok = r >= 0;
            B200PC_DEV_ASSERT(r >= -1 && r < (b + 1) * N);
            float px = 0.0f, py = 0.0f, pz = 0.0f;
            if (live && ok) {
                const float *xr = xyz + (size_t)r * 3;
                px = __ldg(xr + 0); py = __ldg(xr + 1); pz = __ldg(xr + 2);
            }
            issue(kk + NST - 1, st == 0 ? NST - 1 : st - 1);         // into the stage consumed one iteration ago
            if (live) {
                __stcs(o + (size_t)(xoff + 0) * cstride, __fsub_rn(px, cx));
                __stcs(o + (size_t)(xoff + 1) * cstride, __fsub_rn(py, cy));
                __stcs(o + (size_t)(xoff + 2) * cstride, __fsub_rn(pz, cz));
            }
            cp_async_wait<NST - 1>();                                 // tile kk has landed (this lane's share)
            __syncwarp();                                             // ... every lane's share
            const uint32_t rowa = data0 + (uint32_t)st * tile_bytes + (uint32_t)lane * row_stride;
            float *of = o + (size_t)foff * cstride;
            if (live) {
#pragma unroll 4
                for (int q = 0; q < D4; ++q, of += 4 * cstride) {
                    const float4 v = ok ? lds_f4(rowa + 16u * q) : make_float4(0.f, 0.f, 0.f, 0.f);
                    __stcs(of, v.x); __stcs(of + cstride, v.y); __stcs(of + 2 * cstride, v.z); __stcs(of + 3 * cstride, v.w);
                }
            }
            __syncwarp();                                             // every lane is done reading the stage
            st = st + 1 == NST ? 0 : st + 1;
        }
        cp_async_wait<0>();                                           // drain the (empty) tail groups before the ring restarts
    }
}

// ---------------------------------------------------------------------------------------------
// launch plans
// ---------------------------------------------------------------------------------------------
template <typename F>
static int dispatch_nst12(int nst, F &&f) {
    if (nst >= 2) return f(std::integral_constant<int, 2>());
    return f(std::integral_constant<int, 1>());
}

// force == 0: only where measured faster than the register path (16 warps fit: D <= 64 -- 90.7 vs 102.7 us at C3, D = 64;
// with 10 warps at D = 128 it is 210 vs 183 us); force != 0: every shape the kernel can serve (A/B, tests).
int group_bulk(const float *xyz, const float *new_xyz, const float *feat, const int64_t *idx, int B, int N, int S, int K, int D,
               int xyz_first, float *out, int force, cudaStream_t st) {
    if (!force && (long)B * S * K < 32768) return -100;                  // small groupings: one wave of the register kernel is quicker
    if (D < 16 || D % 4 != 0 || D > 1024 || (reinterpret_cast<uintptr_t>(feat) & 15) || K > 256) return -100;
    const int cpr = D / 4;
    if (cpr < 32 && 32 % cpr != 0) return -100;                        // rows shorter than 512 bytes must tile an instruction evenly
    if ((long)B * N >= (1L << 31) || (long)B * ((S + 31) / 32) * K >= (1L << 31)) return -100;     // 32-bit row arithmetic in the kernel
    const int sms = sm_count();
    const uint32_t row_stride = (uint32_t)D * 4u + (((D >> 2) & 1) ? 32u : 16u);
    const size_t tile = (size_t)32 * row_stride;
    // Many warps with a shallow ring beat few warps with a deep one here (the warp's own dependent chain idx -> copy -> LDS ->
    // STG is the limiter): one stage per warp, as many warps as fit; two stages only when 16 warps still fit with them.
    int ksplit = 1, kper = K, nst = 1, nwarps = 0;
    long units = 0;
    for (int pass = 0; pass < 2; ++pass) {
        const long base_units = (long)B * ((S + 31) / 32);
        const long warps_guess = (long)sms * (nwarps > 0 ? nwarps : GR_MAX_WARPS);
        ksplit = 1;
        while (ksplit < K && base_units * ksplit < 6 * warps_guess) ksplit <<= 1;
        if (ksplit > K) ksplit = K;
        kper = (K + ksplit - 1) / ksplit;
        ksplit = (K + kper - 1) / kper;                                  // e.g. K = 10, 8 parts of 2 slots: only 5 hold any
        units = base_units * ksplit;
        const size_t idx_bytes = ((size_t)32 * (kper | 1) * 4 + 127) & ~(size_t)127;
        int w1 = (int)(RM_SMEM_BUDGET / (idx_bytes + tile)), w2 = (int)(RM_SMEM_BUDGET / (idx_bytes + 2 * tile));
        nst = w2 >= GR_MAX_WARPS ? 2 : 1;
        nwarps = nst == 2 ? w2 : w1;
        if (nwarps > GR_MAX_WARPS) nwarps = GR_MAX_WARPS;
        if (nwarps < 4 || (!force && nwarps < GR_MAX_WARPS)) return -100;
    }
    // the kernel re-derives kper from ksplit; every part it numbers must start inside [0, K)
    B200PC_REQUIRE((K + ksplit - 1) / ksplit == kper && (long)(ksplit - 1) * kper < K, "group_bulk: bad plan K=%d ksplit=%d kper=%d",
                   K, ksplit, kper);
    const size_t idx_bytes = ((size_t)32 * (kper | 1) * 4 + 127) & ~(size_t)127;
    const int grid = (int)((units + nwarps - 1) / nwarps < sms ? (units + nwarps - 1) / nwarps : sms);
    const size_t smem = (size_t)nwarps * (idx_bytes + nst * tile);
    return dispatch_nst12(nst, [&](auto tag) -> int {
        constexpr int NST = decltype(tag)::value;
        auto kern = group_async_kernel<NST>;
        B200PC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, nwarps * 32, smem, st>>>(xyz, new_xyz, reinterpret_cast<const char *>(feat), idx, N, S, K, D, xyz_first, ksplit,
                                              (int)units, out);
        B200PC_LAUNCH_CHECK();
        return B200PC_OK;
    });
}

}  // namespace b200pc
