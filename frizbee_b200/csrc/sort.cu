// sort.cu — stable descending-score sort of index-ordered matches.
//
// Reference replaced: radix_sort_matches (src/sort.rs:6-40): a stable 2-pass LSD radix sort on the
// u16 score of a list that is already in index order, giving (score desc, index asc).  Any stable
// sort by descending score yields the identical sequence; here it is a counting sort whose digit is
// the whole score when the score bound allows it (one pass), else the reference's two 8-bit passes.
//
//   k_sort_hist     each "virtual warp" owns a contiguous segment and counts its digits in smem
//   k_sort_scan_rows per-digit exclusive prefix over the segments; its last block adds the descending exclusive prefix
//                   over the digits (digit_base)
//   k_sort_scatter  each virtual warp re-walks its segment IN ORDER, 32 elements at a time;
//                   __match_any_sync gives the in-warp stable rank, a per-warp counter array the rest
//
// The element count lives in device memory (it is produced by the previous stage), so the whole
// match_list pipeline runs without a host round trip until the final copy-out.
#include "frz_device.cuh"
#include "frz_host.h"

namespace {

constexpr int kSortBlocks = 288;              // ~2 blocks per SM
constexpr int kSortWarps = 8;
constexpr int kV = kSortBlocks * kSortWarps;  // 2304 virtual warps = segments: the in-order walk of a segment is latency-bound, so
                                              // more, shorter segments are faster (1024 segments: 22 us scatter at 750 k matches)
static_assert(kV % 128 == 0, "k_sort_scan_rows reads a digit row as 32 lanes x uint4");
constexpr int kMaxBins = 1024;

__device__ __forceinline__ void segment_of(unsigned long long n, int v, unsigned long long* lo, unsigned long long* hi) {
    unsigned long long seg = (n + kV - 1) / kV;
    seg = (seg + 31) & ~31ull;
    unsigned long long a = seg * v;
    *lo = a < n ? a : n;
    unsigned long long b = a + seg;
    *hi = b < n ? b : n;
}

__device__ __forceinline__ uint32_t digit_of(const FrzMatchDev& m, int shift, uint32_t mask) {
    return ((uint32_t)m.score >> shift) & mask;
}

__global__ void __launch_bounds__(kSortWarps * 32) k_sort_hist(const FrzMatchDev* __restrict__ in,
                                                               const unsigned long long* __restrict__ n_ptr, int shift,
                                                               int bins, uint32_t* __restrict__ hist) {
    extern __shared__ uint32_t sm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* cnt = sm + warp * bins;
    for (int d = lane; d < bins; d += 32) cnt[d] = 0;
    __syncwarp();
    const int v = blockIdx.x * kSortWarps + warp;
    unsigned long long lo, hi;
    segment_of(*n_ptr, v, &lo, &hi);
    const uint32_t mask = (uint32_t)bins - 1;
    // four loads in flight per lane: the walk is latency-bound (one 256-byte line per trip)
    unsigned long long i = lo + lane;
    for (; i + 96 < hi; i += 128) {
        const FrzMatchDev a = in[i], b = in[i + 32], c = in[i + 64], d = in[i + 96];
        atomicAdd(&cnt[digit_of(a, shift, mask)], 1u);
        atomicAdd(&cnt[digit_of(b, shift, mask)], 1u);
        atomicAdd(&cnt[digit_of(c, shift, mask)], 1u);
        atomicAdd(&cnt[digit_of(d, shift, mask)], 1u);
    }
    for (; i < hi; i += 32) atomicAdd(&cnt[digit_of(in[i], shift, mask)], 1u);
    __syncwarp();
    for (int d = lane; d < bins; d += 32) hist[(size_t)d * kV + v] = cnt[d];
}

// hist[d][v] → exclusive prefix over v (in place), one warp per digit row; totals[d] = row sum.  The LAST block to
// finish (device counter, self-resetting) then turns the row totals into digit_base[d] = #elements with digit > d
// (descending exclusive prefix over the digits) — one launch instead of two.
__global__ void __launch_bounds__(256) k_sort_scan_rows(uint32_t* __restrict__ hist, int bins, uint32_t* __restrict__ totals,
                                                        uint32_t* __restrict__ digit_base, unsigned int* __restrict__ done_counter) {
    __shared__ bool is_last;
    __shared__ uint32_t wsum[8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int d = blockIdx.x * 8 + warp;
    if (d < bins) {
        constexpr int PER = kV / 32;  // contiguous entries per lane
        uint4* row = reinterpret_cast<uint4*>(hist + (size_t)d * kV + lane * PER);
        uint4 v[PER / 4];
        uint32_t s = 0;
#pragma unroll
        for (int k = 0; k < PER / 4; k++) { v[k] = row[k]; s += v[k].x + v[k].y + v[k].z + v[k].w; }
        uint32_t x = s;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        uint32_t run = x - s;
#pragma unroll
        for (int k = 0; k < PER / 4; k++) {
            uint4 o4;
            o4.x = run; run += v[k].x;
            o4.y = run; run += v[k].y;
            o4.z = run; run += v[k].z;
            o4.w = run; run += v[k].w;
            row[k] = o4;
        }
        if (lane == 31) totals[d] = x;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(done_counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // digit_base over bins <= 1024 entries: thread t owns the PERT digits t*PERT .. of the DESCENDING sequence
    const int PERT = (bins + 255) / 256;
    uint32_t loc[4] = {0, 0, 0, 0}, sum = 0;
    for (int k = 0; k < PERT; k++) {
        const int t = threadIdx.x * PERT + k;
        loc[k] = t < bins ? __ldcg(&totals[bins - 1 - t]) : 0u;
        sum += loc[k];
    }
    uint32_t x = sum;
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < 8 ? wsum[lane] : 0u, xs = w;
        for (int o = 1; o < 8; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, xs, o);
            if (lane >= o) xs += y;
        }
        if (lane < 8) wsum[lane] = xs - w;
    }
    __syncthreads();
    uint32_t run = wsum[warp] + x - sum;
    for (int k = 0; k < PERT; k++) {
        const int t = threadIdx.x * PERT + k;
        if (t < bins) digit_base[bins - 1 - t] = run;
        run += loc[k];
    }
    if (threadIdx.x == 0) *done_counter = 0;   // ready for the next pass
}

__global__ void __launch_bounds__(kSortWarps * 32) k_sort_scatter(const FrzMatchDev* __restrict__ in, FrzMatchDev* __restrict__ out,
                                                                  const unsigned long long* __restrict__ n_ptr, int shift, int bins,
                                                                  const uint32_t* __restrict__ hist,
                                                                  const uint32_t* __restrict__ digit_base) {
    extern __shared__ uint32_t sm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* cnt = sm + warp * bins;
    const int v = blockIdx.x * kSortWarps + warp;
    for (int d = lane; d < bins; d += 32) cnt[d] = digit_base[d] + hist[(size_t)d * kV + v];
    __syncwarp();
    unsigned long long lo, hi;
    segment_of(*n_ptr, v, &lo, &hi);
    const uint32_t mask = (uint32_t)bins - 1;
    // the element of the NEXT trip is loaded before this trip's rank / counter chain (software pipelining: the walk has
    // to stay in order for stability, so the only parallelism inside a segment is load-ahead)
    FrzMatchDev nxt;
    nxt.index = 0; nxt.score = 0; nxt.exact = 0; nxt.pad = 0;
    if (lo + lane < hi) nxt = in[lo + lane];
    for (unsigned long long base = lo; base < hi; base += 32) {
        const unsigned long long i = base + lane;
        const bool valid = i < hi;
        const FrzMatchDev m = nxt;
        if (i + 32 < hi) nxt = in[i + 32];
        uint32_t d = (uint32_t)bins + lane;  // sentinel: matches nobody
        if (valid) d = digit_of(m, shift, mask);
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const uint32_t rank = __popc(peers & ((1u << lane) - 1));
        uint32_t pos = 0;
        if (valid) pos = cnt[d] + rank;
        __syncwarp();
        if (valid && rank == 0) cnt[d] += __popc(peers);
        __syncwarp();
        if (valid) out[pos] = m;
    }
}

}  // namespace

// n_ptr: device pointer to the element count.  score_bound: host-known upper bound of any score.
frz_status frz_launch_sort_by_score_dev(const FrzMatchDev* d_in, FrzMatchDev* d_tmp, FrzMatchDev* d_out,
                                        const unsigned long long* n_ptr, uint32_t score_bound, FrzWorkspace& ws,
                                        cudaStream_t stream, FrzLaunchStats* st) {
    auto pass = [&](const FrzMatchDev* src, FrzMatchDev* dst, int shift, int bins) -> frz_status {
        const size_t smem = (size_t)kSortWarps * bins * sizeof(uint32_t);
        k_sort_hist<<<kSortBlocks, kSortWarps * 32, smem, stream>>>(src, n_ptr, shift, bins, ws.sort_hist);
        uint32_t* totals = ws.sort_hist + (size_t)kMaxBins * kV;
        uint32_t* digit_base = totals + kMaxBins;
        unsigned int* done_counter = reinterpret_cast<unsigned int*>(digit_base + kMaxBins);   // zeroed at allocation, self-resetting
        k_sort_scan_rows<<<(bins + 7) / 8, 256, 0, stream>>>(ws.sort_hist, bins, totals, digit_base, done_counter);
        if (ws.arm_table_ev && ws.table_ev) {   // digit_base is final: the multi-GPU layer publishes it while the scatter runs
            FRZ_CUDA_TRY(cudaEventRecord(ws.table_ev, stream));
            ws.table_ev_recorded = true;
        }
        k_sort_scatter<<<kSortBlocks, kSortWarps * 32, smem, stream>>>(src, dst, n_ptr, shift, bins, ws.sort_hist, digit_base);
        FRZ_CUDA_TRY(cudaGetLastError());
        if (st) st->launches += 3;
        return FRZ_OK;
    };
    if (score_bound < 256) return pass(d_in, d_out, 0, 256);
    if (score_bound < 512) return pass(d_in, d_out, 0, 512);
    if (score_bound < 1024) return pass(d_in, d_out, 0, 1024);
    // the reference's two 8-bit LSD passes (src/sort.rs:8-39)
    FRZ_TRY(pass(d_in, d_tmp, 0, 256));
    return pass(d_tmp, d_out, 8, 256);
}

size_t frz_sort_hist_words() { return (size_t)kMaxBins * kV + 2 * kMaxBins + 4; }   // + the pass-completion counter (must start at zero)
// allocates the sort scratch on the current device (the completion counter of k_sort_scan_rows starts at zero)
frz_status frz_sort_hist_alloc(uint32_t** out) {
    FRZ_CUDA_TRY(cudaMalloc(out, frz_sort_hist_words() * sizeof(uint32_t)));
    FRZ_CUDA_TRY(cudaMemset(*out + (size_t)kMaxBins * kV + 2 * kMaxBins, 0, 4 * sizeof(uint32_t)));
    return FRZ_OK;
}

// digit_base[d] of the LAST pass run on this workspace = number of elements whose digit is greater than d.  After a
// single-pass sort (score bound < 1024) that is, per score s, how many matches of the run score higher than s — the table
// the multi-GPU P2P placement needs (parallel.cu) — so nobody has to binary-search the sorted run for it.
const uint32_t* frz_sort_digit_base(const FrzWorkspace& ws) { return ws.sort_hist ? ws.sort_hist + (size_t)kMaxBins * kV + kMaxBins : nullptr; }
int frz_sort_single_pass_bins(uint32_t score_bound) { return score_bound < 256 ? 256 : score_bound < 512 ? 512 : score_bound < 1024 ? 1024 : 0; }
