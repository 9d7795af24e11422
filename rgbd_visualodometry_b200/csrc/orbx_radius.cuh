// orbx_radius.cuh -- radiusMatch's offsets scan and list ordering (BFMatcher(NORM_HAMMING).radiusMatch, cv2's exact order).
//
// The matcher's count pass writes every list's length to offsets[1 + L]; k_radius_tile_sums / k_radius_scan_sums /
// k_radius_scan_tiles turn them into the 64-bit CSR offsets in place.  The emit pass then writes list L's hits to
// out[offsets[L] .. offsets[L + 1]) in ascending trainIdx: the sequence cv::BFMatcher::radiusMatchImpl hands to std::sort.
// k_radius_order reorders each list the way libstdc++'s std::sort does with DMatch::operator< (distance only), which is
// NOT a sort by (distance, trainIdx):
//   __introsort_loop (depth limit 2 floor(log2 n), threshold 16): __move_median_to_first(first, first + 1, mid, last - 1),
//   Hoare __unguarded_partition on the distance, heap sort (__partial_sort(first, last, last)) of a segment whose depth
//   budget ran out; then __final_insertion_sort.  That insertion sort is stable and every segment the loop leaves is
//   bounded by its neighbours, so the result is each segment's stable sort by distance: segments of <= 16 entries are
//   insertion-sorted one per lane, heap-sorted segments are already in order.
// One warp per list.  The partition runs on all 32 lanes with ballots: scanning from the left, the k-th "left stopper"
// (distance >= pivot) swaps with the k-th "right stopper" (distance <= pivot, scanning from the right) while they have not
// crossed; at the first crossing pair k the cut is min(left stopper k, right stopper k - 1), exactly the position the
// sequential loop returns.  A list of at most RS_SMEM_KEYS entries is sorted in shared memory as 32-bit keys
// distance << 20 | trainIdx; a longer one in place in its own slot of the output buffer (the keys take its first quarter).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace orbx {

constexpr int RS_SCAN_NT = 1024;                 // threads of the scan kernels
constexpr int RS_SCAN_TILE = 4 * RS_SCAN_NT;     // counts per block of k_radius_tile_sums / k_radius_scan_tiles
constexpr int RS_WARPS = 8;                      // lists (warps) per block of k_radius_order
constexpr int RS_SMEM_KEYS = 1024;               // keys per warp in shared memory; longer lists are sorted in global memory
constexpr int RS_THRESHOLD = 16;                 // libstdc++ _S_threshold
constexpr int RS_STACK = 48;                     // pending segments: at most the depth limit 2 floor(log2 n) <= 38, plus one
constexpr int RS_KEY_SHIFT = 20;                 // key = distance << 20 | trainIdx (train sets hold < 2^20 rows)

// ---- 64-bit inclusive scan of counts[0 .. n) in place: tile sums, one-block scan of the sums, tile scans -------------------
__device__ __forceinline__ long long rs_block_excl_scan(long long x, long long* s_warp, long long* total)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    long long inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += y;
    }
    if (lane == 31) s_warp[w] = inc;
    __syncthreads();
    if (w == 0) {
        long long t = lane < RS_SCAN_NT / 32 ? s_warp[lane] : 0, ti = t;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, ti, d);
            if (lane >= d) ti += y;
        }
        s_warp[lane] = ti - t;
        if (lane == 31) *total = ti;
    }
    __syncthreads();
    const long long r = s_warp[w] + inc - x;
    __syncthreads();                                          // s_warp is reused by the caller's next scan
    return r;
}

__global__ void __launch_bounds__(RS_SCAN_NT) k_radius_tile_sums(const long long* __restrict__ v, long long n, long long* __restrict__ sums)
{
    __shared__ long long s_warp[32], s_total;
    const long long i0 = (long long)blockIdx.x * RS_SCAN_TILE + threadIdx.x * 4;
    long long x = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) if (i0 + k < n) x += v[i0 + k];
    rs_block_excl_scan(x, s_warp, &s_total);
    if (threadIdx.x == 0) sums[blockIdx.x] = s_total;
}

// one block: exclusive scan of the nb tile sums in place
__global__ void __launch_bounds__(RS_SCAN_NT) k_radius_scan_sums(long long* __restrict__ sums, long long nb)
{
    __shared__ long long s_warp[32], s_total;
    long long carry = 0;
    for (long long b = 0; b < nb; b += RS_SCAN_NT) {
        const long long i = b + threadIdx.x;
        const long long x = i < nb ? sums[i] : 0;
        const long long e = rs_block_excl_scan(x, s_warp, &s_total);
        if (i < nb) sums[i] = carry + e;
        carry += s_total;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(RS_SCAN_NT) k_radius_scan_tiles(long long* __restrict__ v, long long n, const long long* __restrict__ sums)
{
    __shared__ long long s_warp[32], s_total;
    const long long i0 = (long long)blockIdx.x * RS_SCAN_TILE + threadIdx.x * 4;
    long long x[4], t = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) { x[k] = i0 + k < n ? v[i0 + k] : 0; t += x[k]; }
    long long run = sums[blockIdx.x] + rs_block_excl_scan(t, s_warp, &s_total);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        run += x[k];
        if (i0 + k < n) v[i0 + k] = run;
    }
}

// ---- list ordering ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t rs_dist(uint32_t key) { return key >> RS_KEY_SHIFT; }

// position of the i-th (0-based) set bit of mask; i < popc(mask)
__device__ __forceinline__ int rs_nth_bit(uint32_t mask, int i)
{
    int pos = 0;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const int c = __popc(mask & ((1u << s) - 1u));
        if (c <= i) { pos += s; mask >>= s; i -= c; }
    }
    return pos;
}

// std::__adjust_heap (with __push_heap) on v[0 .. len), comp(a, b) = distance(a) < distance(b)
__device__ void rs_adjust_heap(uint32_t* v, int hole, int len, uint32_t value)
{
    const int top = hole;
    int child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (rs_dist(v[child]) < rs_dist(v[child - 1])) --child;
        v[hole] = v[child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        v[hole] = v[child - 1];
        hole = child - 1;
    }
    int parent = (hole - 1) / 2;
    while (hole > top && rs_dist(v[parent]) < rs_dist(value)) {
        v[hole] = v[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    v[hole] = value;
}

// std::__partial_sort(first, last, last): __make_heap, then __sort_heap
__device__ void rs_heap_sort(uint32_t* v, int n)
{
    if (n < 2) return;
    for (int parent = (n - 2) / 2;; --parent) {
        rs_adjust_heap(v, parent, n, v[parent]);
        if (parent == 0) break;
    }
    for (int last = n - 1; last > 0; --last) {
        const uint32_t value = v[last];
        v[last] = v[0];
        rs_adjust_heap(v, 0, last, value);
    }
}

// std::__insertion_sort on v[first, last) (stable: an entry moves left past strictly larger distances only)
__device__ void rs_insertion_sort(uint32_t* v, int first, int last)
{
    for (int i = first + 1; i < last; ++i) {
        const uint32_t x = v[i];
        int j = i - 1;
        while (j >= first && rs_dist(x) < rs_dist(v[j])) { v[j + 1] = v[j]; --j; }
        v[j + 1] = x;
    }
}

// std::__unguarded_partition_pivot on v[first, last) by the whole warp; returns the cut
__device__ int rs_partition_warp(uint32_t* v, int first, int last)
{
    const int lane = threadIdx.x & 31;
    if (lane == 0) {                                          // __move_median_to_first(first, first + 1, mid, last - 1)
        const int a = first + 1, b = first + (last - first) / 2, c = last - 1;
        const uint32_t da = rs_dist(v[a]), db = rs_dist(v[b]), dc = rs_dist(v[c]);
        int s;
        if (da < db) s = db < dc ? b : da < dc ? c : a;
        else         s = da < dc ? a : db < dc ? c : b;
        const uint32_t t = v[first];
        v[first] = v[s];
        v[s] = t;
    }
    __syncwarp();
    const uint32_t p = rs_dist(v[first]);
    int fl = first + 1, fr = last - 1;                        // next left chunk [fl, fl + 32), right chunk (fr - 32, fr]
    uint32_t ml = 0, mr = 0;                                  // pending stoppers of the current chunks (bit i: fl0 + i / fr0 - i)
    int bl = 0, br = 0, prev_r = last;                        // chunk bases; the last right stopper already swapped
    while (true) {
        while (ml == 0) {                                     // (positions past the segment stop the scan: never reached
            const int i = fl + lane;                          //  before a crossing, whose cut they cannot change)
            ml = __ballot_sync(0xffffffffu, i >= last || rs_dist(v[i]) >= p);
            bl = fl;
            fl += 32;
        }
        while (mr == 0) {
            const int i = fr - lane;
            mr = __ballot_sync(0xffffffffu, i <= first || rs_dist(v[i]) <= p);
            br = fr;
            fr -= 32;
        }
        const int m = min(__popc(ml), __popc(mr));
        int l = 0, r = 0;
        if (lane < m) { l = bl + rs_nth_bit(ml, lane); r = br - rs_nth_bit(mr, lane); }
        const uint32_t crossed = __ballot_sync(0xffffffffu, lane < m && l >= r);
        const int c = crossed ? __ffs(crossed) - 1 : m;       // pairs before the first crossing swap
        uint32_t x = 0, y = 0;
        if (lane < c) { x = v[l]; y = v[r]; }
        __syncwarp();
        if (lane < c) { v[l] = y; v[r] = x; }
        __syncwarp();
        const int lc = __shfl_sync(0xffffffffu, l, c & 31);
        const int rp = __shfl_sync(0xffffffffu, r, (c + 31) & 31);
        if (crossed) return min(lc, c > 0 ? rp : prev_r);
        prev_r = rp;                                          // (c == m >= 1 here)
        const int pl = rs_nth_bit(ml, m - 1), pr = rs_nth_bit(mr, m - 1);   // drop the m paired stoppers
        ml = pl == 31 ? 0u : ml & (0xffffffffu << (pl + 1));
        mr = pr == 31 ? 0u : mr & (0xffffffffu << (pr + 1));
    }
}

// libstdc++ std::sort of v[0, n) by distance, by one warp.  stack / small: this warp's shared scratch.
__device__ void rs_sort_warp(uint32_t* v, int n, int* stack, int* small)
{
    const int lane = threadIdx.x & 31;
    int sp = 0, nsmall = 0;
    int first = 0, last = n, depth = 2 * (31 - __clz(n));
    auto flush = [&]() {                                      // insertion-sort the recorded short segments, one per lane
        __syncwarp();
        if (lane < nsmall) rs_insertion_sort(v, small[2 * lane], small[2 * lane + 1]);
        __syncwarp();
        nsmall = 0;
    };
    while (true) {
        if (last - first > RS_THRESHOLD && depth > 0) {
            --depth;
            const int cut = rs_partition_warp(v, first, last);
            if (lane == 0) { stack[3 * sp] = cut; stack[3 * sp + 1] = last; stack[3 * sp + 2] = depth; }
            ++sp;
            last = cut;
            continue;
        }
        if (last - first > RS_THRESHOLD) {                    // depth limit reached: heap sort, already in final order
            if (lane == 0) rs_heap_sort(v + first, last - first);
            __syncwarp();
        } else {
            if (lane == 0) { small[2 * nsmall] = first; small[2 * nsmall + 1] = last; }
            if (++nsmall == 32) flush();
        }
        if (sp == 0) break;
        __syncwarp();
        --sp;
        first = stack[3 * sp]; last = stack[3 * sp + 1]; depth = stack[3 * sp + 2];
        __syncwarp();
    }
    flush();
}

// One warp per list L < nlists (query L % nq): list records out[offsets[L] .. offsets[L + 1]) in ascending trainIdx ->
// std::sort's order.  Lists ending past cap were not written and are skipped.
__global__ void __launch_bounds__(RS_WARPS * 32) k_radius_order(int4* __restrict__ out, const long long* __restrict__ offsets, long long nlists,
                                                                int nq, long long cap)
{
    __shared__ uint32_t s_keys[RS_WARPS][RS_SMEM_KEYS];
    __shared__ int s_stack[RS_WARPS][3 * RS_STACK];
    __shared__ int s_small[RS_WARPS][64];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long L = (long long)blockIdx.x * RS_WARPS + w;
    if (L >= nlists) return;
    const long long o0 = offsets[L], o1 = offsets[L + 1];
    if (o1 > cap || o1 - o0 < 2) return;
    const int n = (int)(o1 - o0), q = (int)(L % nq);
    int4* rec = out + o0;
    uint32_t* v = n <= RS_SMEM_KEYS ? s_keys[w] : reinterpret_cast<uint32_t*>(rec);
    // records -> keys.  In place (a long list), key i lands in record i / 4, which this or an earlier chunk has read.
    for (int b = 0; b < n; b += 32) {
        const int i = b + lane;
        uint32_t k = 0;
        if (i < n) {
            const int4 r = rec[i];
            k = ((uint32_t)__int_as_float(r.w) << RS_KEY_SHIFT) | (uint32_t)r.y;
        }
        __syncwarp();
        if (i < n) v[i] = k;
    }
    __syncwarp();
    rs_sort_warp(v, n, s_stack[w], s_small[w]);
    __syncwarp();
    // keys -> records from the top: record i covers keys 4i .. 4i + 3, which this or a later chunk has read
    for (int b = (n - 1) & ~31; b >= 0; b -= 32) {
        const int i = b + lane;
        const uint32_t k = i < n ? v[i] : 0u;
        __syncwarp();
        if (i < n) rec[i] = make_int4(q, (int)(k & ((1u << RS_KEY_SHIFT) - 1u)), 0, __float_as_int((float)rs_dist(k)));
    }
}

}  // namespace orbx
