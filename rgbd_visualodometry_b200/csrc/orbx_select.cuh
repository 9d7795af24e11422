// orbx_select.cuh -- A.4 - A.6 of cv::ORB::detectAndCompute (src/frontend.cpp:153): border-filtered FAST survivors ->
// KeyPointsFilter::retainBest(2 n_l) on the FAST score -> Harris response -> retainBest(n_l) on Harris, in libstdc++'s order.
//
// Two kernel families, identical results, both gathering the per-row FAST lists in raster order with gather_rows:
//   k_select         one CTA of SEL_NT threads per (frame, level), all three steps (frames with long candidate lists)
//   the warp trio, so that the inherently sequential part is as short as it can be and the rest is wide:
//   k_select_fast    one WARP per (frame, level): gathers the per-row FAST lists in raster order and runs retainBest(2 n_l)
//   k_harris         one THREAD per surviving candidate of the whole batch: the 7x7 Harris response (A.5)
//   k_select_harris  one WARP per (frame, level): retainBest(n_l) on the Harris response; the final list is left as the prefix of
//                    the level's workspace, its length in fincnt
// retainBest = std::nth_element + std::partition; its output ORDER is whatever libstdc++'s __introselect (median-of-3 to first,
// Hoare __unguarded_partition, insertion sort of <= 3, __heap_select once the depth budget is spent) and the bidirectional
// std::partition leave behind, and OpenCV's keypoint order -- and through index tie-breaks the matcher -- depends on it.  In the
// warp kernels a warp owns a problem: no block barrier, elements interleaved over the lanes (conflict-free shared / coalesced
// global access).
//   long ranges: one warp-parallel Hoare pass (SURVEY A.6 / probe E21): with L = ascending positions of !(a > piv) and R = descending
//     positions of !(piv > a) (original contents), the sequential loop swaps a[L[k]] <-> a[R[k]] for k < K, K = #{k : L[k] < R[k]}, and
//     returns cut = min(L[K], R[K-1]).  Ranks come from ballots and popcounts, K from a monotone scan, swaps run 32 at a time.
//   short ranges and the std::partition tail: the warp-cooperative sequential emulation below, shared with k_select.
// The working array lives in shared memory when the problem fits, else in the level's global workspace (same code).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "orbx_geom.h"
#include "orbx_device.cuh"

namespace orbx {

// Loads the compiler may not sink next to their first use: issued back to back, they are all in flight together.
__device__ __forceinline__ uint32_t ldg_u32_now(const void* p) { uint32_t v; asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p)); return v; }

// ------------------------------------------------------------------------------------------------ A.6 retainBest
// Exact emulation of KeyPointsFilter::retainBest = libstdc++ std::nth_element (__introselect: median-of-3 to
// first, Hoare __unguarded_partition, insertion sort of <= 3) + bidirectional std::partition.  The resulting ORDER
// is libstdc++'s, which OpenCV's output order (and, through index tie-breaks, the matcher) depends on.
//   - ranges longer than SEL_PAR_MIN: one whole-CTA data-parallel Hoare pass (SURVEY A.6 / probe E21): with
//     L = ascending positions of !(a > piv) and R = descending positions of !(piv > a) (original contents), the
//     sequential loop swaps a[L[k]] <-> a[R[k]] for k < K, K = #{k : L[k] < R[k]}, and returns
//     cut = min(L[K], R[K-1]).  Ranks come from a block scan, K from a block reduction, swaps run in parallel.
//   - short ranges and the std::partition tail: warp-cooperative sequential emulation, scans vectorised with ballots.
// `v` may live in shared or global memory.
__device__ __forceinline__ void elem_swap(Elem* v, int a, int b) { const Elem t = v[a]; v[a] = v[b]; v[b] = t; }

// first i in [start, end) with stopper(v[i]); `end` if none.  MODE 0: !(r > piv)   1: !(r >= piv)
template <int MODE>
__device__ __forceinline__ int scan_up(const Elem* v, int start, int end, float piv, int lane)
{
    for (int base = start; base < end; base += 32) {
        const int i = base + lane;
        bool p = false;
        if (i < end) { const float r = v[i].response; p = MODE == 0 ? !(r > piv) : !(r >= piv); }
        const unsigned b = __ballot_sync(0xffffffffu, p);
        if (b) return base + __ffs(b) - 1;
    }
    return end;
}
// last i in (stop, start] with stopper(v[i]); `stop` if none.  MODE 0: !(piv > r)   1: (r >= piv)
template <int MODE>
__device__ __forceinline__ int scan_down(const Elem* v, int start, int stop, float piv, int lane)
{
    for (int base = start; base > stop; base -= 32) {
        const int i = base - lane;
        bool p = false;
        if (i > stop) { const float r = v[i].response; p = MODE == 0 ? !(piv > r) : (r >= piv); }
        const unsigned b = __ballot_sync(0xffffffffu, p);
        if (b) return base - (__ffs(b) - 1);
    }
    return stop;
}

__device__ __forceinline__ int median3_pick(const Elem* v, int a, int b, int c)
{
    const float ra = v[a].response, rb = v[b].response, rc = v[c].response;
    if (ra > rb) return (rb > rc) ? b : ((ra > rc) ? c : a);
    return (ra > rc) ? a : ((rb > rc) ? c : b);
}

// libstdc++'s depth-limit fallback of __introselect (bits/stl_heap.h, comp(a, b) = a.response > b.response):
// __heap_select(first, nth + 1, last) = __make_heap on [first, middle), then every later element that beats the heap's
// top (the smallest kept response) is __pop_heap'ed in; finally iter_swap(first, nth).  Sequential by nature and rare
// (about one frame in a hundred hits the depth limit on some level): one lane runs it verbatim.
__device__ __forceinline__ void heap_push(Elem* b, int hole, int top, Elem value)
{
    int parent = (hole - 1) / 2;
    while (hole > top && b[parent].response > value.response) {
        b[hole] = b[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    b[hole] = value;
}
__device__ __forceinline__ void heap_adjust(Elem* b, int hole, int len, Elem value)
{
    const int top = hole;
    int child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (b[child].response > b[child - 1].response) --child;
        b[hole] = b[child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        b[hole] = b[child - 1];
        hole = child - 1;
    }
    heap_push(b, hole, top, value);
}
__device__ void heap_select_fallback(Elem* v, int first, int nth, int last, int lane)
{
    __syncwarp();
    if (lane == 0) {
        Elem* b = v + first;
        const int middle = nth + 1, len = middle - first;
        if (len >= 2) {
            int parent = (len - 2) / 2;
            for (;;) {
                const Elem value = b[parent];
                heap_adjust(b, parent, len, value);
                if (parent == 0) break;
                --parent;
            }
        }
        for (int i = middle; i < last; ++i)
            if (v[i].response > b[0].response) {
                const Elem value = v[i];
                v[i] = b[0];
                heap_adjust(b, 0, len, value);
            }
        elem_swap(v, first, nth);
    }
    __syncwarp();
}

// warp-cooperative __introselect on [first, last) with the remaining depth budget (heap-select fallback included)
__device__ void introselect_warp(Elem* v, int first, int last, int nth, int depth, int lane)
{
    while (last - first > 3) {
        if (depth == 0) { heap_select_fallback(v, first, nth, last, lane); return; }
        --depth;
        const int pick = median3_pick(v, first + 1, first + (last - first) / 2, last - 1);
        __syncwarp();
        if (lane == 0) elem_swap(v, first, pick);
        __syncwarp();
        const float piv = v[first].response;
        int f = first + 1, l = last;
        for (;;) {
            f = scan_up<0>(v, f, last, piv, lane);
            --l;
            l = scan_down<0>(v, l, first, piv, lane);
            if (!(f < l)) break;
            if (lane == 0) elem_swap(v, f, l);
            __syncwarp();
            ++f;
        }
        if (f <= nth) first = f; else last = f;
    }
    __syncwarp();
    if (lane == 0) {                                         // __insertion_sort, descending, <= 3 elements
        for (int i = first + 1; i < last; ++i) {
            const Elem val = v[i];
            int j = i;
            while (j > first && val.response > v[j - 1].response) { v[j] = v[j - 1]; --j; }
            v[j] = val;
        }
    }
    __syncwarp();
}

// warp-cooperative bidirectional std::partition(v + m, v + len, response >= thr); returns the partition point
__device__ int partition_tail_warp(Elem* v, int m, int len, float thr, int lane)
{
    int f = m, l = len;
    for (;;) {
        f = scan_up<1>(v, f, l, thr, lane);                  // first !pred in [f, l)
        if (f == l) return f;
        --l;
        l = scan_down<1>(v, l, f, thr, lane);                // last pred in (f, l]; f if none
        if (f == l) return f;
        if (lane == 0) elem_swap(v, f, l);
        __syncwarp();
        ++f;
    }
}

constexpr int SEL_NT = 512;             // threads per CTA of k_select: level 0 holds tens of thousands of candidates above 0.6 Mpixel
constexpr int SEL_SMEM_ELEMS = 2048;    // candidates of one level held in shared memory (more: the global workspace)
constexpr int SEL_PAR_MIN = 32;         // ranges up to this length are finished by one warp

struct SelShared {
    int warp_a[SEL_NT / 32], warp_b[SEL_NT / 32];   // one slot per warp
    int n;
};

// Whole-CTA KeyPointsFilter::retainBest(v, m).  All SEL_NT threads must call it.  PosT scratch lists Lp / Rp hold
// `len` positions each.  Returns the new length (valid on every thread).
template <typename PosT>
__device__ int retain_best_block(Elem* v, int len, int m, PosT* Lp, PosT* Rp, SelShared* sh)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (m < 0 || len <= m) return len;
    if (m == 0) return 0;
    const int nth = m - 1;
    int first = 0, last = len, depth = 2 * (31 - __clz(len));
    bool fallback = false;
    // ---- data-parallel Hoare passes while the range is long
    while (last - first > SEL_PAR_MIN) {
        if (depth == 0) { fallback = true; break; }          // depth budget spent: libstdc++ switches to __heap_select
        --depth;
        if (tid == 0) elem_swap(v, first, median3_pick(v, first + 1, first + (last - first) / 2, last - 1));
        __syncthreads();
        const float piv = v[first].response;
        const int lo = first + 1, n = last - lo;
        const int cs = (n + SEL_NT - 1) / SEL_NT;
        const int b = min(lo + tid * cs, last), e = min(b + cs, last);
        int cL = 0, cR = 0;
        for (int i = b; i < e; ++i) { const float r = v[i].response; cL += !(r > piv); cR += !(piv > r); }
        int iL = cL, iR = cR;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int oL = __shfl_up_sync(0xffffffffu, iL, d), oR = __shfl_up_sync(0xffffffffu, iR, d);
            if (lane >= d) { iL += oL; iR += oR; }
        }
        if (lane == 31) { sh->warp_a[wid] = iL; sh->warp_b[wid] = iR; }
        __syncthreads();
        int totL = 0, totR = 0, exL = iL - cL, exR = iR - cR;
#pragma unroll
        for (int i = 0; i < SEL_NT / 32; ++i) {
            const int a = sh->warp_a[i], c = sh->warp_b[i];
            if (i < wid) { exL += a; exR += c; }
            totL += a; totR += c;
        }
        {
            int kL = exL, kR = totR - 1 - exR;               // L: ascending rank;  R: rank counted from the right end
            for (int i = b; i < e; ++i) {
                const float r = v[i].response;
                if (!(r > piv)) Lp[kL++] = (PosT)i;
                if (!(piv > r)) Rp[kR--] = (PosT)i;
            }
        }
        __syncthreads();
        const int mm = min(totL, totR);
        int cnt = 0;
        for (int k = tid; k < mm; k += SEL_NT) cnt += ((int)Lp[k] < (int)Rp[k]);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
        if (lane == 0) sh->warp_a[wid] = cnt;                // safe: all reads of warp_a finished before the last barrier
        __syncthreads();
        int K = 0;
#pragma unroll
        for (int i = 0; i < SEL_NT / 32; ++i) K += sh->warp_a[i];
        for (int k = tid; k < K; k += SEL_NT) elem_swap(v, (int)Lp[k], (int)Rp[k]);
        int cut = 0x7fffffff;
        if (K < totL) cut = (int)Lp[K];
        if (K > 0) cut = min(cut, (int)Rp[K - 1]);
        __syncthreads();
        if (cut <= nth) first = cut; else last = cut;
    }
    // ---- finish with one warp: short-range introselect + insertion sort, then the std::partition tail
    if (wid == 0) {
        if (fallback) heap_select_fallback(v, first, nth, last, lane);
        else introselect_warp(v, first, last, nth, depth, lane);
        const int res = partition_tail_warp(v, m, len, v[m - 1].response, lane);
        if (lane == 0) sh->n = res;
    }
    __syncthreads();
    const int res = sh->n;
    __syncthreads();
    return res;
}


// ------------------------------------------------------------------------------------------------ A.5 Harris
__device__ __forceinline__ float harris_response(const uint8_t* __restrict__ img, int pitch, int x, int y)
{
    // The 9 x 9 neighbourhood as 9 rows x 3 aligned words, ALL loaded before anything is used: the candidate's loads are
    // in flight together (one L2 round trip per candidate instead of a chain of byte loads -- the selection kernel is
    // latency-bound and Harris was a third of its critical path).  The Sobel sums are taken separably per row:
    //   d[i] = p[i+1] - p[i-1],  s[i] = p[i-1] + 2 p[i] + p[i+1]   ->   Ix = d(r-1) + 2 d(r) + d(r+1),  Iy = s(r+1) - s(r-1)
    const int xa = (x - 4) & ~3;
    const unsigned shb = (unsigned)((x - 4) & 3) * 8u;
    const uint8_t* p = img + (size_t)(y - 4) * pitch + xa;
    uint32_t w[9][3];
#pragma unroll
    for (int r = 0; r < 9; ++r, p += pitch) {
        w[r][0] = ldg_u32_now(p); w[r][1] = ldg_u32_now(p + 4); w[r][2] = ldg_u32_now(p + 8);
    }
    int a = 0, b = 0, c = 0;
    int d0[7] = {}, d1[7] = {}, d2[7] = {}, s0[7] = {}, s1[7] = {}, s2[7] = {};   // rows r-2, r-1, r of the horizontal differences / sums
#pragma unroll
    for (int r = 0; r < 9; ++r) {
        const uint32_t v0 = __funnelshift_r(w[r][0], w[r][1], shb), v1 = __funnelshift_r(w[r][1], w[r][2], shb), v2 = w[r][2] >> shb;
        int px[9];
#pragma unroll
        for (int i = 0; i < 4; ++i) { px[i] = (int)((v0 >> (8 * i)) & 255u); px[4 + i] = (int)((v1 >> (8 * i)) & 255u); }
        px[8] = (int)(v2 & 255u);
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            d0[i] = d1[i]; d1[i] = d2[i]; s0[i] = s1[i]; s1[i] = s2[i];
            d2[i] = px[i + 2] - px[i];
            s2[i] = px[i] + 2 * px[i + 1] + px[i + 2];
        }
        if (r >= 2) {
#pragma unroll
            for (int i = 0; i < 7; ++i) {
                const int Ix = d0[i] + 2 * d1[i] + d2[i];
                const int Iy = s2[i] - s0[i];
                a += Ix * Ix; b += Iy * Iy; c += Ix * Iy;
            }
        }
    }
    const float fa = (float)a, fb = (float)b, fc = (float)c;
    const float det = __fsub_rn(__fmul_rn(fa, fb), __fmul_rn(fc, fc));
    const float tr = __fadd_rn(fa, fb);
    const float ktr2 = __fmul_rn(__fmul_rn(__int_as_float(0x3d23d70a), tr), tr);       // 0.04f
    return __fmul_rn(__fsub_rn(det, ktr2), __int_as_float(0x25ddced1));                // (1/7140)^4, rounded stepwise
}

// ------------------------------------------------------------------------------------------------ row-list gather
// Rows [rb, re) of a level's per-row FAST lists (entries x | score << 16, in x order) -> v[o ..] in raster order.
// Rows in groups of four: the first 128-bit chunk of each row's list (row lists are 32-byte aligned and most hold
// fewer than four survivors) is requested for all four rows before any is consumed, so a thread's gather costs
// about one memory round trip per group instead of one per entry.
__device__ __forceinline__ void gather_rows(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ ent, int ent_pitch,
                                            int rb, int re, int o, Elem* v)
{
    for (int r0 = rb; r0 < re; r0 += 4) {
        int cc[4];
        uint4 w4[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) cc[k] = r0 + k < re ? (int)__ldg(cnt + r0 + k) : 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            w4[k] = make_uint4(0u, 0u, 0u, 0u);
            if (cc[k] > 0) w4[k] = __ldg(reinterpret_cast<const uint4*>(ent + (size_t)(r0 + k) * ent_pitch));
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = r0 + k, c = cc[k];
            const uint32_t ypart = (uint32_t)(r + ORBX_EDGE) << 16;
            const uint32_t first[4] = {w4[k].x, w4[k].y, w4[k].z, w4[k].w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (i < c) {
                    Elem el;
                    el.response = (float)(first[i] >> 16);
                    el.pos = ypart | (first[i] & 0xffffu);
                    v[o++] = el;
                }
            if (c > 4) {
                const uint32_t* e = ent + (size_t)r * ent_pitch;
                for (int i = 4; i < c; ++i) {
                    const uint32_t w = __ldg(e + i);
                    Elem el;
                    el.response = (float)(w >> 16);
                    el.pos = ypart | (w & 0xffffu);
                    v[o++] = el;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ selection kernel
// One CTA per (level, frame): gather the per-row FAST lists (raster order) -> retainBest(2 n_l) on the FAST score
// -> Harris on the survivors -> retainBest(n_l) on Harris.  The final list is left as the prefix of the level's
// global workspace; its length goes to fincnt.  The working array (and the partition scratch) lives in shared
// memory when the level's candidate count fits, else in global memory.
struct SelSmem {
    Elem v[SEL_SMEM_ELEMS];
    uint16_t pos[2 * SEL_SMEM_ELEMS];
    SelShared sh;
};
// grid = (frames, levels): level-major dispatch, so the long level-0 CTAs of every frame start in the first wave and
// the short upper levels fill the tail
__global__ void __launch_bounds__(SEL_NT, 2) k_select(const __grid_constant__ Geom g, const uint8_t* __restrict__ pyr,
                                                      const uint32_t* __restrict__ rowcnt, const uint32_t* __restrict__ rowent,
                                                      Elem* __restrict__ work, uint32_t* __restrict__ selpos, int* __restrict__ fincnt)
{
    __shared__ SelSmem sm;
    Elem* const s_v = sm.v;
    uint16_t* const s_pos = sm.pos;
    SelShared& sh = sm.sh;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int l = blockIdx.y, f = blockIdx.x;
    const LevelGeom& L = g.L[l];
    Elem* gv = work + (size_t)f * g.ws_frame + L.ws_off;
    if (L.in_w <= 0 || L.in_h <= 0) { if (tid == 0) fincnt[f * g.nlevels + l] = 0; return; }
    const uint32_t* cnt = rowcnt + (size_t)f * g.cnt_frame + L.cnt_off;
    const uint32_t* ent = rowent + (size_t)f * g.ent_frame + L.ent_off;
    // ---- gather rows in raster order
    const int nr = L.in_h;
    const int rpt = (nr + SEL_NT - 1) / SEL_NT;
    const int rb = min(tid * rpt, nr), re = min(rb + rpt, nr);
    int mine = 0;
    for (int r = rb; r < re; ++r) mine += (int)cnt[r];
    int inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
    if (lane == 31) sh.warp_a[wid] = inc;
    __syncthreads();
    int woff = 0, total = 0;
#pragma unroll
    for (int i = 0; i < SEL_NT / 32; ++i) { const int s = sh.warp_a[i]; if (i < wid) woff += s; total += s; }
    const int N = total;
    const bool in_smem = N <= SEL_SMEM_ELEMS;
    Elem* v = in_smem ? s_v : gv;
    gather_rows(cnt, ent, L.ent_pitch, rb, re, woff + inc - mine, v);
    __syncthreads();
    uint32_t* gpos = selpos + 2 * ((size_t)f * g.ws_frame + L.ws_off);
    // ---- retainBest(2 n_l) on the FAST score
    const int n1 = in_smem ? retain_best_block<uint16_t>(v, N, 2 * L.quota, s_pos, s_pos + SEL_SMEM_ELEMS, &sh)
                           : retain_best_block<uint32_t>(v, N, 2 * L.quota, gpos, gpos + N, &sh);
    // ---- Harris on the unblurred level
    const uint8_t* img = pyr + (size_t)f * g.pyr_frame + L.img_off;
    for (int i = tid; i < n1; i += SEL_NT) {
        const uint32_t pos = v[i].pos;
        v[i].response = harris_response(img, L.pitch, (int)(pos & 0xffffu), (int)(pos >> 16));
    }
    __syncthreads();
    // ---- retainBest(n_l) on Harris
    const int n2 = in_smem ? retain_best_block<uint16_t>(v, n1, L.quota, s_pos, s_pos + SEL_SMEM_ELEMS, &sh)
                           : retain_best_block<uint32_t>(v, n1, L.quota, gpos, gpos + N, &sh);
    if (tid == 0) fincnt[f * g.nlevels + l] = n2;
    if (v != gv) for (int i = tid; i < n2; i += SEL_NT) gv[i] = v[i];
}

// ------------------------------------------------------------------------------------------------ warp kernels
// Whole-WARP KeyPointsFilter::retainBest(v, m).  Lp / Rp: position scratch, `len` entries each.  Returns the new length (on every lane).
template <typename PosT>
__device__ int retain_best_warp(Elem* v, int len, int m, PosT* Lp, PosT* Rp, int lane)
{
    if (m < 0 || len <= m) return len;
    if (m == 0) return 0;
    const unsigned lt = lanemask_lt();
    const int nth = m - 1;
    int first = 0, last = len, depth = 2 * (31 - __clz(len));
    bool fallback = false;
    while (last - first > SEL_PAR_MIN) {
        if (depth == 0) { fallback = true; break; }          // depth budget spent: libstdc++ switches to __heap_select
        --depth;
        __syncwarp();
        if (lane == 0) elem_swap(v, first, median3_pick(v, first + 1, first + (last - first) / 2, last - 1));
        __syncwarp();
        const float piv = v[first].response;
        const int lo = first + 1;
        int cntL = 0, cntR = 0;                              // Lp: ascending L positions; Rp: ascending R positions (R[k] = Rp[cntR - 1 - k])
#pragma unroll 2
        for (int base = lo; base < last; base += 32) {
            const int i = base + lane;
            bool pL = false, pR = false;
            if (i < last) { const float r = v[i].response; pL = !(r > piv); pR = !(piv > r); }
            const unsigned bL = __ballot_sync(0xffffffffu, pL), bR = __ballot_sync(0xffffffffu, pR);
            if (pL) Lp[cntL + __popc(bL & lt)] = (PosT)i;
            if (pR) Rp[cntR + __popc(bR & lt)] = (PosT)i;
            cntL += __popc(bL); cntR += __popc(bR);
        }
        __syncwarp();
        const int mm = min(cntL, cntR);
        int K = 0;                                           // L ascends, R descends: L[k] < R[k] holds for k < K and fails from K on
        for (int base = 0; base < mm; base += 32) {
            const int k = base + lane;
            const bool c = k < mm && (int)Lp[k] < (int)Rp[cntR - 1 - k];
            const unsigned b = __ballot_sync(0xffffffffu, c);
            K += __popc(b);
            if (b != 0xffffffffu) break;
        }
        for (int k = lane; k < K; k += 32) elem_swap(v, (int)Lp[k], (int)Rp[cntR - 1 - k]);
        int cut = 0x7fffffff;
        if (K < cntL) cut = (int)Lp[K];
        if (K > 0) cut = min(cut, (int)Rp[cntR - K]);
        __syncwarp();
        if (cut <= nth) first = cut; else last = cut;
    }
    if (fallback) heap_select_fallback(v, first, nth, last, lane);
    else introselect_warp(v, first, last, nth, depth, lane);
    return partition_tail_warp(v, m, len, v[m - 1].response, lane);
}

struct SelFastSmem { Elem v[SEL_SMEM_ELEMS]; uint16_t pos[2 * SEL_SMEM_ELEMS]; };

// One warp per (frame, level): gather the per-row FAST lists (raster order) and retainBest(2 n_l) on the FAST score; survivors ->
// the prefix of the level's global workspace, their number -> selcnt.
__global__ void __launch_bounds__(32) k_select_fast(const __grid_constant__ Geom g, const uint32_t* __restrict__ rowcnt,
                                                    const uint32_t* __restrict__ rowent, Elem* __restrict__ work, uint32_t* __restrict__ selpos,
                                                    int* __restrict__ selcnt, int* __restrict__ fincnt)
{
    __shared__ SelFastSmem sm;
    const int lane = threadIdx.x, f = blockIdx.x, l = blockIdx.y;
    const LevelGeom& L = g.L[l];
    Elem* gv = work + (size_t)f * g.ws_frame + L.ws_off;
    if (L.in_w <= 0 || L.in_h <= 0) { if (lane == 0) { selcnt[f * g.nlevels + l] = 0; fincnt[f * g.nlevels + l] = 0; } return; }
    const uint32_t* cnt = rowcnt + (size_t)f * g.cnt_frame + L.cnt_off;
    const uint32_t* ent = rowent + (size_t)f * g.ent_frame + L.ent_off;
    // ---- rows in raster order: lane owns a contiguous block of rows; exclusive prefix of the block sums by shuffles
    const int nr = L.in_h;
    const int rpt = (nr + 31) / 32;
    const int rb = min(lane * rpt, nr), re = min(rb + rpt, nr);
    int mine = 0;
    for (int r = rb; r < re; ++r) mine += (int)__ldg(cnt + r);
    int inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
    const int N = __shfl_sync(0xffffffffu, inc, 31);
    const bool in_smem = N <= SEL_SMEM_ELEMS;
    Elem* v = in_smem ? sm.v : gv;
    gather_rows(cnt, ent, L.ent_pitch, rb, re, inc - mine, v);
    __syncwarp();
    uint32_t* gpos = selpos + 2 * ((size_t)f * g.ws_frame + L.ws_off);
    const int n1 = in_smem ? retain_best_warp<uint16_t>(v, N, 2 * L.quota, sm.pos, sm.pos + SEL_SMEM_ELEMS, lane)
                           : retain_best_warp<uint32_t>(v, N, 2 * L.quota, gpos, gpos + N, lane);
    __syncwarp();
    if (lane == 0) selcnt[f * g.nlevels + l] = n1;
    if (v != gv) for (int i = lane; i < n1; i += 32) gv[i] = v[i];
}

// One thread per candidate that survived the first selection: response <- Harris (A.5) on the unblurred level.
// Block -> (level, chunk of HARRIS_NT candidates) through the per-level block prefix g.L[l].hblk0; a level with more survivors than
// its blocks cover (ties) is finished by striding.
constexpr int HARRIS_NT = 128;
__global__ void __launch_bounds__(HARRIS_NT) k_harris(const __grid_constant__ Geom g, const uint8_t* __restrict__ pyr, Elem* __restrict__ work,
                                                      const int* __restrict__ selcnt)
{
    const int f = blockIdx.y;
    int l = 0;
#pragma unroll 1
    for (int i = 1; i < g.nlevels; ++i) if ((int)blockIdx.x >= g.L[i].hblk0) l = i;
    const LevelGeom& L = g.L[l];
    const int n1 = __ldg(selcnt + f * g.nlevels + l);
    const int nblk = L.hblk;
    Elem* v = work + (size_t)f * g.ws_frame + L.ws_off;
    const uint8_t* img = pyr + (size_t)f * g.pyr_frame + L.img_off;
    for (int i = ((int)blockIdx.x - L.hblk0) * HARRIS_NT + (int)threadIdx.x; i < n1; i += nblk * HARRIS_NT) {
        const uint32_t pos = v[i].pos;
        v[i].response = harris_response(img, L.pitch, (int)(pos & 0xffffu), (int)(pos >> 16));
    }
}

// One warp per (frame, level): retainBest(n_l) on the Harris response.  Dynamic shared memory: `elems` Elem + 2 x `elems` u16.
__global__ void __launch_bounds__(32) k_select_harris(const __grid_constant__ Geom g, Elem* __restrict__ work, uint32_t* __restrict__ selpos,
                                                      const int* __restrict__ selcnt, int* __restrict__ fincnt, int elems)
{
    extern __shared__ __align__(16) uint8_t selh_smem[];
    Elem* s_v = reinterpret_cast<Elem*>(selh_smem);
    uint16_t* s_pos = reinterpret_cast<uint16_t*>(selh_smem + (size_t)elems * sizeof(Elem));
    const int lane = threadIdx.x, f = blockIdx.x, l = blockIdx.y;
    const LevelGeom& L = g.L[l];
    if (L.in_w <= 0 || L.in_h <= 0) return;                  // (fincnt already 0)
    Elem* gv = work + (size_t)f * g.ws_frame + L.ws_off;
    const int n1 = __ldg(selcnt + f * g.nlevels + l);
    const bool in_smem = n1 <= elems && n1 <= 65535;
    Elem* v = gv;
    if (in_smem && n1 > L.quota) {                           // (nothing to select otherwise: the list stays as it is)
        for (int i = lane; i < n1; i += 32) s_v[i] = gv[i];
        v = s_v;
    }
    __syncwarp();
    uint32_t* gpos = selpos + 2 * ((size_t)f * g.ws_frame + L.ws_off);
    const int n2 = v == s_v ? retain_best_warp<uint16_t>(v, n1, L.quota, s_pos, s_pos + elems, lane)
                            : retain_best_warp<uint32_t>(v, n1, L.quota, gpos, gpos + n1, lane);
    __syncwarp();
    if (lane == 0) fincnt[f * g.nlevels + l] = n2;
    if (v != gv) for (int i = lane; i < n2; i += 32) gv[i] = v[i];
}

}  // namespace orbx
