// orbx_select.cuh -- A.4 - A.6 of cv::ORB::detectAndCompute (src/frontend.cpp:153): border-filtered FAST survivors ->
// KeyPointsFilter::retainBest(2 n_l) on the FAST score -> Harris response -> retainBest(n_l) on Harris, in libstdc++'s order.
//
// Three kernels, so that the inherently sequential part is as short as it can be and the rest is wide:
//   k_select_fast    one WARP per (frame, level): gathers the per-row FAST lists in raster order and runs retainBest(2 n_l)
//   k_harris         one THREAD per surviving candidate of the whole batch: the 7x7 Harris response (A.5)
//   k_select_harris  one WARP per (frame, level): retainBest(n_l) on the Harris response; the final list is left as the prefix of
//                    the level's workspace, its length in fincnt
// retainBest = std::nth_element + std::partition; its output ORDER is whatever libstdc++'s __introselect (median-of-3 to first,
// Hoare __unguarded_partition, insertion sort of <= 3, __heap_select once the depth budget is spent) and the bidirectional
// std::partition leave behind, and OpenCV's keypoint order -- and through index tie-breaks the matcher -- depends on it.  A warp
// owns a problem: no block barrier, elements interleaved over the lanes (conflict-free shared / coalesced global access).
//   long ranges: one warp-parallel Hoare pass (SURVEY A.6 / probe E21): with L = ascending positions of !(a > piv) and R = descending
//     positions of !(piv > a) (original contents), the sequential loop swaps a[L[k]] <-> a[R[k]] for k < K, K = #{k : L[k] < R[k]}, and
//     returns cut = min(L[K], R[K-1]).  Ranks come from ballots and popcounts, K from a monotone scan, swaps run 32 at a time.
//   short ranges and the std::partition tail: the warp-cooperative sequential emulation of orbx_kernels.cuh.
// The working array lives in shared memory when the problem fits, else in the level's global workspace (same code).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "orbx_geom.h"

namespace orbx {

constexpr int SELW_PAR_MIN = 32;       // ranges up to this length are finished by the sequential warp emulation

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
    while (last - first > SELW_PAR_MIN) {
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

constexpr int SELF_SMEM_ELEMS = 2048;  // k_select_fast: candidates of one level held in shared memory (more: the global workspace)
struct SelFastSmem { Elem v[SELF_SMEM_ELEMS]; uint16_t pos[2 * SELF_SMEM_ELEMS]; };

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
    const bool in_smem = N <= SELF_SMEM_ELEMS;
    Elem* v = in_smem ? sm.v : gv;
    {
        // Rows in groups of four: the first 128-bit chunk of each row's list (row lists are 32-byte aligned and most hold fewer
        // than four survivors) is requested for all four rows before any is consumed.
        int o = inc - mine;
        for (int r0 = rb; r0 < re; r0 += 4) {
            int cc[4];
            uint4 w4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) cc[k] = r0 + k < re ? (int)__ldg(cnt + r0 + k) : 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                w4[k] = make_uint4(0u, 0u, 0u, 0u);
                if (cc[k] > 0) w4[k] = __ldg(reinterpret_cast<const uint4*>(ent + (size_t)(r0 + k) * L.ent_pitch));
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
                    const uint32_t* e = ent + (size_t)r * L.ent_pitch;
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
    __syncwarp();
    uint32_t* gpos = selpos + 2 * ((size_t)f * g.ws_frame + L.ws_off);
    const int n1 = in_smem ? retain_best_warp<uint16_t>(v, N, 2 * L.quota, sm.pos, sm.pos + SELF_SMEM_ELEMS, lane)
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
