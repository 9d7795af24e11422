// orbx_kernels.cuh -- sm_100a kernels of the ORB extraction path (one stage of cv::ORB::detectAndCompute each;
// the reference invokes that operator at src/frontend.cpp:153).  Stage arithmetic follows SURVEY.md Appendix A
// and is bit-exact against OpenCV: integer stages in integer arithmetic, float stages with explicit
// round-to-nearest intrinsics (never contracted) and __fmaf_rn only where OpenCV's own build uses FMA (A.8).
//
//   k_gray          A.1   BGR -> gray (level 0)                         HBM-bound, 16 px / thread
//   k_pyr_down      A.2   INTER_LINEAR_EXACT level l from level l-1     thread = 8 output columns x 16 rows, source rows streamed by cp.async
//   k_fast_bands    A.3   FAST-9/16 score + 3x3 NMS -> per-row lists    smem tiles with halos, u16x2 SIMD min/max,
//                                                                       ballot compaction, raster order kept
//   k_select        A.4-6 retainBest(2n) -> Harris -> retainBest(n)     libstdc++ introselect order reproduced
//   k_blur          A.8   7x7 float-FMA Gaussian of the samplable region of every level (register sliding window)
// The descriptor stage (A.7-10) is k_describe_tma in orbx_desc.cuh.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "orbx_geom.h"

namespace orbx {

// ------------------------------------------------------------------------------------------------ helpers
__device__ __forceinline__ unsigned lanemask_lt() { unsigned m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }
__device__ __forceinline__ unsigned vmin2(unsigned a, unsigned b) { return __vminu2(a, b); }
__device__ __forceinline__ unsigned vmax2(unsigned a, unsigned b) { return __vmaxu2(a, b); }
__device__ __forceinline__ unsigned vmax3(unsigned a, unsigned b, unsigned c) { return __vimax3_u16x2(a, b, c); }
__device__ __forceinline__ unsigned vmin3(unsigned a, unsigned b, unsigned c) { return __vimin3_u16x2(a, b, c); }

// Loads the compiler may not sink next to their first use: issued back to back, they are all in flight together.
__device__ __forceinline__ uint32_t ldg_u8_now(const uint8_t* p) { uint32_t v; asm volatile("ld.global.nc.u8 %0, [%1];" : "=r"(v) : "l"(p)); return v; }
__device__ __forceinline__ uint32_t ldg_u32_now(const void* p) { uint32_t v; asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p)); return v; }

// cp.async (LDGSTS): global -> shared copies that cost neither registers nor scoreboards while in flight (a warp has six
// scoreboards; a deep register-prefetch pipeline ends up sharing them and the oldest load waits for the youngest).
__device__ __forceinline__ void cp_async_4(unsigned dst, const void* src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(dst), "l"(src) : "memory"); }
__device__ __forceinline__ void cp_async_8(unsigned dst, const void* src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(dst), "l"(src) : "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }
__device__ __forceinline__ uint2 lds_v2(unsigned addr)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ unsigned lds_u32(unsigned addr) { unsigned v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v; }
__device__ __forceinline__ unsigned lds_u16(unsigned addr) { unsigned short v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr) : "memory"); return v; }
__device__ __forceinline__ unsigned lds_u8(unsigned addr) { unsigned v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v; }
__device__ __forceinline__ void sts_u8(unsigned addr, unsigned v) { asm volatile("st.shared.u8 [%0], %1;" :: "r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_u16(unsigned addr, unsigned v) { asm volatile("st.shared.u16 [%0], %1;" :: "r"(addr), "h"((unsigned short)v) : "memory"); }
__device__ __forceinline__ uint4 lds_v4(unsigned addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ int dp4a_us(unsigned a_u8x4, unsigned b_s8x4, int c)       // sum of u8 * s8 products + c
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_u8x4), "r"(b_s8x4), "r"(c));
    return d;
}

// ------------------------------------------------------------------------------------------------ A.1 gray
// g = (3735 B + 19235 G + 9798 R + 16384) >> 15.
// 4 gray pixels from 12 BGR bytes: coefficients split into high / low bytes so each pixel is two IDP.4A
//   3735 B + 19235 G + 9798 R + 16384 = 256 (14 B + 75 G + 38 R) + (151 B + 35 G + 70 R) + 16384      (exact)
__device__ __forceinline__ uint32_t gray4(uint32_t w0, uint32_t w1, uint32_t w2)
{
    constexpr uint32_t CH_ = 14u | (75u << 8) | (38u << 16), CL_ = 151u | (35u << 8) | (70u << 16);
    const uint32_t p0 = w0, p1 = __byte_perm(w0, w1, 0x0543), p2 = __byte_perm(w1, w2, 0x0432), p3 = w2 >> 8;
    const uint32_t g0 = (__dp4a(p0, CH_, 0u) * 256u + __dp4a(p0, CL_, 16384u)) >> 15;
    const uint32_t g1 = (__dp4a(p1, CH_, 0u) * 256u + __dp4a(p1, CL_, 16384u)) >> 15;
    const uint32_t g2 = (__dp4a(p2, CH_, 0u) * 256u + __dp4a(p2, CL_, 16384u)) >> 15;
    const uint32_t g3 = (__dp4a(p3, CH_, 0u) * 256u + __dp4a(p3, CL_, 16384u)) >> 15;
    return g0 | (g1 << 8) | (g2 << 16) | (g3 << 24);
}

// One thread = 16 consecutive pixels of one row: three 128-bit loads (48 BGR bytes), one 128-bit store -- the kernel
// is a pure HBM stream (3 bytes in, 1 byte out per pixel).  Unaligned inputs / row tails fall back to byte loads.
template <int CH>
__global__ void __launch_bounds__(256) k_gray(const uint8_t* __restrict__ in, unsigned long long frame_stride,
                                              unsigned long long step, int aligned16, const __grid_constant__ Geom g,
                                              uint8_t* __restrict__ pyr)
{
    const LevelGeom& L = g.L[0];
    const int x = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int f = blockIdx.z;
    if (y >= L.h || x >= L.pitch) return;
    const uint8_t* src = in + (size_t)f * frame_stride + (size_t)y * step + (size_t)x * CH;
    uint4 out = make_uint4(0u, 0u, 0u, 0u);
    if (aligned16 && x + 15 < L.w) {
        const uint4* s4 = reinterpret_cast<const uint4*>(src);
        if (CH == 3) {
            const uint4 a = __ldg(s4), b = __ldg(s4 + 1), c = __ldg(s4 + 2);
            out = make_uint4(gray4(a.x, a.y, a.z), gray4(a.w, b.x, b.y), gray4(b.z, b.w, c.x), gray4(c.y, c.z, c.w));
        } else {
            out = __ldg(s4);
        }
    } else {
        uint32_t o[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if (x + k < L.w) {
                const uint8_t* s = src + (size_t)k * CH;
                const uint32_t p = CH == 3 ? (3735u * __ldg(s) + 19235u * __ldg(s + 1) + 9798u * __ldg(s + 2) + 16384u) >> 15 : (uint32_t)__ldg(s);
                o[k >> 2] |= p << (8 * (k & 3));
            }
        out = make_uint4(o[0], o[1], o[2], o[3]);
    }
    *reinterpret_cast<uint4*>(pyr + (size_t)f * g.pyr_frame + L.img_off + (size_t)y * L.pitch + x) = out;   // pitch, offsets: multiples of 16
}

// ------------------------------------------------------------------------------------------------ A.2 pyramid
// dst(x,y) = (h0*(256-cy) + h1*cy + 32768) >> 16,  h = p[i0]*(256-cx) + p[i1]*cx  (8.8 taps from host tables).
// A quad of 4 adjacent output columns keeps its taps, byte offsets and funnel-shift amounts in registers; a source row
// costs it three (wide: four) aligned 32-bit words (the 4 outputs read <= 9 consecutive source bytes at the reference's
// ratio 1.2); each output's horizontal pass is one funnel shift + one IDP.2A (u16 taps x u8 pixels), taken once per
// source row and reused by the next output row that needs the same row.
constexpr int PYR_RH = 16;          // output rows per thread
struct PyrRow { uint32_t h[4]; };
// One level per launch.  The kernel is organised around the SOURCE rows: the thread streams the source rows it needs, in order,
// through a private shared-memory ring filled by cp.async (PYR_DEPTH rows in flight), takes the horizontal pass of
// each once, and emits an output row as soon as its lower source row has passed.  Load latency sits under the
// arithmetic of the rows already there instead of in front of every output row.
// A thread owns PYR_NQ = 2 adjacent column quads (8 output columns) of a strip of PYR_RH rows: the per-row control work
// (ring slot, emission test, tap prefetch, pointer updates -- more than half of the instructions of a one-quad thread) is
// shared by both quads, each of which keeps its own 3- or 4-word source window.  Work items (column octet, strip) of a
// level are flattened over the CTAs, so warps stay full on narrow levels.
constexpr int PYR_DEPTH = 8;
constexpr int PYR_NT = 128;
constexpr int PYR_NQ = 2;
// WIDE = false: the 4 outputs of a quad reach at most 7 bytes past its aligned first source byte (scale factors up to
// ~1.5, the reference's 1.2 included): 3 source words, one predicated select per operand.  WIDE = true: up to 11 bytes
// (scale factors up to ~2.6): 4 source words, two selects per operand.
template <bool WIDE>
__global__ void __launch_bounds__(PYR_NT) k_pyr_down(const __grid_constant__ Geom g, int l, uint8_t* pyr, const uint32_t* __restrict__ tabs)
{
    __shared__ __align__(16) uint8_t s_ring[PYR_DEPTH * PYR_NQ * PYR_NT * 16];
    const LevelGeom& D = g.L[l];
    const LevelGeom& S = g.L[l - 1];
    const int noct = D.pitch >> 3;                           // column octets per row (pitch is a multiple of 16)
    const int item = blockIdx.x * PYR_NT + threadIdx.x;
    const int strip = item / noct, oct = item - strip * noct;
    const int x = oct * 8;
    const int ys = strip * PYR_RH, ye = min(ys + PYR_RH, D.h);
    const int f = blockIdx.y;
    if (ys >= ye) return;
    uint8_t* dst = pyr + (size_t)f * g.pyr_frame + D.img_off + (size_t)ys * D.pitch + x;
    if (x >= D.w) {                                          // row padding: keep it zero
        for (int y = ys; y < ye; ++y, dst += D.pitch) *reinterpret_cast<uint2*>(dst) = make_uint2(0u, 0u);
        return;
    }
    uint32_t coef[PYR_NQ][4], sh[PYR_NQ][4];
    bool hi[PYR_NQ][4], hi2[PYR_NQ][4];
    int a[PYR_NQ];                                           // aligned source byte each quad is addressed from
    bool w2ok[PYR_NQ], w3ok[PYR_NQ];
#pragma unroll
    for (int q = 0; q < PYR_NQ; ++q) {
        const int xq = x + 4 * q;
        a[q] = xq < D.w ? ((int)(__ldg(tabs + D.xtab + xq) & 0xffffu) & ~3) : a[0];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t t = (xq + k < D.w) ? __ldg(tabs + D.xtab + xq + k) : (uint32_t)a[q];   // padding columns: taps 0 -> output 0
            const int off = (int)(t & 0xffffu) - a[q];       // 0 .. 7 (narrow), 0 .. 11 (wide)
            const uint32_t c1 = t >> 16;
            coef[q][k] = (xq + k < D.w) ? ((256u - c1) | (c1 << 16)) : 0u;
            hi[q][k] = off >= 4;
            hi2[q][k] = off >= 8;
            sh[q][k] = (uint32_t)(off & 3) * 8u;
        }
        w2ok[q] = a[q] + 8 < S.pitch;
        w3ok[q] = WIDE && a[q] + 12 < S.pitch;
    }
    const uint32_t* ytab = tabs + D.ytab;
    const int s0 = (int)(__ldg(ytab + ys) & 0xffffu);
    const int s1 = min((int)(__ldg(ytab + ye - 1) & 0xffffu) + 1, S.h - 1);         // last source row needed
    const uint8_t* src = pyr + (size_t)f * g.pyr_frame + S.img_off + (size_t)s0 * S.pitch;
    // ring slot d: [quad 0: 16 B x PYR_NT threads][quad 1: 16 B x PYR_NT threads]  (each LDS.128 conflict-free)
    const unsigned ring = (unsigned)__cvta_generic_to_shared(s_ring) + threadIdx.x * 16u;
    constexpr unsigned SLOT = PYR_NQ * PYR_NT * 16u;
    auto fetch = [&](unsigned slot_addr, const uint8_t* row) {
#pragma unroll
        for (int q = 0; q < PYR_NQ; ++q) {
            const unsigned sa = slot_addr + q * (PYR_NT * 16u);
            const uint8_t* p = row + a[q];
            cp_async_4(sa, p); cp_async_4(sa + 4u, p + 4);
            if (w2ok[q]) cp_async_4(sa + 8u, p + 8);
            if (w3ok[q]) cp_async_4(sa + 12u, p + 12);
        }
    };
#pragma unroll
    for (int d = 0; d < PYR_DEPTH; ++d) {
        if (s0 + d <= s1) fetch(ring + d * SLOT, src + (size_t)d * S.pitch);
        cp_async_commit();
    }
    src += (size_t)PYR_DEPTH * S.pitch;
    // Output-row bookkeeping: `emit_at` is the source row at which the pending output row y can be produced
    // (y1 = min(y0 + 1, S.h - 1)); the taps of row y + 1 are fetched one row ahead.
    int y = ys;
    uint32_t ty = __ldg(ytab + y), ty_next = y + 1 < ye ? __ldg(ytab + y + 1) : 0u;
    int emit_at = min((int)(ty & 0xffffu) + 1, S.h - 1);
    int to_fetch = (s1 - s0 + 1) - PYR_DEPTH;               // source rows not yet requested
    unsigned sa = ring;
    const unsigned ring_end = ring + PYR_DEPTH * SLOT;
    PyrRow hA[PYR_NQ], hB[PYR_NQ];                           // horizontal passes of the last two source rows (ping-pong)
#pragma unroll
    for (int q = 0; q < PYR_NQ; ++q)
#pragma unroll
        for (int k = 0; k < 4; ++k) { hA[q].h[k] = 0; hB[q].h[k] = 0; }
    // one source row: wait, read, refill the slot, horizontal pass into `hc`, emit what became complete
    auto step = [&](int s, const PyrRow* hp, PyrRow* hc) {
        cp_async_wait<PYR_DEPTH - 1>();
        uint4 w[PYR_NQ];
#pragma unroll
        for (int q = 0; q < PYR_NQ; ++q) w[q] = lds_v4(sa + q * (PYR_NT * 16u));
        if (to_fetch > 0) fetch(sa, src);
        cp_async_commit();
        --to_fetch;
        src += S.pitch;
        sa += SLOT;
        if (sa == ring_end) sa = ring;
#pragma unroll
        for (int q = 0; q < PYR_NQ; ++q) {
            const uint32_t w2 = w2ok[q] ? w[q].z : 0u, w3 = w3ok[q] ? w[q].w : 0u;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint32_t lo = hi[q][k] ? w[q].y : w[q].x, up = hi[q][k] ? w2 : w[q].y;
                if (WIDE) { lo = hi2[q][k] ? w2 : lo; up = hi2[q][k] ? w3 : up; }
                hc[q].h[k] = __dp2a_lo(coef[q][k], __funnelshift_r(lo, up, sh[q][k]), 0u);
            }
        }
        while (emit_at == s && y < ye) {                     // (two outputs per source row only when the bottom row clamps)
            const bool clamped = (int)(ty & 0xffffu) == s;   // y1 == y0: both taps read the last source row
            const uint32_t cy1 = ty >> 16, cy0 = 256u - cy1;
            uint32_t out[PYR_NQ];
            // vertical pass: h <= 255 * 256, so top * cy0 + cur * cy1 + 2^15 < 2^24 and its byte 2 IS the rounded pixel
            // (never above 255): two IMADs per pixel on the FMA pipe and three PRMTs per quad to gather the bytes
            auto blend = [&](const PyrRow* top) {
#pragma unroll
                for (int q = 0; q < PYR_NQ; ++q) {
                    uint32_t v[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) v[k] = top[q].h[k] * cy0 + (hc[q].h[k] * cy1 + 32768u);
                    out[q] = __byte_perm(__byte_perm(v[0], v[1], 0x0062), __byte_perm(v[2], v[3], 0x0062), 0x5410);
                }
            };
            if (clamped) blend(hc); else blend(hp);
            *reinterpret_cast<uint2*>(dst) = make_uint2(out[0], out[1]);
            dst += D.pitch;
            ++y;
            ty = ty_next;
            emit_at = min((int)(ty & 0xffffu) + 1, S.h - 1);
            if (y + 1 < ye) ty_next = __ldg(ytab + y + 1);
        }
    };
#pragma unroll 1
    for (int s = s0; s <= s1; s += 2) {
        step(s, hA, hB);
        if (s + 1 <= s1) step(s + 1, hB, hA);
    }
}

// ------------------------------------------------------------------------------------------------ A.3 FAST + NMS
// One CTA = one band of R inner rows of one level of one frame, walked left to right in chunks of CWO = 248 output
// columns, so every row's survivors come out in x order and the per-row lists concatenate to OpenCV's raster order.
// Only the region that can survive the 31-px border filter is evaluated (SURVEY A.10).
//
// Per chunk (score tile = (R+2) rows x 256 columns, x = ox0-4 .. ox0+251), four block barriers:
//   load      (R+8) x 288 pixels widened to u16 into smem with 128-bit global loads (16-byte aligned tile origin)
//   phase A   per WARP, on its own (row, 128-pixel half) items: 4-compass-point rejection test of every pixel quad in
//             u16x2 SIMD (native VIMNMX.U16x2) from five 64-bit shared loads; a quad with any passing pixel becomes one
//             entry of the warp's private quad queue (one ballot per item, no atomics, no block scan, no barrier)
//   phase A2  the same warp, on its queued quads: second rejection test on the two diagonal pairs of the circle, then the
//             surviving pixels are expanded to pixel entries (bit-sliced warp prefix), in place
//   phase B   the same warp runs the full 16-point test on its pixel queue.  Each circle pixel is packed
//             (p | (255-p) << 16) so ONE sliding max over the 16 nine-long arcs (VIMNMX3.U16x2) yields both
//             min-of-max(p) and max-of-min(p):  A = v - min_arcs max p,  -B = max_arcs min p - v,
//             score = max(A, -B) - 1 (corner iff > t).  Corners inside the output region go to a private NMS queue.
//   phase C   3x3 NMS (strict >) of the queued corners on the shared score tile -> per-row bit masks
//   phase D   ordered extraction of the bit masks (popc prefix) -> global per-row lists
// Measured and dropped (tools/stage_times.py, DESIGN.md section 8): register-prefetched next tile with three barriers per chunk,
// persistent CTAs over (band, frame) items with static or ticket scheduling, a CTA-wide survivor queue that balances
// phase B across warps, a u8 image tile (half the shared-memory wavefronts, more PRMT), 6-7 CTAs per SM by register cap.
template <int R, int NT>
__global__ void __launch_bounds__(NT) k_fast_bands(const __grid_constant__ Geom g, const uint8_t* __restrict__ pyr,
                                                   uint32_t* __restrict__ rowcnt, uint32_t* __restrict__ rowent)
{
    constexpr int CWO = 248;               // output columns per chunk
    constexpr int SP = 256;                // score tile pitch (bytes) = pixels evaluated per row
    constexpr int SR = R + 2;              // score tile rows
    constexpr int TP = SP + 32;            // image tile pitch (pixels, u16 each): 16-pixel aligned origin <= ox0-8, 18 x 16 pixels
    constexpr int TPW = TP / 2;            // ... in 32-bit words
    constexpr int TR = R + 8;              // image tile rows
    constexpr int MW = 8;                  // mask words per row (248 bits used)
    constexpr int T = ORBX_FAST_T;
    constexpr int NWARP = NT / 32;
    constexpr int ITEMS = (2 * SR + NWARP - 1) / NWARP;   // (row, half) items per warp
    constexpr int QCAP = ITEMS * 128;      // private queue capacity: every pixel of the warp's items
    static_assert(R * MW <= NT, "phase D needs one thread per mask word");
    static_assert((R * MW) % 32 == 0, "phase D shuffles with a full-warp mask: its threads must be whole warps (R = 14 hangs)");

    __shared__ __align__(16) uint16_t s_img[TR * TP];
    __shared__ __align__(16) uint8_t s_score[SR * SP];
    __shared__ uint16_t s_q[NWARP][QCAP];  // pass queues:   sy << 8 | sx; compacted IN PLACE to the corner queues (NMS candidates
                                           // inside the output region) as phase B consumes them: a corner's slot index never
                                           // passes the entries still to be read, so no second queue is needed
    __shared__ uint32_t s_mask[R * MW];
    __shared__ uint32_t s_rowcnt[R];

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned lt = lanemask_lt();
    const int f = blockIdx.y;
    int l = 0;
#pragma unroll 1
    for (int i = 1; i < g.nlevels; ++i) if ((int)blockIdx.x >= g.L[i].band0) l = i;
    const LevelGeom& L = g.L[l];
    const int band = blockIdx.x - L.band0;
    if (band >= L.nbands) return;
    const int y0 = ORBX_EDGE + band * R;
    const int y1 = min(y0 + R, L.h - ORBX_EDGE);           // output rows [y0, y1)
    const int nsr = y1 - y0 + 2;                            // score rows in use
    const int xend = L.w - ORBX_EDGE;                       // output cols [31, xend)
    const uint8_t* img = pyr + (size_t)f * g.pyr_frame + L.img_off;
    uint32_t* cnt_out = rowcnt + (size_t)f * g.cnt_frame + L.cnt_off;
    uint32_t* ent_out = rowent + (size_t)f * g.ent_frame + L.ent_off;

    if (tid < R) s_rowcnt[tid] = 0;
    uint16_t* myq = s_q[wid];
    uint16_t* mycq = s_q[wid];

    for (int ox0 = 28; ox0 < xend; ox0 += CWO) {
        const int ox1 = min(ox0 + CWO, xend);
        const int ix0 = (ox0 - 8) & ~15;                     // 16-byte aligned tile origin
        const int xo = (ox0 - 8) - ix0;                      // 0, 4, 8 or 12: tile x of score column sx is sx + 4 + xo
        const int need = min(ox1 - ox0 + 6, SP);             // score columns that matter: x = ox0-4 .. ox1+1
        __syncthreads();                                     // previous chunk fully consumed
        // ---- load tile rows [y0-4, y1+4): 128-bit loads, 16 pixels widened to u16 per thread and step
        {
            const int rows = y1 - y0 + 8;
            constexpr int CPR = TP / 16;                     // 16-pixel columns per tile row
            const int clast = (xo + need + 16) >> 4;         // last column holding a pixel phase A / B can touch
            for (int i = tid; i < rows * CPR; i += NT) {
                const int ty = i / CPR, col = i - ty * CPR;
                if (col > clast) continue;
                const int gx = ix0 + col * 16;
                uint4 w = make_uint4(0, 0, 0, 0);
                if (gx < L.pitch) w = __ldg(reinterpret_cast<const uint4*>(img + (size_t)(y0 - 4 + ty) * L.pitch + gx));
                uint4* d = reinterpret_cast<uint4*>(&s_img[ty * TP + col * 16]);
                d[0] = make_uint4(__byte_perm(w.x, 0, 0x4140), __byte_perm(w.x, 0, 0x4342), __byte_perm(w.y, 0, 0x4140), __byte_perm(w.y, 0, 0x4342));
                d[1] = make_uint4(__byte_perm(w.z, 0, 0x4140), __byte_perm(w.z, 0, 0x4342), __byte_perm(w.w, 0, 0x4140), __byte_perm(w.w, 0, 0x4342));
            }
            for (int i = tid; i < SR * SP / 16; i += NT) reinterpret_cast<uint4*>(s_score)[i] = make_uint4(0, 0, 0, 0);
            if (tid < R * MW) s_mask[tid] = 0;
        }
        __syncthreads();
        // ---- phase A (per warp): compass rejection on (row, 128-pixel half) items -> private QUAD queue
        // Shared memory is addressed through one precomputed 32-bit base per chunk (LDS with immediate offsets).  Only about
        // one pixel in 13 passes, so the per-item bookkeeping is kept to ONE ballot: a lane whose quad has any passing
        // pixel appends one 16-bit quad entry (sy << 10 | quad column << 4 | 4 pass flags).  The quad queue sits in the
        // last quarter of the warp's queue region.
        int qn4 = 0;
        constexpr int QQ0 = QCAP - ITEMS * 32;               // first slot of the quad queue
        {
            constexpr unsigned K = ((511u - T) << 16) | (511u - T);
            const unsigned qq_s = (unsigned)__cvta_generic_to_shared(myq + QQ0);
            // 8-byte aligned: word index (sy+3)*TPW + 2q + 2 + xo/2 is even (TPW, xo/2 even)
            const unsigned lane_s = (unsigned)__cvta_generic_to_shared(s_img) + (unsigned)(3 * TPW + 2 * lane + 2 + (xo >> 1)) * 4u;
            for (int item = wid; item < 2 * nsr; item += NWARP) {
                const int sy = item >> 1, half = item & 1;
                if (half * 128 >= need) continue;            // warp-uniform: no needed pixel in this half
                const int q = half * 32 + lane;              // quad column
                unsigned m0 = 0, m1 = 0;
                if (4 * q < need) {
                    const unsigned ad = lane_s + (unsigned)(sy * TPW + half * 64) * 4u;
                    const uint2 c = lds_v2(ad), n = lds_v2(ad - 3 * TPW * 4), s = lds_v2(ad + 3 * TPW * 4), e2 = lds_v2(ad + 8), w2 = lds_v2(ad - 8);
                    const unsigned e0 = __byte_perm(c.y, e2.x, 0x5432), e1 = __byte_perm(e2.x, e2.y, 0x5432);
                    const unsigned w0 = __byte_perm(w2.x, w2.y, 0x5432), w1 = __byte_perm(w2.y, c.x, 0x5432);
                    const unsigned D0 = vmax2(vmin2(n.x, s.x), vmin2(e0, w0)), B0 = vmin2(vmax2(n.x, s.x), vmax2(e0, w0));
                    const unsigned D1 = vmax2(vmin2(n.y, s.y), vmin2(e1, w1)), B1 = vmin2(vmax2(n.y, s.y), vmax2(e1, w1));
                    m0 = (c.x + K - D0) | (B0 + K - c.x);
                    m1 = (c.y + K - D1) | (B1 + K - c.y);
                }
                // pass flags of the quad's four pixels: bits 9 / 25 of m0 and (moved up one) bits 10 / 26 of m1, folded to
                // a nibble: bit 0 = pixel 0, bit 1 = pixel 2, bit 2 = pixel 1, bit 3 = pixel 3
                const unsigned pf = (m0 & 0x02000200u) | ((m1 << 1) & 0x04000400u);
                const unsigned nib = ((pf | (pf >> 14)) >> 9) & 15u;
                const unsigned any = __ballot_sync(0xffffffffu, nib != 0u);
                if (nib) sts_u16(qq_s + 2u * (unsigned)(qn4 + __popc(any & lt)), (unsigned)(sy << 10) | (unsigned)(q << 4) | nib);
                qn4 += __popc(any);
            }
        }
        __syncwarp();
        // ---- phase A2 (same warp): quad entries -> pixel entries (sy << 8 | sx), 32 quad entries at a time.
        // First the SECOND rejection test, on the quads that survived only: the two diagonal opposite pairs of the circle
        // ((+-2, +-2): points 2/10 and 6/14) must also hold a darker or a brighter pixel each -- same u16x2 arithmetic as
        // phase A, from three loads per row +-2.  It roughly halves the pixels that reach the 16-point test, whose 17
        // scattered 16-bit loads (bank conflicts) are the expensive part.  (The flags of the two tests are ANDed per pixel
        // without their polarity: still a necessary condition.)
        // Then each lane counts its 0..4 flagged pixels; the counts' three bit planes go through three ballots (prefix =
        // popc of the lower lanes' bits, weighted 1 / 2 / 4) and the lane writes its entries back to back.  (Queue order is
        // free: phase B scores every entry, the NMS works on bits.)  In place: after k quad entries at most
        // 4k <= 3 * ITEMS * 32 + k pixel slots are written, which never reaches the unread part of the quad queue.
        int qn = 0;
        {
            constexpr unsigned K = ((511u - T) << 16) | (511u - T);
            const unsigned q_s = (unsigned)__cvta_generic_to_shared(myq);
            const unsigned img_q = (unsigned)__cvta_generic_to_shared(s_img) + (unsigned)(3 * TPW + 2 + (xo >> 1)) * 4u;   // quad (sy, q) at + (sy * TPW + 2q) * 4
            for (int i0 = 0; i0 < qn4; i0 += 32) {
                const int i = i0 + lane;
                unsigned e = 0;
                if (i < qn4) {
                    e = lds_u16(q_s + 2u * (unsigned)(QQ0 + i));
                    const unsigned ad = img_q + ((e >> 10) * TPW + ((e >> 3) & 0x7Eu)) * 4u;
                    const unsigned up = ad - 2 * TPW * 4, dn = ad + 2 * TPW * 4;
                    const uint2 c = lds_v2(ad), u = lds_v2(up), d = lds_v2(dn);
                    const unsigned um = lds_u32(up - 4), upp = lds_u32(up + 8), dm = lds_u32(dn - 4), dpp = lds_u32(dn + 8);
                    // pixels 0,1: NW = um, NE = u.y, SW = dm, SE = d.y;   pixels 2,3: NW = u.x, NE = upp, SW = d.x, SE = dpp
                    const unsigned D0 = vmax2(vmin2(um, d.y), vmin2(u.y, dm)), B0 = vmin2(vmax2(um, d.y), vmax2(u.y, dm));
                    const unsigned D1 = vmax2(vmin2(u.x, dpp), vmin2(upp, d.x)), B1 = vmin2(vmax2(u.x, dpp), vmax2(upp, d.x));
                    const unsigned m0 = (c.x + K - D0) | (B0 + K - c.x);
                    const unsigned m1 = (c.y + K - D1) | (B1 + K - c.y);
                    const unsigned pf = (m0 & 0x02000200u) | ((m1 << 1) & 0x04000400u);
                    e &= 0xFFF0u | (((pf | (pf >> 14)) >> 9) & 15u);
                }
                const unsigned cnt = (unsigned)__popc(e & 15u);      // 0 .. 4
                const unsigned c0 = __ballot_sync(0xffffffffu, cnt & 1u), c1 = __ballot_sync(0xffffffffu, cnt & 2u), c2 = __ballot_sync(0xffffffffu, cnt & 4u);
                const unsigned pos = (unsigned)qn + __popc(c0 & lt) + 2u * __popc(c1 & lt) + 4u * __popc(c2 & lt);
                qn += __popc(c0) + 2 * __popc(c1) + 4 * __popc(c2);
                const unsigned ent = (e >> 2) & 0x3FFCu;             // sy << 8 | 4 * quad column
                unsigned sa = q_s + 2u * pos;
                if (e & 1u) { sts_u16(sa, ent); sa += 2u; }
                if (e & 4u) { sts_u16(sa, ent + 1u); sa += 2u; }
                if (e & 2u) { sts_u16(sa, ent + 2u); sa += 2u; }
                if (e & 8u) sts_u16(sa, ent + 3u);
            }
        }
        __syncwarp();
        // ---- phase B (same warp): full segment test + score; corners inside the output region -> private NMS queue
        int cn = 0;
        {
            const unsigned q_s = (unsigned)__cvta_generic_to_shared(myq);
            const unsigned img_s = (unsigned)__cvta_generic_to_shared(s_img) + (unsigned)(3 * TP + 4 + xo) * 2u;   // pixel (sy, sx) at + (sy * TP + sx) * 2
            const unsigned sc_s = (unsigned)__cvta_generic_to_shared(s_score);
            // sx window of corners that belong to this chunk's output region: x = ox0 - 4 + sx in [max(ox0, EDGE), ox1)
            const int sx_lo = max(ox0, ORBX_EDGE) - (ox0 - 4), sx_hi = ox1 - (ox0 - 4), sy_hi = y1 - y0;
            for (int i0 = 0; i0 < qn; i0 += 32) {
                const int i = i0 + lane;
                bool corner = false;
                unsigned e = 0;
                if (i < qn) {
                    e = lds_u16(q_s + 2u * (unsigned)i);
                    const unsigned sy = e >> 8, sx = e & 255u;
                    const unsigned c = img_s + (sy * TP + sx) * 2u;
                    const int v = (int)lds_u16(c);
                    unsigned q[16];
#define ORBX_PK(k, dx, dy) q[k] = lds_u16(c + ((dy) * TP + (dx)) * 2) * 0xFFFF0001u + 0x00FF0000u
                    ORBX_PK(0, 0, 3);   ORBX_PK(1, 1, 3);   ORBX_PK(2, 2, 2);    ORBX_PK(3, 3, 1);
                    ORBX_PK(4, 3, 0);   ORBX_PK(5, 3, -1);  ORBX_PK(6, 2, -2);   ORBX_PK(7, 1, -3);
                    ORBX_PK(8, 0, -3);  ORBX_PK(9, -1, -3); ORBX_PK(10, -2, -2); ORBX_PK(11, -3, -1);
                    ORBX_PK(12, -3, 0); ORBX_PK(13, -3, 1); ORBX_PK(14, -2, 2);  ORBX_PK(15, -1, 3);
#undef ORBX_PK
                    unsigned m3[16], m9[16];
#pragma unroll
                    for (int k = 0; k < 16; ++k) m3[k] = vmax3(q[k], q[(k + 1) & 15], q[(k + 2) & 15]);
#pragma unroll
                    for (int k = 0; k < 16; ++k) m9[k] = vmax3(m3[k], m3[(k + 3) & 15], m3[(k + 6) & 15]);
                    unsigned mm = vmin3(vmin3(vmin3(m9[0], m9[1], m9[2]), vmin3(m9[3], m9[4], m9[5]), vmin3(m9[6], m9[7], m9[8])),
                                        vmin3(vmin3(m9[9], m9[10], m9[11]), vmin3(m9[12], m9[13], m9[14]), m9[15]),
                                        0xFFFFFFFFu);
                    const int A = v - (int)(mm & 0xffffu);
                    const int nB = 255 - (int)(mm >> 16) - v;
                    const int sc = max(A, nB);
                    if (sc > T) {
                        sts_u8(sc_s + sy * SP + sx, (unsigned)(sc - 1));
                        corner = (int)sx >= sx_lo && (int)sx < sx_hi && sy - 1u < (unsigned)sy_hi;   // 1 <= sy <= y1 - y0
                    }
                }
                const unsigned bc = __ballot_sync(0xffffffffu, corner);
                __syncwarp();                                // every lane has read its entry of this batch before slots <= i0 + 31 are rewritten
                if (corner) sts_u16(q_s + 2u * (unsigned)(cn + __popc(bc & lt)), e);
                cn += __popc(bc);
            }
        }
        __syncthreads();                                     // every score of the tile is in place
        // ---- phase C (per warp): 3x3 NMS of its queued corners
        for (int i = lane; i < cn; i += 32) {
            const int e = mycq[i];
            const int sy = e >> 8, sx = e & 255;
            const uint8_t* p = &s_score[sy * SP + sx];
            const int s = p[0];
            if (s > p[-1] && s > p[1] && s > p[-SP - 1] && s > p[-SP] && s > p[-SP + 1] && s > p[SP - 1] && s > p[SP] && s > p[SP + 1]) {
                const int bit = sx - 4;
                atomicOr(&s_mask[(sy - 1) * MW + (bit >> 5)], 1u << (bit & 31));
            }
        }
        __syncthreads();
        // ---- phase D: ordered extraction; thread t owns mask word t (MW consecutive lanes = one row)
        if (tid < R * MW) {
            const int row = tid / MW, wi = tid - row * MW;
            uint32_t m = s_mask[tid];
            const int cnt = __popc(m);
            int pre = cnt;                                   // inclusive prefix inside the row's MW-lane group
#pragma unroll
            for (int d = 1; d < MW; d <<= 1) {
                const int o = __shfl_up_sync(0xffffffffu, pre, d, MW);
                if (wi >= d) pre += o;
            }
            const uint32_t base = s_rowcnt[row];
            __syncwarp();
            uint32_t slot = base + pre - cnt;
            uint32_t* dst = ent_out + (size_t)(y0 - ORBX_EDGE + row) * L.ent_pitch;
            while (m) {
                const int b = __ffs(m) - 1;
                m &= m - 1;
                const int bit = wi * 32 + b;
                const uint32_t sc = s_score[(row + 1) * SP + bit + 4];
                dst[slot++] = (uint32_t)(ox0 + bit) | (sc << 16);
            }
            if (wi == MW - 1) s_rowcnt[row] = base + pre;
        }
    }
    __syncthreads();
    if (tid < y1 - y0) cnt_out[y0 - ORBX_EDGE + tid] = s_rowcnt[tid];
}

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
__device__ bool introselect_warp(Elem* v, int first, int last, int nth, int depth, int lane)
{
    while (last - first > 3) {
        if (depth == 0) { heap_select_fallback(v, first, nth, last, lane); return true; }
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
    return true;
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

constexpr int SEL_NT = 128;             // threads per CTA of the default instantiation
constexpr int SEL_NT_WIDE = 512;        // ... for frames above 0.6 Mpixel: level 0 holds tens of thousands of candidates there
constexpr int SEL_SMEM_ELEMS = 2048;
constexpr int SEL_PAR_MIN = 32;        // ranges up to this length are finished by one warp

struct SelShared {
    int warp_a[32], warp_b[32];            // one slot per warp of the widest instantiation
    int n, first, last, depth, ok;
};

// Whole-CTA KeyPointsFilter::retainBest(v, m).  All NT threads must call it.  PosT scratch lists Lp / Rp hold
// `len` positions each.  Returns the new length (valid on every thread); *flag |= 1 on the heap-select fallback.
template <typename PosT, int NT>
__device__ int retain_best_block(Elem* v, int len, int m, PosT* Lp, PosT* Rp, SelShared* sh, int* flag)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (m < 0 || len <= m) return len;
    if (m == 0) return 0;
    const int nth = m - 1;
    int first = 0, last = len, depth = 2 * (31 - __clz(len));
    bool ok = true, fallback = false;
    // ---- data-parallel Hoare passes while the range is long
    while (last - first > SEL_PAR_MIN) {
        if (depth == 0) { fallback = true; break; }          // depth budget spent: libstdc++ switches to __heap_select
        --depth;
        if (tid == 0) elem_swap(v, first, median3_pick(v, first + 1, first + (last - first) / 2, last - 1));
        __syncthreads();
        const float piv = v[first].response;
        const int lo = first + 1, n = last - lo;
        const int cs = (n + NT - 1) / NT;
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
        for (int i = 0; i < NT / 32; ++i) {
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
        for (int k = tid; k < mm; k += NT) cnt += ((int)Lp[k] < (int)Rp[k]);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
        if (lane == 0) sh->warp_a[wid] = cnt;                // safe: all reads of warp_a finished before the last barrier
        __syncthreads();
        int K = 0;
#pragma unroll
        for (int i = 0; i < NT / 32; ++i) K += sh->warp_a[i];
        for (int k = tid; k < K; k += NT) elem_swap(v, (int)Lp[k], (int)Rp[k]);
        int cut = 0x7fffffff;
        if (K < totL) cut = (int)Lp[K];
        if (K > 0) cut = min(cut, (int)Rp[K - 1]);
        __syncthreads();
        if (cut <= nth) first = cut; else last = cut;
    }
    // ---- finish with one warp: short-range introselect + insertion sort, then the std::partition tail
    if (wid == 0) {
        int res = m;
        if (fallback) heap_select_fallback(v, first, nth, last, lane);
        else ok = introselect_warp(v, first, last, nth, depth, lane);
        if (ok) res = partition_tail_warp(v, m, len, v[m - 1].response, lane);
        if (lane == 0) { sh->n = res; sh->ok = ok ? 1 : 0; }
    }
    __syncthreads();
    const int res = sh->n;
    if (!sh->ok) *flag |= 1;
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
template <int NT>
__device__ __forceinline__ void select_body(const Geom& g, const uint8_t* __restrict__ pyr, const uint32_t* __restrict__ rowcnt,
                                            const uint32_t* __restrict__ rowent, Elem* __restrict__ work, uint32_t* __restrict__ selpos,
                                            int* __restrict__ fincnt, int* __restrict__ status, int l, int f, SelSmem& sm)
{
    Elem* const s_v = sm.v;
    uint16_t* const s_pos = sm.pos;
    SelShared& sh = sm.sh;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const LevelGeom& L = g.L[l];
    Elem* gv = work + (size_t)f * g.ws_frame + L.ws_off;
    if (L.in_w <= 0 || L.in_h <= 0) { if (tid == 0) fincnt[f * g.nlevels + l] = 0; return; }
    const uint32_t* cnt = rowcnt + (size_t)f * g.cnt_frame + L.cnt_off;
    const uint32_t* ent = rowent + (size_t)f * g.ent_frame + L.ent_off;
    // ---- gather rows in raster order
    const int nr = L.in_h;
    const int rpt = (nr + NT - 1) / NT;
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
    for (int i = 0; i < NT / 32; ++i) { const int s = sh.warp_a[i]; if (i < wid) woff += s; total += s; }
    const int N = total;
    const bool in_smem = N <= SEL_SMEM_ELEMS;
    Elem* v = in_smem ? s_v : gv;
    {
        // Rows in groups of four: the first 128-bit chunk of each row's list (row lists are 32-byte aligned and most hold
        // fewer than four survivors) is requested for all four rows before any is consumed, so a thread's gather costs
        // about one memory round trip per group instead of one per entry.
        int o = woff + inc - mine;
        for (int r0 = rb; r0 < re; r0 += 4) {
            int cc[4];
            uint4 w4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) cc[k] = r0 + k < re ? (int)cnt[r0 + k] : 0;
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
                        const uint32_t w = e[i];
                        Elem el;
                        el.response = (float)(w >> 16);
                        el.pos = ypart | (w & 0xffffu);
                        v[o++] = el;
                    }
                }
            }
        }
    }
    __syncthreads();
    int flag = 0;
    uint32_t* gpos = selpos + 2 * ((size_t)f * g.ws_frame + L.ws_off);
    // ---- retainBest(2 n_l) on the FAST score
    const int n1 = in_smem ? retain_best_block<uint16_t, NT>(v, N, 2 * L.quota, s_pos, s_pos + SEL_SMEM_ELEMS, &sh, &flag)
                           : retain_best_block<uint32_t, NT>(v, N, 2 * L.quota, gpos, gpos + N, &sh, &flag);
    // ---- Harris on the unblurred level
    const uint8_t* img = pyr + (size_t)f * g.pyr_frame + L.img_off;
    for (int i = tid; i < n1; i += NT) {
        const uint32_t pos = v[i].pos;
        v[i].response = harris_response(img, L.pitch, (int)(pos & 0xffffu), (int)(pos >> 16));
    }
    __syncthreads();
    // ---- retainBest(n_l) on Harris
    const int n2 = in_smem ? retain_best_block<uint16_t, NT>(v, n1, L.quota, s_pos, s_pos + SEL_SMEM_ELEMS, &sh, &flag)
                           : retain_best_block<uint32_t, NT>(v, n1, L.quota, gpos, gpos + N, &sh, &flag);
    if (tid == 0) { fincnt[f * g.nlevels + l] = n2; if (flag) atomicOr(&status[f], flag); }
    if (v != gv) for (int i = tid; i < n2; i += NT) gv[i] = v[i];
}

// grid = (frames, levels): level-major dispatch, so the long level-0 CTAs of every frame start in the first wave and
// the short upper levels fill the tail
template <int NT>
__global__ void __launch_bounds__(NT, NT <= 128 ? 8 : 2) k_select(const __grid_constant__ Geom g, const uint8_t* __restrict__ pyr,
                                                   const uint32_t* __restrict__ rowcnt, const uint32_t* __restrict__ rowent,
                                                   Elem* __restrict__ work, uint32_t* __restrict__ selpos, int* __restrict__ fincnt,
                                                   int* __restrict__ status)
{
    __shared__ SelSmem sm;
    select_body<NT>(g, pyr, rowcnt, rowent, work, selpos, fincnt, status, blockIdx.y, blockIdx.x, sm);
}


// ------------------------------------------------------------------------------------------------ A.7 / A.9 scalar math
__device__ __forceinline__ float fast_atan2_deg(float y, float x)
{
    const float P1 = __int_as_float(0x4265226f), P3 = __int_as_float(0xc19556ee);
    const float P5 = __int_as_float(0x410e9fbf), P7 = __int_as_float(0xc0228ad9);
    const float eps = __int_as_float(0x25800000);            // (float)DBL_EPSILON
    const float ax = fabsf(x), ay = fabsf(y);
    float a, c, c2;
    if (ax >= ay) { c = __fdiv_rn(ay, __fadd_rn(ax, eps)); }
    else          { c = __fdiv_rn(ax, __fadd_rn(ay, eps)); }
    c2 = __fmul_rn(c, c);
    a = __fmul_rn(P7, c2); a = __fadd_rn(a, P5); a = __fmul_rn(a, c2); a = __fadd_rn(a, P3);
    a = __fmul_rn(a, c2);  a = __fadd_rn(a, P1); a = __fmul_rn(a, c);
    if (!(ax >= ay)) a = __fsub_rn(90.0f, a);
    if (x < 0.0f) a = __fsub_rn(180.0f, a);
    if (y < 0.0f) a = __fsub_rn(360.0f, a);
    return a;
}

// glibc 2.39 sinf/cosf restated in FP64 with separate roundings (SURVEY A.9); valid for |ang| < 120.
__device__ __forceinline__ float sin_poly_d(double x, double x2)
{
    const double S0 = -0x1.555545995a603p-3, S1 = 0x1.1107605230bc4p-7, S2 = -0x1.994eb3774cf24p-13;
    const double x3 = __dmul_rn(x, x2);
    const double s1 = __dadd_rn(S1, __dmul_rn(x2, S2));
    const double x7 = __dmul_rn(x3, x2);
    const double s = __dadd_rn(x, __dmul_rn(x3, S0));
    return (float)__dadd_rn(s, __dmul_rn(x7, s1));
}
__device__ __forceinline__ float cos_poly_d(double x2)
{
    const double C0 = 1.0, C1 = -0x1.ffffffd0c621cp-2, C2 = 0x1.55553e1068f19p-5, C3 = -0x1.6c087e89a359dp-10, C4 = 0x1.99343027bf8c3p-16;
    const double x4 = __dmul_rn(x2, x2);
    const double c2 = __dadd_rn(C3, __dmul_rn(x2, C4));
    const double c1 = __dadd_rn(C0, __dmul_rn(x2, C1));
    const double x6 = __dmul_rn(x4, x2);
    const double c = __dadd_rn(c1, __dmul_rn(x4, C2));
    return (float)__dadd_rn(c, __dmul_rn(x6, c2));
}
// glibc negates the polynomial's coefficients (cos) or its argument (sin) for the quadrant sign; round-to-nearest is
// sign-symmetric, so negating the float result is bit-identical and both polynomials are evaluated once, unsigned.
__device__ __forceinline__ void glibc_sincosf(float ang, float* sn, float* cs)
{
    const unsigned top = (__float_as_uint(ang) >> 20) & 0x7ffu;
    double x = (double)ang;
    if (top < ((0x3f490fdbu >> 20) & 0x7ffu)) {               // |ang| < pi/4 (top-12-bit compare, as glibc)
        if (top < ((0x39800000u >> 20) & 0x7ffu)) { *sn = ang; *cs = 1.0f; return; }   // |ang| < 2^-12
        const double x2 = __dmul_rn(x, x);
        *sn = sin_poly_d(x, x2);
        *cs = cos_poly_d(x2);
        return;
    }
    const double r = __dmul_rn(x, 0x1.45F306DC9C883p+23);
    const int n = (__double2int_rz(r) + 0x800000) >> 24;
    x = __dsub_rn(x, __dmul_rn((double)n, 0x1.921FB54442D18p0));
    const double x2 = __dmul_rn(x, x);
    const float ps = sin_poly_d(x, x2), pc = cos_poly_d(x2);
    const unsigned sneg = ((n & 3) == 1 || (n & 3) == 2) ? 0x80000000u : 0u;   // sign applied to the sine polynomial
    const unsigned cneg = (n & 2) ? 0x80000000u : 0u;                          // ... to the cosine polynomial
    const float s_ = __uint_as_float(__float_as_uint(ps) ^ sneg), c_ = __uint_as_float(__float_as_uint(pc) ^ cneg);
    if (n & 1) { *sn = c_; *cs = s_; }
    else       { *sn = s_; *cs = c_; }
}

// ------------------------------------------------------------------------------------------------ A.8 blur
// 7x7 sigma-2 Gaussian of every level in OpenCV's float sepFilter2D arithmetic (SURVEY A.8):
//   row pass   acc = F(k0*p[x-3]); acc = fma(p[x-3+i], k_i, acc), i = 1..6
//   col pass   acc = F(k3*r[y]);   acc = fma(F(r[y+j] + r[y-j]), k_{3+j}, acc), j = 1..3;  out = rint(acc)
// Only the region a descriptor can sample is produced: [12, w-13) x [13, h-13) (keypoints keep 31 px from the
// border, rBRIEF reaches 18).  One thread = 8 adjacent columns walked down a strip of rows with a 7-deep register
// window of row-pass values (rotated by unrolling, no moves), so every input byte is loaded once per thread and
// converted to float once (exactly: PRMT into the mantissa of 2^23, one FADD).  Work items (column group, strip)
// of a level are flattened so warps stay full on narrow levels.  No clamp is needed: the taps sum to < 1.
constexpr int BLUR_NT = 128;           // work items per CTA
constexpr int BLUR_LO = 12;            // first produced column (8-column groups start at 12 + 8q, so x0 - 4 is 8-byte aligned)


__device__ __forceinline__ float u8f(uint32_t w, uint32_t sel) { return __uint_as_float(__byte_perm(w, 0x4B000000u, sel)) - 8388608.0f; }

__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi)
{
    return (unsigned long long)__float_as_uint(lo) | ((unsigned long long)__float_as_uint(hi) << 32);
}
__device__ __forceinline__ unsigned long long f2_mul(unsigned long long a, unsigned long long b)
{
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long f2_add(unsigned long long a, unsigned long long b)
{
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long f2_fma(unsigned long long a, unsigned long long b, unsigned long long c)
{
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float f2_lo(unsigned long long v) { return __uint_as_float((unsigned)v); }
__device__ __forceinline__ float f2_hi(unsigned long long v) { return __uint_as_float((unsigned)(v >> 32)); }

// Packed-FP32 version: Blackwell's FFMA2 / FMUL2 / FADD2 do two IEEE-rounded FP32 operations per issue slot, so the
// thread's 8 columns are held as 4 packs (column m, column m + 4).  With that pairing every tap of the row pass reads
// an aligned register pair P(i) = (p[i], p[i+4]), i = 0..9, built once per source row straight from the loaded words
// (PRMT into the mantissa of 2^23, one FADD2 with -2^23 converts both halves exactly).  No mul feeds an add here (the
// pattern ptxas would contract): products feed FMA addends, sums feed FMA multiplicands.
constexpr int BLUR_DEPTH = 7;          // source rows in flight per thread (cp.async ring slots = the 7-row window)
template <int N> struct ic { static constexpr int value = N; };   // compile-time window slot
constexpr int BLUR_RING_BYTES = BLUR_DEPTH * BLUR_NT * 16;
// tile = index of the CTA's work inside the frame's blur tile list, f = frame, s_ring = BLUR_RING_BYTES of shared memory
__device__ __forceinline__ void blur_body(const Geom& g, const uint8_t* __restrict__ pyr, uint8_t* __restrict__ blur, int tile, int f, uint8_t* s_ring)
{
    int l = 0;
#pragma unroll 1
    for (int i = 1; i < g.nlevels; ++i) if (tile >= g.L[i].blur0) l = i;
    const LevelGeom& L = g.L[l];
    const int item = (tile - L.blur0) * BLUR_NT + threadIdx.x;
    const int strip = item / L.blur_cgs, cg = item - strip * L.blur_cgs;
    const int x0 = BLUR_LO + cg * 8;                                              // first of this thread's 8 columns
    const int rh = L.blur_rh;                                                     // strip height, a multiple of 7
    const int ys = 13 + strip * rh;                                               // first output row
    const int nout = min(rh, L.h - 13 - ys);                                      // output rows this strip really has
    if (tile - L.blur0 >= L.nblur || nout <= 0) return;
    const float k0 = __int_as_float(0x3d8fafb1), k1 = __int_as_float(0x3e06387e), k2 = __int_as_float(0x3e434a39), k3 = __int_as_float(0x3e5d4ae0);
    const unsigned long long K0 = f2_pack(k0, k0), K1 = f2_pack(k1, k1), K2 = f2_pack(k2, k2), K3 = f2_pack(k3, k3);
    const unsigned long long NEG23 = f2_pack(-8388608.0f, -8388608.0f), RND = f2_pack(12582912.0f, 12582912.0f);
    const uint8_t* src = pyr + (size_t)f * g.pyr_frame + L.img_off + (size_t)(ys - 3) * L.pitch + (x0 - 4);
    uint8_t* dst = blur + (size_t)f * g.pyr_frame + L.img_off + (size_t)ys * L.pitch + x0;
    unsigned long long w[4][7];
    // Source rows stream through a thread-private shared-memory ring filled by cp.async (LDGSTS): 7 rows are in flight
    // per thread with no register and -- the point -- no scoreboard cost (a warp has six scoreboards, so 14 register
    // loads in flight end up sharing them and the oldest load waits for the youngest).  A thread reads back only the
    // 16 bytes it copied itself, so cp.async.wait_group is all the synchronisation there is.  The ring has as many
    // slots as the row window (slot of source row r = r % 7, a compile-time index in the unrolled loop), every strip
    // runs the same rh + 6 source rows (rows past a short last strip only feed outputs whose stores are masked; the
    // pyramid buffer carries slack for them), and the first 6 rows -- which produce no output yet -- are a prologue: the
    // steady-state body has no per-row bounds checks at all.
    const unsigned ring = (unsigned)__cvta_generic_to_shared(s_ring) + threadIdx.x * 16u;
#pragma unroll
    for (int d = 0; d < 7; ++d) {
        cp_async_8(ring + d * (BLUR_NT * 16u), src + (size_t)d * L.pitch);
        cp_async_8(ring + d * (BLUR_NT * 16u) + 8u, src + (size_t)d * L.pitch + 8);
        cp_async_commit();
    }
    src += (size_t)7 * L.pitch;
    // one source row in window slot K: wait, read it back, refill the slot with the row 7 further down, row pass
    auto row_pass = [&](auto kc) {
        constexpr int K = decltype(kc)::value;
        cp_async_wait<6>();
        const unsigned sa = ring + K * (BLUR_NT * 16u);
        const uint4 ab = lds_v4(sa);
        cp_async_8(sa, src); cp_async_8(sa + 8u, src + 8);
        cp_async_commit();
        src += L.pitch;
        const uint32_t W[4] = {ab.x, ab.y, ab.z, ab.w};                            // bytes x0-4 .. x0+11; pixel i = x0-3+i is byte i+1
        unsigned long long P[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) {
            const uint32_t lo = __byte_perm(W[(i + 1) >> 2], 0x4B000000u, 0x7650u | ((i + 1) & 3));
            const uint32_t hi = __byte_perm(W[(i + 5) >> 2], 0x4B000000u, 0x7650u | ((i + 5) & 3));
            P[i] = f2_add((unsigned long long)lo | ((unsigned long long)hi << 32), NEG23);
        }
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            unsigned long long acc = f2_mul(K0, P[m]);
            acc = f2_fma(P[m + 1], K1, acc); acc = f2_fma(P[m + 2], K2, acc); acc = f2_fma(P[m + 3], K3, acc);
            acc = f2_fma(P[m + 4], K2, acc); acc = f2_fma(P[m + 5], K1, acc); acc = f2_fma(P[m + 6], K0, acc);
            w[m][K] = acc;
        }
    };
    // output row centred 3 rows above the newest source row (window slot K)
    auto col_pass = [&](auto kc, bool store) {
        constexpr int K = decltype(kc)::value;
        uint32_t q[8];
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            unsigned long long o = f2_mul(K3, w[m][(K + 4) % 7]);                                   // row r-3
            o = f2_fma(f2_add(w[m][(K + 5) % 7], w[m][(K + 3) % 7]), K2, o);                        // r-2, r-4
            o = f2_fma(f2_add(w[m][(K + 6) % 7], w[m][(K + 2) % 7]), K1, o);                        // r-1, r-5
            o = f2_fma(f2_add(w[m][K], w[m][(K + 1) % 7]), K0, o);                                  // r,   r-6
            const unsigned long long rb = f2_add(o, RND);                                           // rint via 1.5 * 2^23
            q[m] = (uint32_t)rb; q[m + 4] = (uint32_t)(rb >> 32);
        }
        const uint32_t o0 = __byte_perm(__byte_perm(q[0], q[1], 0x0040), __byte_perm(q[2], q[3], 0x0040), 0x5410);
        const uint32_t o1 = __byte_perm(__byte_perm(q[4], q[5], 0x0040), __byte_perm(q[6], q[7], 0x0040), 0x5410);
        if (store) {
            reinterpret_cast<uint32_t*>(dst)[0] = o0;                                               // x0 = 4 mod 8: two word stores
            reinterpret_cast<uint32_t*>(dst)[1] = o1;
        }
        dst += L.pitch;
    };
    row_pass(ic<0>{}); row_pass(ic<1>{}); row_pass(ic<2>{}); row_pass(ic<3>{}); row_pass(ic<4>{}); row_pass(ic<5>{});
    int j = 0;                                                                     // output row inside the strip
#pragma unroll 1
    for (int grp = 0; grp < rh; grp += 7) {                                       // source rows 6 + grp .. 12 + grp: window slots 6, 0, 1, .., 5
        row_pass(ic<6>{}); col_pass(ic<6>{}, j + 0 < nout);
        row_pass(ic<0>{}); col_pass(ic<0>{}, j + 1 < nout);
        row_pass(ic<1>{}); col_pass(ic<1>{}, j + 2 < nout);
        row_pass(ic<2>{}); col_pass(ic<2>{}, j + 3 < nout);
        row_pass(ic<3>{}); col_pass(ic<3>{}, j + 4 < nout);
        row_pass(ic<4>{}); col_pass(ic<4>{}, j + 5 < nout);
        row_pass(ic<5>{}); col_pass(ic<5>{}, j + 6 < nout);
        j += 7;
    }
    cp_async_wait<0>();                                                            // nothing of this thread may still land in shared memory after it exits
}

__global__ void __launch_bounds__(BLUR_NT) k_blur(const __grid_constant__ Geom g, const uint8_t* __restrict__ pyr, uint8_t* __restrict__ blur)
{
    __shared__ __align__(16) uint8_t s_ring[BLUR_RING_BYTES];
    blur_body(g, pyr, blur, blockIdx.x, blockIdx.y, s_ring);
}

}  // namespace orbx
