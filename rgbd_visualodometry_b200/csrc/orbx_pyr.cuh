// orbx_pyr.cuh -- A.1 BGR -> gray and A.2 INTER_LINEAR_EXACT pyramid (cv::cvtColor and the cv::resize inside
// cv::ORB::detectAndCompute, src/frontend.cpp:153), sm_100a.
//
//   k_gray          A.1   BGR -> gray (level 0)                         HBM-bound, 16 px / thread
//   k_pyr_down      A.2   level l from level l-1, CTA-cooperative       thread = 8 output columns x 16 rows, source rows streamed by cp.async
//   k_pyr_tma       A.2   level l from level l-1, warp-private          warp = 128 output columns x a stack of strips, source rows by TMA
//
// k_pyr_tma (large launches):
//
//   dst(x, y) = (h0 * (256 - cy) + h1 * cy + 32768) >> 16,   h = p[i0] * (256 - cx) + p[i0 + 1] * cx     (8.8 taps, host tables)
//
// Unit of work: one WARP owns a column tile of 128 output columns (lane = 4 adjacent columns) and walks a few strips of PT_RH
// output rows down it.  The source rows a strip needs arrive as ONE cp.async.bulk.tensor box (TMA; the box dimensions are fitted
// per level on the host and baked into the level's tensor map), double-buffered: the box of the next strip lands while the
// current one is computed.  No block barrier, no per-thread copy instructions.
//   horizontal pass  the lane's 4 outputs read at most 7 consecutive source bytes: three aligned 32-bit shared loads and two
//                    funnel shifts put them at the bottom of a 64-bit window; per output ONE PRMT gathers (p0, p0, p1, p1) and ONE
//                    IDP.4A multiplies by the tap weights split into bytes (c0 = a + b, c1 = c + d, each <= 128): exact.
//   vertical pass    the horizontal pass of a source row is taken once and reused by the next output row (ping-pong registers);
//                    two IMADs per pixel (h <= 255 * 256, so byte 2 of the 24-bit sum IS the rounded pixel) and three PRMTs per quad.
// ALU pipe (SHF, PRMT) and FMA pipe (IDP, IMAD) carry about the same number of instructions.
// Levels whose scale factor makes a lane's 4 outputs span more than 7 source bytes, or whose boxes would not fit, keep the
// register-window kernel k_pyr_down.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "orbx_geom.h"
#include "orbx_device.cuh"

namespace orbx {

__device__ __forceinline__ void cp_async_4(unsigned dst, const void* src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(dst), "l"(src) : "memory"); }

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

// ------------------------------------------------------------------------------------------------ A.2 pyramid, TMA-fed
constexpr int PT_RH = 16;                // output rows per strip
constexpr int PT_CW = 128;               // output columns per column tile
constexpr int PT_NWARP = 4;              // warps per CTA (independent units)

struct PyrMaps { CUtensorMap m[ORBX_LEVELS_MAX]; };   // m[l]: SOURCE level l-1 as (x, y, frame), box pt_bw x pt_bh x 1 of destination level l

__host__ __device__ inline int pt_buf_bytes(int bw, int bh) { return (bw * bh + 16 + 127) / 128 * 128; }   // + 16: a lane's third word may lie past the last row
__host__ __device__ inline int pt_warp_bytes(int bw, int bh) { return 2 * pt_buf_bytes(bw, bh) + 128; }   // two boxes + two mbarriers

// (min 6 CTAs per SM stated: ptxas then spends 70 instead of 56 registers per thread and the seven levels take 0.163 instead of 0.175 ms)
__global__ void __launch_bounds__(PT_NWARP * 32, 6) k_pyr_tma(const __grid_constant__ Geom g, const __grid_constant__ CUtensorMap map, int l, int f0,
                                                           uint8_t* __restrict__ pyr, const uint32_t* __restrict__ tabs, int* __restrict__ status)
{
    extern __shared__ __align__(128) uint8_t pt_smem[];
    const LevelGeom& D = g.L[l];
    const LevelGeom& S = g.L[l - 1];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int task = blockIdx.x * PT_NWARP + wid;
    if (task >= D.pt_ntask) return;                          // warps are independent: no block-level synchronisation anywhere
    const int cx = task % D.pt_ncx, sg = task / D.pt_ncx;
    const int nstrips = (D.h + PT_RH - 1) / PT_RH;
    const int strip0 = sg * D.pt_k, strip1 = min(strip0 + D.pt_k, nstrips);
    const int f = blockIdx.y;
    const int bw = D.pt_bw, bh = D.pt_bh;
    const unsigned bufb = (unsigned)pt_buf_bytes(bw, bh);
    const unsigned base_s = (((unsigned)__cvta_generic_to_shared(pt_smem) + 127u) & ~127u) + (unsigned)wid * (unsigned)pt_warp_bytes(bw, bh);
    const unsigned bar_s = base_s + 2u * bufb;
    const uint32_t* xtab = tabs + D.xtab;
    const uint32_t* ytab = tabs + D.ytab;
    const int x = cx * PT_CW + 4 * lane;
    const int X0 = (int)(__ldg(xtab + cx * PT_CW) & 0xffffu) & ~15;      // first source column of the warp's boxes (TMA: 16-byte granularity)

    // ---- per-lane constants of the horizontal pass
    unsigned sel[4], wgt[4], a_off, sh;
    {
        const bool live = x < D.w;
        const int b0 = live ? (int)(__ldg(xtab + x) & 0xffffu) : X0;     // first source byte the lane needs
        const int rel = b0 - X0;
        a_off = (unsigned)(rel & ~3);
        sh = (unsigned)(rel & 3) * 8u;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            unsigned s = 0x1100u, w = 0u;                                // columns past the level's width: weights 0 -> pixel 0 (row padding stays zero)
            if (x + k < D.w) {
                const uint32_t t = __ldg(xtab + x + k);
                const unsigned off = (t & 0xffffu) - (unsigned)b0;       // 0 .. 6
                const unsigned c1 = t >> 16, c0 = 256u - c1;
                const unsigned c0a = min(c0, 128u), c1a = min(c1, 128u);
                s = off | (off << 4) | ((off + 1u) << 8) | ((off + 1u) << 12);
                w = c0a | ((c0 - c0a) << 8) | (c1a << 16) | ((c1 - c1a) << 24);
            }
            sel[k] = s; wgt[k] = w;
        }
    }
    if (lane == 0) {
        mbar_init(bar_s, 1);
        mbar_init(bar_s + 8u, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    auto request = [&](int strip, unsigned b) {
        if (lane == 0) {
            const int s_first = (int)(__ldg(ytab + strip * PT_RH) & 0xffffu);
            mbar_expect_tx(bar_s + 8u * b, (unsigned)(bw * bh));
            tma_load_tile_3d(base_s + b * bufb, &map, X0, s_first, f0 + f, bar_s + 8u * b);
        }
    };
    // horizontal pass of the box row whose (lane-adjusted) shared address is ad
    auto hpass = [&](unsigned ad, unsigned* h) {
        const unsigned w0 = lds_u32(ad), w1 = lds_u32(ad + 4u), w2 = lds_u32(ad + 8u);
        const unsigned lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
#pragma unroll
        for (int k = 0; k < 4; ++k) h[k] = __dp4a(__byte_perm(lo, hi, sel[k]), wgt[k], 0u);
    };

    request(strip0, 0u);
    unsigned par0 = 0u, par1 = 0u;
    const int pitch = D.pitch, sh1 = S.h - 1;
    const bool store = x < pitch;
    uint8_t* const dst0 = pyr + (size_t)(f0 + f) * g.pyr_frame + D.img_off + x;   // (pyr is the whole buffer: TMA coordinates are absolute frames)
#pragma unroll 1
    for (int strip = strip0; strip < strip1; ++strip) {
        const unsigned b = (unsigned)(strip - strip0) & 1u;
        if (strip + 1 < strip1) request(strip + 1, b ^ 1u);              // the other box was consumed before the __syncwarp() that ended the last strip
        const unsigned buf_s = base_s + b * bufb;
        if (!mbar_wait(bar_s + 8u * b, b ? par1 : par0)) { if (lane == 0) atomicOr(&status[f], 2); return; }
        if (b) par1 ^= 1u; else par0 ^= 1u;
        const int ys = strip * PT_RH, nr = min(PT_RH, D.h - ys);
        // vertical taps of the strip's rows: lane r holds row ys + r, handed out by one shuffle per row
        const uint32_t ty_all = lane < nr ? __ldg(ytab + ys + lane) : 0u;
        const int s_first = (int)(__shfl_sync(0xffffffffu, ty_all, 0) & 0xffffu);
        const unsigned row0_s = buf_s + a_off - (unsigned)(s_first * bw);  // box row of source row s at row0_s + s * bw
        int have = -1;                                                   // source row whose horizontal pass sits in the "top" registers
        unsigned hA[4], hB[4];
        uint8_t* dst = dst0 + (size_t)ys * pitch;
        // one output row: T = horizontal pass of its upper source row (already there unless the mapping skipped a row), N = lower
        auto row = [&](int r, unsigned* T, unsigned* N) {
            const uint32_t ty = __shfl_sync(0xffffffffu, ty_all, r);
            const int s0 = (int)(ty & 0xffffu), s1 = min(s0 + 1, sh1);
            const unsigned cy1 = ty >> 16, cy0 = 256u - cy1;
            if (s0 != have) hpass(row0_s + (unsigned)(s0 * bw), T);      // warp-uniform
            hpass(row0_s + (unsigned)(s1 * bw), N);                      // (the image's bottom row clamps: s1 == s0, taken twice -- no branch)
            unsigned v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = T[k] * cy0 + (N[k] * cy1 + 32768u);
            if (store) *reinterpret_cast<uint32_t*>(dst) = __byte_perm(__byte_perm(v[0], v[1], 0x0062), __byte_perm(v[2], v[3], 0x0062), 0x5410);
            dst += pitch;
            have = s1;
        };
        int r = 0;
#pragma unroll 1
        for (; r + 1 < nr; r += 2) { row(r, hA, hB); row(r + 1, hB, hA); }   // ping-pong without register copies
        if (r < nr) row(r, hA, hB);
        __syncwarp();                                                    // every lane is done with this box
    }
}

}  // namespace orbx
