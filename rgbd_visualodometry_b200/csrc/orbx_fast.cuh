// orbx_fast.cuh -- A.3 FAST-9/16 score + 3x3 NMS (the detector inside cv::ORB::detectAndCompute, src/frontend.cpp:153),
// sm_100a.  Two kernels, identical results: k_fast_bands (CTA-cooperative, small launches) and k_fast_warp (WARP-PRIVATE
// tiles fed by TMA: no block barrier anywhere in the kernel), described here.
//
// Unit of work: one WARP owns one band of FW_R inner rows of one level of one frame and walks it left to right in chunks of
// FW_CW output columns, so every row's survivors leave in x order and the per-row lists concatenate to OpenCV's raster
// order (same output format as before: rowcnt / rowent, consumed by k_select).  Only the region that can survive the
// 31-px border filter is evaluated (SURVEY A.10).
//
// Per chunk the warp's u8 image tile (FW_TR rows x FW_TP bytes, halo included) arrives by ONE cp.async.bulk.tensor (TMA, 3-D
// tensor map (x, y, frame) per level, box FW_TP x FW_TR x 1, completion on the warp's mbarrier): no load instructions, no
// widening pass, no alignment arithmetic beyond the 16-byte column granularity TMA demands.  The tile of the next chunk is
// requested as soon as the last pixel of the current one has been scored and lands under the NMS / list phases.
//
//   phase A   every pixel, in BYTES: |c - n|, |c - s|, |c - e|, |c - w| with VABSDIFF4.U8 (4 pixels per instruction),
//             pass iff (max(|c-n|, |c-s|) > t) & (max(|c-e|, |c-w|) > t) -- the polarity-blind form of the 4-compass-point test (any
//             9-arc holds one of each opposite pair); threshold by carry-free byte arithmetic.  A lane's quad with any passing pixel
//             becomes one entry of the warp's quad queue (one ballot per row).
//   phase A2  32 queued quads at a time: polarity-AWARE test of the two diagonal opposite pairs (u16x2 VIMNMX); a surviving
//             pixel becomes a pixel entry that carries the only polarity it can still be a corner of (both -> two entries).
//   phase B   64 queued pixels at a time, TWO per lane: the 16 circle pixels of both candidates are packed into the halves
//             of u16x2 words, complemented for the "brighter" polarity (f(p) = 255 - p) by the integer FMAs that pack them, so ONE
//             sliding-max network (VIMNMX3.U16x2) yields min over the 16 arcs of max over the arc for both candidates:
//             score = f(c) - that - 1, corner iff > t.  Scores go to the warp's score tile, corners inside the output region to
//             its NMS queue.
//   phase C   3x3 NMS (strict >) of the queued corners on the score tile -> per-row bit masks
//   phase D   ordered extraction of the bit masks -> global per-row lists
// The queues are LIFO and bounded: A runs A2 as soon as 32 quads are waiting, A2 runs B as soon as 64 pixels are waiting, so B
// and A2 always work on full batches except for one drain per tile, and shared memory per warp stays under 8 KB.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "orbx_geom.h"
#include "orbx_device.cuh"

namespace orbx {

__device__ __forceinline__ unsigned vmin2(unsigned a, unsigned b) { return __vminu2(a, b); }
__device__ __forceinline__ unsigned vmax2(unsigned a, unsigned b) { return __vmaxu2(a, b); }
__device__ __forceinline__ unsigned vmax3(unsigned a, unsigned b, unsigned c) { return __vimax3_u16x2(a, b, c); }
__device__ __forceinline__ unsigned vmin3(unsigned a, unsigned b, unsigned c) { return __vimin3_u16x2(a, b, c); }
__device__ __forceinline__ uint2 lds_v2(unsigned addr)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ unsigned lds_u16(unsigned addr) { unsigned short v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr) : "memory"); return v; }
__device__ __forceinline__ void sts_u16(unsigned addr, unsigned v) { asm volatile("st.shared.u16 [%0], %1;" :: "r"(addr), "h"((unsigned short)v) : "memory"); }

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

// ------------------------------------------------------------------------------------------------ A.3 FAST + NMS, TMA-fed
constexpr int FW_R = 16;                 // output rows per band
constexpr int FW_CW = 124;               // output columns per chunk (score columns 3 .. 126 of 128)
constexpr int FW_TP = 160;               // image tile pitch in bytes = TMA box width (16-byte aligned origin <= ox0 - 7, + 4 + 128 + 3)
constexpr int FW_TR = FW_R + 8;          // image tile rows
constexpr int FW_SR = FW_R + 2;          // score tile rows
constexpr int FW_SP = 128;               // score tile pitch = pixels evaluated per row (32 lanes x 4)
constexpr int FW_QQ = 64;                // quad queue capacity (entries): < 32 waiting + <= 32 per row
constexpr int FW_PQ = 320;               // pixel queue: < 64 waiting + <= 32 quads x 4 pixels x 2 polarities per A2 batch
constexpr int FW_CQ = 256;               // NMS queue; on overflow the tile falls back to a dense NMS scan
constexpr int FW_OFF_SCORE = FW_TP * FW_TR;
constexpr int FW_OFF_QQ = FW_OFF_SCORE + FW_SR * FW_SP;
constexpr int FW_OFF_PQ = FW_OFF_QQ + FW_QQ * 2;
constexpr int FW_OFF_CQ = FW_OFF_PQ + FW_PQ * 2;
constexpr int FW_OFF_MASK = FW_OFF_CQ + FW_CQ * 2;
constexpr int FW_OFF_ROWCNT = FW_OFF_MASK + FW_R * 4 * 4;
constexpr int FW_OFF_BAR = FW_OFF_ROWCNT + FW_R * 4;
constexpr int FW_WARP_BYTES = (FW_OFF_BAR + 8 + 127) / 128 * 128;
constexpr int FW_CLR = (FW_SR * FW_SP / 16 + 31) / 32;   // 128-bit stores per lane that clear the score tile
static_assert(FW_CLR * 32 * 16 <= FW_OFF_CQ - FW_OFF_SCORE, "the score-tile clear may only spill into the (empty) quad / pixel queues");
static_assert(FW_OFF_SCORE % 16 == 0 && FW_OFF_MASK % 4 == 0 && FW_OFF_BAR % 8 == 0, "layout");

struct FastMaps { CUtensorMap m[ORBX_LEVELS_MAX]; };   // one (x, y, frame) u8 tensor map per pyramid level

template <int NWARP>
__global__ void __launch_bounds__(NWARP * 32, 28 / NWARP) k_fast_warp(const __grid_constant__ Geom g, const __grid_constant__ FastMaps maps, int f0,
                                                          int band_lo, int band_hi, uint32_t* __restrict__ rowcnt, uint32_t* __restrict__ rowent, int* __restrict__ status)
{
    extern __shared__ __align__(128) uint8_t fw_smem[];
    constexpr int T = ORBX_FAST_T;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned lt = lanemask_lt();
    const int f = blockIdx.y;
    const int gb = band_lo + blockIdx.x * NWARP + wid;       // band index inside the frame; this launch covers bands [band_lo, band_hi)
    if (gb >= band_hi) return;                               // (no block-level synchronisation anywhere: warps are independent)
    int l = 0;
#pragma unroll 1
    for (int i = 1; i < g.nlevels; ++i) if (gb >= g.L[i].band0) l = i;
    const LevelGeom& L = g.L[l];
    const int band = gb - L.band0;
    if (band >= L.nbands) return;
    const int y0 = ORBX_EDGE + band * FW_R;
    const int y1 = min(y0 + FW_R, L.h - ORBX_EDGE);         // output rows [y0, y1)
    const int nrows = y1 - y0, nsr = nrows + 2;
    const int xend = L.w - ORBX_EDGE;                       // output cols [31, xend)
    uint32_t* cnt_out = rowcnt + (size_t)f * g.cnt_frame + L.cnt_off;
    uint32_t* ent_out = rowent + (size_t)f * g.ent_frame + L.ent_off;
    const CUtensorMap* map = &maps.m[l];

    const unsigned base_s = (((unsigned)__cvta_generic_to_shared(fw_smem) + 127u) & ~127u) + (unsigned)wid * FW_WARP_BYTES;   // TMA destinations: 128-byte aligned
    const unsigned img_s = base_s, score_s = base_s + FW_OFF_SCORE, qq_s = base_s + FW_OFF_QQ, pq_s = base_s + FW_OFF_PQ;
    const unsigned cq_s = base_s + FW_OFF_CQ, mask_s = base_s + FW_OFF_MASK, rcnt_s = base_s + FW_OFF_ROWCNT, bar_s = base_s + FW_OFF_BAR;

    if (lane == 0) {
        mbar_init(bar_s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (lane < FW_R) asm volatile("st.shared.u32 [%0], %1;" :: "r"(rcnt_s + 4u * lane), "r"(0u) : "memory");
    asm volatile("st.shared.u32 [%0], %1;" :: "r"(mask_s + 4u * lane), "r"(0u) : "memory");
    asm volatile("st.shared.u32 [%0], %1;" :: "r"(mask_s + 128u + 4u * lane), "r"(0u) : "memory");
    __syncwarp();
    // chunk k: output columns [ox0, ox1), ox0 = 31 + 124 k; score column sx <-> x = ox0 - 3 + sx; tile byte of score column sx in
    // tile row ty: ty * FW_TP + xo + 4 + sx, where the tile's first column X0 = (ox0 - 7) & ~15 and xo = ox0 - 7 - X0 (0, 4, 8, 12:
    // a lane's quad is one aligned word); tile row of score row sy: sy + 3 (tile row 0 = image row y0 - 4)
    auto request = [&](int ox0) {
        if (lane == 0) {
            mbar_expect_tx(bar_s, FW_TP * FW_TR);
            tma_load_tile_3d(img_s, map, (ox0 - 7) & ~15, y0 - 4, f0 + f, bar_s);
        }
    };
    request(ORBX_EDGE);
    unsigned phase = 0;
    int overflow_any = 0;

#pragma unroll 1
    for (int ox0 = ORBX_EDGE; ox0 < xend; ox0 += FW_CW) {
        const int ncols = min(FW_CW, xend - ox0);
        const int need = ncols + 4;                          // score columns that matter: sx = 0 .. ncols + 3
        const unsigned xo = (unsigned)((ox0 - 7) & 15);
        const unsigned quad0_s = img_s + xo + 4u;            // tile byte of score column 0 in tile row 0
        // ---- clear the score tile: 160 x 16 B (the 16 x 16 B past its end fall into the quad / pixel queues, empty right now)
#pragma unroll
        for (int i = 0; i < FW_CLR; ++i)
            asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" :: "r"(score_s + 16u * (unsigned)(i * 32 + lane)), "r"(0u) : "memory");
        __syncwarp();
        if (!mbar_wait(bar_s, phase)) { if (lane == 0) atomicOr(&status[f], 2); return; }
        phase ^= 1u;

        int nq = 0, np = 0, cn = 0, overflow = 0;
        const int sx_hi = 3 + ncols;                         // corners that belong to this chunk: 3 <= sx < sx_hi, 1 <= sy <= nrows

        // ---- phase B on pixel entries [first, first + cnt): two per lane (lane, lane + 32)
        auto phaseB = [&](int first, int cnt) {
            unsigned ea = 0, eb = 0;
            const bool va = lane < cnt, vb = lane + 32 < cnt;
            if (va) ea = lds_u16(pq_s + 2u * (unsigned)(first + lane));
            if (vb) eb = lds_u16(pq_s + 2u * (unsigned)(first + lane + 32));
            const unsigned sya = (ea >> 8) & 31u, sxa = ea & 127u, syb = (eb >> 8) & 31u, sxb = eb & 127u;
            const unsigned ca = quad0_s + (sya + 3u) * FW_TP + sxa, cb = quad0_s + (syb + 3u) * FW_TP + sxb;
            // f(p) = p (candidate of the "darker arc" polarity) or 255 - p ("brighter arc"): V = fa(pa) | fb(pb) << 16 by two IMADs
            const unsigned ma = (ea & 0x8000u) ? 0xFFFFFFFFu : 1u, mb = (eb & 0x8000u) ? 0xFFFF0000u : 0x00010000u;
            const unsigned add = ((ea & 0x8000u) ? 255u : 0u) | ((eb & 0x8000u) ? (255u << 16) : 0u);
            unsigned q[16];
#define ORBX_PK(k, dx, dy) q[k] = lds_u8(cb + ((dy) * FW_TP + (dx))) * mb + (lds_u8(ca + ((dy) * FW_TP + (dx))) * ma + add)
            ORBX_PK(0, 0, 3);   ORBX_PK(1, 1, 3);   ORBX_PK(2, 2, 2);    ORBX_PK(3, 3, 1);
            ORBX_PK(4, 3, 0);   ORBX_PK(5, 3, -1);  ORBX_PK(6, 2, -2);   ORBX_PK(7, 1, -3);
            ORBX_PK(8, 0, -3);  ORBX_PK(9, -1, -3); ORBX_PK(10, -2, -2); ORBX_PK(11, -3, -1);
            ORBX_PK(12, -3, 0); ORBX_PK(13, -3, 1); ORBX_PK(14, -2, 2);  ORBX_PK(15, -1, 3);
            const unsigned vc = lds_u8(cb) * mb + (lds_u8(ca) * ma + add);
#undef ORBX_PK
            unsigned m3[16], m9[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) m3[k] = vmax3(q[k], q[(k + 1) & 15], q[(k + 2) & 15]);
#pragma unroll
            for (int k = 0; k < 16; ++k) m9[k] = vmax3(m3[k], m3[(k + 3) & 15], m3[(k + 6) & 15]);
            const unsigned mm = vmin3(vmin3(vmin3(m9[0], m9[1], m9[2]), vmin3(m9[3], m9[4], m9[5]), vmin3(m9[6], m9[7], m9[8])),
                                      vmin3(vmin3(m9[9], m9[10], m9[11]), vmin3(m9[12], m9[13], m9[14]), m9[15]),
                                      0xFFFFFFFFu);
            const int sca = (int)(vc & 0xffffu) - (int)(mm & 0xffffu), scb = (int)(vc >> 16) - (int)(mm >> 16);
            bool cora = false, corb = false;
            if (va && sca > T) {
                sts_u8(score_s + sya * FW_SP + sxa, (unsigned)(sca - 1));
                cora = (int)sxa >= 3 && (int)sxa < sx_hi && sya - 1u < (unsigned)nrows;
            }
            if (vb && scb > T) {
                sts_u8(score_s + syb * FW_SP + sxb, (unsigned)(scb - 1));
                corb = (int)sxb >= 3 && (int)sxb < sx_hi && syb - 1u < (unsigned)nrows;
            }
            const unsigned ba = __ballot_sync(0xffffffffu, cora), bb = __ballot_sync(0xffffffffu, corb);
            const int na = __popc(ba), nb = __popc(bb);
            if (cn + na + nb > FW_CQ) overflow = 1;          // warp-uniform; the tile's NMS then scans the score tile instead
            else {
                if (cora) sts_u16(cq_s + 2u * (unsigned)(cn + __popc(ba & lt)), ea & 0x1FFFu);
                if (corb) sts_u16(cq_s + 2u * (unsigned)(cn + na + __popc(bb & lt)), eb & 0x1FFFu);
                cn += na + nb;
            }
        };

        // ---- phase A2 on the cnt quad entries at shared address first_s: diagonal pairs, polarity aware; pixel entries pol << 15 | sy << 8 | sx
        auto phaseA2 = [&](unsigned first_s, int cnt) {
            constexpr unsigned K = ((511u - T) << 16) | (511u - T);
            unsigned m8 = 0, ent = 0;
            if (lane < cnt) {
                const unsigned e = lds_u16(first_s + 2u * (unsigned)lane);
                const unsigned sy = e >> 9, q4 = (e >> 2) & 0x7Cu;               // 4 * quad column
                const unsigned a = quad0_s + (sy + 3u) * FW_TP + q4;
                const unsigned up = a - 2 * FW_TP, dn = a + 2 * FW_TP;
                const unsigned c = lds_u32(a);
                const unsigned u0 = lds_u32(up - 4), u1 = lds_u32(up), u2 = lds_u32(up + 4);
                const unsigned d0 = lds_u32(dn - 4), d1 = lds_u32(dn), d2 = lds_u32(dn + 4);
                const unsigned NW = __byte_perm(u0, u1, 0x5432), NE = __byte_perm(u1, u2, 0x5432);   // columns x - 2 / x + 2 of row y - 2
                const unsigned SW = __byte_perm(d0, d1, 0x5432), SE = __byte_perm(d1, d2, 0x5432);   // ... of row y + 2
                unsigned md[2], mb[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const unsigned sel = h ? 0x4342u : 0x4140u;                  // pixels (2, 3) / (0, 1) widened to u16x2
                    const unsigned ch = __byte_perm(c, 0, sel), nw = __byte_perm(NW, 0, sel), ne = __byte_perm(NE, 0, sel);
                    const unsigned sw = __byte_perm(SW, 0, sel), se = __byte_perm(SE, 0, sel);
                    const unsigned D = vmax2(vmin2(se, nw), vmin2(ne, sw));      // a darker pixel in each pair:    c - D > t
                    const unsigned Bm = vmin2(vmax2(se, nw), vmax2(ne, sw));     // a brighter pixel in each pair:  Bm - c > t
                    md[h] = ch + K - D;                                          // bits 9 / 25 = pass flags of the half's two pixels
                    mb[h] = Bm + K - ch;
                }
                // natural pixel order: bits 9, 25 of half 0 and (moved up two) 11, 27 of half 1, folded to bits 9 .. 12
                const unsigned pd = (md[0] & 0x02000200u) | ((md[1] << 2) & 0x08000800u);
                const unsigned pb = (mb[0] & 0x02000200u) | ((mb[1] << 2) & 0x08000800u);
                const unsigned fd = ((pd | (pd >> 15)) >> 9) & e & 15u, fb = ((pb | (pb >> 15)) >> 9) & e & 15u;
                m8 = fd | (fb << 4);
                ent = (sy << 8) | q4;
            }
            const int mine = __popc(m8);
            int inc = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
            const int total = __shfl_sync(0xffffffffu, inc, 31);
            unsigned sa = pq_s + 2u * (unsigned)(np + inc - mine);
#pragma unroll
            for (int b = 0; b < 8; ++b)
                if (m8 & (1u << b)) { sts_u16(sa, ent + (unsigned)(b & 3) + ((b & 4) ? 0x8000u : 0u)); sa += 2u; }
            np += total;
            __syncwarp();
            while (np >= 64) { phaseB(np - 64, 64); np -= 64; __syncwarp(); }
        };

        // ---- phase A: one score row (128 pixels) per step
        {
            constexpr unsigned M7 = 0x7f7f7f7fu, KT = (127u - T) * 0x01010101u;
            unsigned livemask = 4 * lane < need ? 0x80808080u : 0u;            // lanes past the chunk's last needed column never flag
            unsigned qq_full = qq_s + 64u;
            livemask = __shfl_sync(0xffffffffu, livemask, lane);               // (identity shuffles: opaque to ptxas, which otherwise
            qq_full = __shfl_sync(0xffffffffu, qq_full, lane);                 //  rematerialises both values in every row of the loop)
            unsigned a = quad0_s + 3u * FW_TP + 4u * lane;
            unsigned ent = (unsigned)lane << 4;                                // quad entry: sy << 9 | quad column << 4 | pixel flags
            unsigned qt = qq_s;                                                // byte address of the quad queue's tail
#pragma unroll 2
            for (int sy = 0; sy < nsr; ++sy, a += FW_TP, ent += 512u) {
                const unsigned c = lds_u32(a), pv = lds_u32(a - 4), nx = lds_u32(a + 4), n = lds_u32(a - 3 * FW_TP), s = lds_u32(a + 3 * FW_TP);
                const unsigned e = __byte_perm(c, nx, 0x6543), w = __byte_perm(pv, c, 0x4321);
                const unsigned dn = __vabsdiffu4(n, c), ds = __vabsdiffu4(s, c), de = __vabsdiffu4(e, c), dw = __vabsdiffu4(w, c);
                // bit 7 of ((d & 0x7f) + (127 - t)) | d  <=>  d > t, per byte, no carries between bytes
                const unsigned ns = ((dn & M7) + KT) | dn | ((ds & M7) + KT) | ds;
                const unsigned ew = ((de & M7) + KT) | de | ((dw & M7) + KT) | dw;
                const unsigned nib = ((ns & ew & livemask) * 0x00204081u) >> 28;   // bit i = pixel i of the quad
                const unsigned any = __ballot_sync(0xffffffffu, nib != 0u);
                if (nib) sts_u16(qt + 2u * (unsigned)__popc(any & lt), ent | nib);
                qt += 2u * (unsigned)__popc(any);
                if (qt >= qq_full) { __syncwarp(); qt -= 64u; phaseA2(qt, 32); }
            }
            nq = (int)(qt - qq_s) >> 1;
        }
        // ---- drain
        __syncwarp();
        if (nq > 0) phaseA2(qq_s, nq);
        if (np > 0) { phaseB(0, np); }
        __syncwarp();                                        // every lane is done with the image tile
        overflow_any |= overflow;
        if (ox0 + FW_CW < xend) request(ox0 + FW_CW);        // next chunk's tile lands under the NMS / list phases

        // ---- phase C: 3x3 NMS of the queued corners (or, after a queue overflow, of every scored pixel of the region)
        if (!overflow) {
            for (int i = lane; i < cn; i += 32) {
                const unsigned e = lds_u16(cq_s + 2u * (unsigned)i);
                const unsigned sy = e >> 8, sx = e & 255u;
                const unsigned p = score_s + sy * FW_SP + sx;
                const unsigned s = lds_u8(p);
                const unsigned nmax = max(max(max(lds_u8(p - 1), lds_u8(p + 1)), max(lds_u8(p - FW_SP - 1), lds_u8(p - FW_SP))),
                                          max(max(lds_u8(p - FW_SP + 1), lds_u8(p + FW_SP - 1)), max(lds_u8(p + FW_SP), lds_u8(p + FW_SP + 1))));
                if (s > nmax) {
                    const unsigned bit = sx - 3u;
                    asm volatile("red.shared.or.b32 [%0], %1;" :: "r"(mask_s + ((sy - 1u) * 4u + (bit >> 5)) * 4u), "r"(1u << (bit & 31u)) : "memory");
                }
            }
        } else {
            for (int sy = 1; sy <= nrows; ++sy)
                for (int k = 0; k < 4; ++k) {
                    const int sx = 4 * lane + k;
                    if (sx < 3 || sx >= sx_hi) continue;
                    const unsigned p = score_s + (unsigned)sy * FW_SP + (unsigned)sx;
                    const unsigned s = lds_u8(p);
                    if (s == 0u) continue;
                    const unsigned nmax = max(max(max(lds_u8(p - 1), lds_u8(p + 1)), max(lds_u8(p - FW_SP - 1), lds_u8(p - FW_SP))),
                                              max(max(lds_u8(p - FW_SP + 1), lds_u8(p + FW_SP - 1)), max(lds_u8(p + FW_SP), lds_u8(p + FW_SP + 1))));
                    if (s > nmax) {
                        const unsigned bit = (unsigned)sx - 3u;
                        asm volatile("red.shared.or.b32 [%0], %1;" :: "r"(mask_s + ((unsigned)(sy - 1) * 4u + (bit >> 5)) * 4u), "r"(1u << (bit & 31u)) : "memory");
                    }
                }
        }
        __syncwarp();
        // ---- phase D: ordered extraction; mask word idx = row * 4 + wi (4 consecutive lanes = one row), two rounds of 8 rows
#pragma unroll
        for (int rd = 0; rd < 2; ++rd) {
            const int idx = rd * 32 + lane, row = idx >> 2, wi = idx & 3;
            uint32_t m = lds_u32(mask_s + 4u * (unsigned)idx);
            asm volatile("st.shared.u32 [%0], %1;" :: "r"(mask_s + 4u * (unsigned)idx), "r"(0u) : "memory");
            const int cnt = __popc(m);
            int pre = cnt;                                   // inclusive prefix inside the row's 4-lane group
#pragma unroll
            for (int d = 1; d < 4; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, pre, d, 4); if (wi >= d) pre += o; }
            const uint32_t base = lds_u32(rcnt_s + 4u * (unsigned)row);
            __syncwarp();
            uint32_t slot = base + pre - cnt;
            uint32_t* dst = ent_out + (size_t)(y0 - ORBX_EDGE + row) * L.ent_pitch;
            while (m) {
                const int b = __ffs(m) - 1;
                m &= m - 1;
                const int bit = wi * 32 + b;
                const uint32_t sc = lds_u8(score_s + (unsigned)(row + 1) * FW_SP + (unsigned)bit + 3u);
                dst[slot++] = (uint32_t)(ox0 + bit) | (sc << 16);
            }
            if (wi == 3) asm volatile("st.shared.u32 [%0], %1;" :: "r"(rcnt_s + 4u * (unsigned)row), "r"(base + pre) : "memory");
        }
        __syncwarp();
    }
    if (lane < nrows) cnt_out[y0 - ORBX_EDGE + lane] = lds_u32(rcnt_s + 4u * (unsigned)lane);
    (void)overflow_any;
}

}  // namespace orbx
