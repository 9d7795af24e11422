// orbx_desc.cuh -- A.7 IC orientation, A.9 steered rBRIEF-256, A.10 cv::KeyPoint records (the descriptor half of
// cv::ORB::detectAndCompute, src/frontend.cpp:153), sm_100a.  Warp-private windows fed by TMA, no block barrier.
//
// Unit of work: one WARP walks `gpw` GROUPS of 4 consecutive output slots of one frame.  Per keypoint two windows arrive
// by cp.async.bulk.tensor (3-D u8 tensor maps (x, y, frame) per level, completion on the warp's mbarriers):
//     unblurred  rows y-15 .. y+15, 48 bytes from (x-15) & ~15   (31 x 48)  -> IC moments
//     blurred    rows y-18 .. y+18, 64 bytes from (x-18) & ~15   (37 x 64)  -> rBRIEF samples
//   (TMA wants the first byte of a box 16-byte aligned; both windows stay inside the level: keypoints keep 31 px from the border)
// through two-deep rings that are refilled the moment a window has been consumed, with the NEXT group's keypoints already
// located (their selection records are read a whole group ahead), so in the steady state no load latency is exposed and
// there is not a single per-lane copy instruction (the cp.async version spent 22 % of its instructions on them).
// Measured and dropped: PERSISTENT warps (one wave of CTAs, every warp walking (group, frame) items strided over the whole
// batch, general ring bookkeeping for partial groups in mid-stream): parity-green, but 0.216 ms against 0.185 ms -- short-lived
// warps that work on neighbouring groups of one frame keep the windows' lines in L1 / L2 and stagger the phases; so do more
// groups per warp (gpw 8 / 16: 0.205 / 0.259 ms).
//   phase 1  IC moments of the group's 4 keypoints: lane <-> (row mod 4, 4-column chunk); sum(u I), sum(I) by DP4A on
//            disc-masked words, m01 = sum(v * row sum); shuffle reduction; lane k keeps the moments of keypoint k
//   phase 2  LANE-PARALLEL over the 4 keypoints: fastAtan2, the glibc-exact sinf / cosf in FP64 and the seven record fields are
//            computed once per group instead of once per keypoint on all 32 lanes
//   phase 3  per keypoint: lane <-> descriptor byte, the lane's 8 test pairs in registers for the warp's lifetime,
//            packed FMUL2 rotation, magic-number cvRound folded into the sample address
//   flush    the group's 4 x 32 descriptor bytes and 4 x 28 record bytes leave shared memory as 128-bit stores
//            (8 + 7 lanes; scalar stores when the caller's record array is not 16-byte aligned or the group is partial)
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "orbx_geom.h"

namespace orbx {

constexpr int DS_NW = 4;                          // warps per CTA (independent units)
constexpr int DS_G = 4;                           // keypoints per group
constexpr int DS_ICW = 48, DS_ICH = 31;           // unblurred box
constexpr int DS_BLW = 64, DS_BLH = 37;           // blurred box
constexpr int DS_IC_BYTES = (DS_ICW * DS_ICH + 127) / 128 * 128 + 128;   // + 128: the lanes of row "31" (masked out) still read
constexpr int DS_BL_BYTES = (DS_BLW * DS_BLH + 127) / 128 * 128;
constexpr int DS_OFF_BL = 2 * DS_IC_BYTES;
constexpr int DS_OFF_ODESC = DS_OFF_BL + 2 * DS_BL_BYTES;
constexpr int DS_OFF_OKPS = DS_OFF_ODESC + DS_G * 32;
constexpr int DS_OFF_BAR = DS_OFF_OKPS + 128;
constexpr int DS_WARP_BYTES = (DS_OFF_BAR + 4 * 8 + 127) / 128 * 128;

struct DescMaps { CUtensorMap ic[ORBX_LEVELS_MAX], bl[ORBX_LEVELS_MAX]; };   // pyramid level / blurred level as (x, y, frame)

struct DsKp { int x, y, lvl; float resp; bool ok; };

// (5 resident CTAs per SM = 95 registers per thread: 0.171 ms per 256 VGA frames; 6 CTAs / 80 registers 0.181, 4 / 128 0.181, 3 / 147 0.220)
__global__ void __launch_bounds__(DS_NW * 32, 5) k_describe_tma(const __grid_constant__ Geom g, const __grid_constant__ DescMaps maps, int f0,
                                                                const Elem* __restrict__ work, const int* __restrict__ fincnt,
                                                                const float4* __restrict__ pattern, float* __restrict__ kps_out,
                                                                uint8_t* __restrict__ desc_out, int* __restrict__ counts_out, int cap, int gpw,
                                                                int* __restrict__ status)
{
    extern __shared__ __align__(128) uint8_t ds_smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, f = blockIdx.y;
    // ---- per-level counts -> inclusive prefix across lanes (lane l <-> level l)
    int pre = lane < g.nlevels ? __ldg(fincnt + f * g.nlevels + lane) : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, pre, d); if (lane >= d) pre += o; }
    const int total = __shfl_sync(0xffffffffu, pre, 31);
    if (blockIdx.x == 0 && threadIdx.x == 0) counts_out[f] = total;
    const int nkp = min(total, cap);
    const int ngroups = (nkp + DS_G - 1) / DS_G;
    int gi = blockIdx.x * (DS_NW * gpw) + wid;               // this warp's groups: gi, gi + DS_NW, ...
    if (gi >= ngroups) return;                               // warp-uniform; warps are independent
    const int g_end = min(ngroups, blockIdx.x * (DS_NW * gpw) + DS_NW * gpw);

    const unsigned base_s = (((unsigned)__cvta_generic_to_shared(ds_smem) + 127u) & ~127u) + (unsigned)wid * DS_WARP_BYTES;
    const unsigned bar_ic = base_s + DS_OFF_BAR, bar_bl = bar_ic + 16u;
    const unsigned odesc_s = base_s + DS_OFF_ODESC, okps_s = base_s + DS_OFF_OKPS;
    if (lane == 0) {
        mbar_init(bar_ic, 1); mbar_init(bar_ic + 8u, 1); mbar_init(bar_bl, 1); mbar_init(bar_bl + 8u, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    // group -> its keypoints, lane-parallel: lane (k, k + 4, ...) takes slot 4 * group + k
    const int kq = lane & 3;
    auto locate = [&](int grp) -> DsKp {
        const int slot = grp * DS_G + kq;
        DsKp k;
        k.ok = slot < nkp;
        const int s = k.ok ? slot : 0;
        int lvl = 0;
        for (int j = 0; j < g.nlevels - 1; ++j) lvl += (__shfl_sync(0xffffffffu, pre, j) <= s) ? 1 : 0;
        const int before = __shfl_sync(0xffffffffu, pre, max(lvl - 1, 0));
        const Elem e = work[(size_t)f * g.ws_frame + g.L[lvl].ws_off + (s - (lvl > 0 ? before : 0))];
        k.x = (int)(e.pos & 0xffffu); k.y = (int)(e.pos >> 16); k.lvl = lvl; k.resp = e.response;
        return k;
    };
    auto load_ic = [&](const DsKp& k, unsigned b) {          // called by ONE lane
        mbar_expect_tx(bar_ic + 8u * b, DS_ICW * DS_ICH);
        tma_load_tile_3d(base_s + b * DS_IC_BYTES, &maps.ic[k.lvl], (k.x - 15) & ~15, k.y - 15, f0 + f, bar_ic + 8u * b);
    };
    auto load_bl = [&](const DsKp& k, unsigned b) {
        mbar_expect_tx(bar_bl + 8u * b, DS_BLW * DS_BLH);
        tma_load_tile_3d(base_s + DS_OFF_BL + b * DS_BL_BYTES, &maps.bl[k.lvl], (k.x - 18) & ~15, k.y - 18, f0 + f, bar_bl + 8u * b);
    };

    DsKp cur = locate(gi);
    bool has_next = gi + DS_NW < g_end;
    DsKp nxt = cur;
    if (has_next) nxt = locate(gi + DS_NW); else nxt.ok = false;
    if (lane < 2 && cur.ok) { load_ic(cur, (unsigned)lane); load_bl(cur, (unsigned)lane); }

    // ---- this lane's 8 test pairs: (x0, x1) and (y0, y1) packs, read once with coalesced 128-bit loads (the host transposes
    //      the pattern table to [t][lane]); a per-keypoint gather of 128-byte-strided float4s costs 32 L1 wavefronts per
    //      load and makes the LSU the bound
    unsigned long long PX[8], PY[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const float4 pt = __ldg(pattern + t * 32 + lane);
        PX[t] = f2_pack(pt.x, pt.z);
        PY[t] = f2_pack(pt.y, pt.w);
    }
    // ---- IC disc: lane <-> (q = row mod 4, j = 4-column chunk); rows 4 i + q, i = 0 .. 7 (row 31 does not exist: mask 0)
    const int icq = lane >> 3, icj = lane & 7;
    uint32_t icmask[8];
    {
        // umax[|v|] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3} as nibbles (no local array)
        constexpr unsigned long long UMAXP = 0x3689ABCDDEEEFFFFull;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int row = 4 * i + icq, v = row - 15;
            const int um = row <= 30 ? (int)((UMAXP >> (4 * (v < 0 ? -v : v))) & 15ull) : -1;
            uint32_t m = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int u = 4 * icj + b - 15;
                if ((u < 0 ? -u : u) <= um) m |= 0xFFu << (8 * b);
            }
            icmask[i] = m;
        }
    }
    const int u0 = 4 * icj - 15;
    const uint32_t iccoef = (uint32_t)(u0 & 255) | ((uint32_t)((u0 + 1) & 255) << 8) | ((uint32_t)((u0 + 2) & 255) << 16) | ((uint32_t)((u0 + 3) & 255) << 24);
    const bool vec_kps = ((cap & 3) == 0) && ((reinterpret_cast<uintptr_t>(kps_out) & 15) == 0);
    const bool vec_desc = (reinterpret_cast<uintptr_t>(desc_out) & 15) == 0;

    unsigned n = 0;                                          // keypoints of this warp consumed so far: ring slot n & 1, parity (n >> 1) & 1
#pragma unroll 1
    for (;;) {
        const int nv = min(DS_G, nkp - gi * DS_G);           // keypoints of this group (< 4 only for the frame's last group)
        // ---- phase 1: IC moments
        int M10 = 0, M01 = 0;
#pragma unroll 1
        for (int k = 0; k < nv; ++k) {
            const unsigned m = n + (unsigned)k, b = m & 1u;
            if (!mbar_wait(bar_ic + 8u * b, (m >> 1) & 1u)) { if (lane == 0) atomicOr(&status[f], 2); return; }
            const int xk = __shfl_sync(0xffffffffu, cur.x, k);
            const unsigned off = (unsigned)(xk - 15) & 15u;                                    // window column u = -15 sits at this byte of the box row
            const unsigned ra = base_s + b * DS_IC_BYTES + (unsigned)icq * DS_ICW + (unsigned)icj * 4u + (off & ~3u);
            const unsigned shb = (off & 3u) * 8u;
            int m10 = 0, m01 = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const unsigned w0 = lds_u32(ra + i * 4 * DS_ICW), w1 = lds_u32(ra + i * 4 * DS_ICW + 4u);
                const uint32_t w = __funnelshift_r(w0, w1, shb) & icmask[i];
                m10 = dp4a_us(w, iccoef, m10);
                m01 += (4 * i - 15 + icq) * dp4a_us(w, 0x01010101u, 0);
            }
            m10 = __reduce_add_sync(0xffffffffu, m10);       // REDUX: one instruction per sum instead of five shuffle + add steps
            m01 = __reduce_add_sync(0xffffffffu, m01);
            if (kq == k) { M10 = m10; M01 = m01; }
            // the window is consumed (the reductions above ordered every lane's reads): refill its slot with keypoint m + 2
            if (lane == ((k + 2) & 3)) {
                if (k < 2) { if (cur.ok) load_ic(cur, b); }
                else if (nxt.ok) load_ic(nxt, b);
            }
        }
        // ---- phase 2 (lane-parallel over the group's keypoints): angle, sin / cos, record
        const float ang = fast_atan2_deg((float)M01, (float)M10);
        float sn, cs;
        glibc_sincosf(__fmul_rn(ang, __int_as_float(0x3c8efa35)), &sn, &cs);
        if (lane < nv) {
            const float sc = g.L[cur.lvl].scale;
            const unsigned o = okps_s + (unsigned)lane * 28u;
            asm volatile("st.shared.f32 [%0], %1;" :: "r"(o), "f"(__fmul_rn((float)cur.x, sc)) : "memory");
            asm volatile("st.shared.f32 [%0], %1;" :: "r"(o + 4u), "f"(__fmul_rn((float)cur.y, sc)) : "memory");
            asm volatile("st.shared.f32 [%0], %1;" :: "r"(o + 8u), "f"(__fmul_rn(31.0f, sc)) : "memory");
            asm volatile("st.shared.f32 [%0], %1;" :: "r"(o + 12u), "f"(ang) : "memory");
            asm volatile("st.shared.f32 [%0], %1;" :: "r"(o + 16u), "f"(cur.resp) : "memory");
            asm volatile("st.shared.u32 [%0], %1;" :: "r"(o + 20u), "r"(cur.lvl) : "memory");
            asm volatile("st.shared.u32 [%0], %1;" :: "r"(o + 24u), "r"(-1) : "memory");
        }
        // ---- phase 3: steered rBRIEF, lane <-> descriptor byte
#pragma unroll 1
        for (int k = 0; k < nv; ++k) {
            const unsigned m = n + (unsigned)k, b = m & 1u;
            if (!mbar_wait(bar_bl + 8u * b, (m >> 1) & 1u)) { if (lane == 0) atomicOr(&status[f], 2); return; }
            const float snk = __shfl_sync(0xffffffffu, sn, k), csk = __shfl_sync(0xffffffffu, cs, k);
            const int xk = __shfl_sync(0xffffffffu, cur.x, k);
            // (v + MAGIC) holds rint(v) in its low mantissa bits, exactly for |v| < 2^22; MAGIC = 1.5 * 2^23 + 18 moves the
            // origin to the window's corner (18 is even, so ties-to-even is unchanged).  addr = DS_BLW * bits(y) + bits(x) + cbase  (mod 2^32)
            // The rotation's products are packed FMUL2 (mul / add .f32x2 are IEEE per half); the subtraction / addition stays
            // scalar because ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even under -fmad=false.
            const unsigned long long MAGIC2 = f2_pack(12582930.0f, 12582930.0f);
            const unsigned long long cs2 = f2_pack(csk, csk), sn2 = f2_pack(snk, snk);
            const unsigned cbase = base_s + DS_OFF_BL + b * DS_BL_BYTES + ((unsigned)(xk - 18) & 15u) - (unsigned)(DS_BLW + 1) * 0x4B400000u;
            unsigned byte = 0;
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const unsigned long long xc = f2_mul(PX[t], cs2), ys = f2_mul(PY[t], sn2);
                const unsigned long long xs = f2_mul(PX[t], sn2), yc = f2_mul(PY[t], cs2);
                const float fx0 = __fsub_rn(f2_lo(xc), f2_lo(ys)), fx1 = __fsub_rn(f2_hi(xc), f2_hi(ys));
                const float fy0 = __fadd_rn(f2_lo(xs), f2_lo(yc)), fy1 = __fadd_rn(f2_hi(xs), f2_hi(yc));
                const unsigned long long bx = f2_add(f2_pack(fx0, fx1), MAGIC2), by = f2_add(f2_pack(fy0, fy1), MAGIC2);
                const unsigned a0 = (unsigned)by * (unsigned)DS_BLW + (unsigned)bx + cbase;
                const unsigned a1 = (unsigned)(by >> 32) * (unsigned)DS_BLW + (unsigned)(bx >> 32) + cbase;
                const unsigned t0 = lds_u8(a0), t1 = lds_u8(a1);
                byte |= (unsigned)(t0 < t1) << t;
            }
            sts_u8(odesc_s + (unsigned)k * 32u + (unsigned)lane, byte);
            __syncwarp();                                    // every lane has sampled this window
            if (lane == ((k + 2) & 3)) {
                if (k < 2) { if (cur.ok) load_bl(cur, b); }
                else if (nxt.ok) load_bl(nxt, b);
            }
        }
        // ---- flush the group's outputs: 128-bit stores
        {
            const size_t o = (size_t)f * cap + (size_t)gi * DS_G;
            if (vec_desc) {
                if (lane < 2 * nv) *reinterpret_cast<uint4*>(desc_out + o * 32 + (size_t)lane * 16) = lds_v4(odesc_s + (unsigned)lane * 16u);
            } else {
                for (int k = 0; k < nv; ++k) desc_out[(o + k) * 32 + lane] = (uint8_t)lds_u8(odesc_s + (unsigned)k * 32u + (unsigned)lane);
            }
            if (vec_kps && nv == DS_G) {
                if (lane < 7) *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(kps_out) + o * 28 + (size_t)lane * 16) = lds_v4(okps_s + (unsigned)lane * 16u);
            } else if (lane < 7 * nv) {
                reinterpret_cast<uint32_t*>(kps_out)[o * 7 + lane] = lds_u32(okps_s + (unsigned)lane * 4u);
            }
        }
        if (!has_next) break;
        __syncwarp();                                        // the staging rows are read before the next group overwrites them
        n += DS_G;
        gi += DS_NW;
        cur = nxt;
        has_next = gi + DS_NW < g_end;
        if (has_next) nxt = locate(gi + DS_NW); else nxt.ok = false;
    }
}

}  // namespace orbx
