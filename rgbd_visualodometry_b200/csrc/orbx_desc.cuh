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
#include "orbx_device.cuh"

namespace orbx {

__device__ __forceinline__ void cp_async_8(unsigned dst, const void* src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(dst), "l"(src) : "memory"); }
__device__ __forceinline__ int dp4a_us(unsigned a_u8x4, unsigned b_s8x4, int c)       // sum of u8 * s8 products + c
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_u8x4), "r"(b_s8x4), "r"(c));
    return d;
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

// ------------------------------------------------------------------------------------------------ A.7 / A.9 / A.10 describe
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
