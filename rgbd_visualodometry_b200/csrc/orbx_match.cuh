// orbx_match.cuh -- brute-force Hamming matcher on the sm_100a int8 tensor cores (tcgen05 / TMEM).
//
// Replaces cv::DescriptorMatcher::match at src/frontend.cpp:187 (query = map-point candidates, M x 32 B;
// train = frame descriptors, N x 32 B) with exact BFMatcher(NORM_HAMMING) semantics (SURVEY A.11):
// argmin over train rows of popcount(q ^ t), ties -> lowest train index.
//
// Identity used: expand every descriptor bit to a +-1 int8 (bit 1 -> +1, bit 0 -> -1); then
//   dot(q, t) = 256 - 2 * hamming(q, t)   =>   hamming = (256 - dot) / 2          (exact, |dot| <= 256)
// so the M x N distance matrix is one int8 GEMM with K = 256 and int32 accumulation.
//
// One CTA owns 256 query rows (two 128-row A tiles).  The map is shared by every frame, so the A operand is expanded
// ONCE per CTA and parked in TENSOR MEMORY (tcgen05.st; the MMA then takes A from TMEM, "TS" form), which removes
// half of the shared-memory operand traffic of every MMA.  The CTA then walks train sets and, inside a set, tiles of
// 96 train rows (B tiles).  Warp roles (ids chosen so that the latency-critical roles sit on the higher warp ids):
//   warps 0-5   expanders : two groups of 96 threads on alternate tiles; 32-byte descriptor rows -> +-1 int8 rows written
//                           straight into the 128B-swizzled K-major UMMA layout; the bit expansion is pure ALU
//                           (multiply-spread), never touches HBM or a LUT; raw rows arrive through a cp.async ring
//   warps 15, 6 issuers   : alternate tiles; per tile 2 x (8 + 1) tcgen05.mma.kind::i8 (N96 K32, A from TMEM) into a
//                           double-buffered pair of TMEM accumulators, commits to mbarriers
//   warps 7-14  epilogue  : tcgen05.ld of the tile's 96 columns PACKED to 16 bits, TMEM buffer released right away, row
//                           maximum by VIMNMX3.S16x2; per set one packed key  dot << 20 | (0xFFFFF - j)
// Index tie-break folded into the GEMM: query bits expand to +-127, and one extra k-step multiplies a constant A
// tile (a single 1 per row) with a constant B tile whose row jl holds the code (MT_BN-1 - jl).  The accumulator then reads
// 127 * dot + code: its plain integer maximum over a tile IS "largest dot, lowest train index", so the epilogue is one
// packed max per four columns instead of a multiply-and-pack per column, and the winner's index is decoded from the code.
// The same body runs as a single CTA per query tile (k_hamming_umma, cta_group::1, M = 128) and as a CTA PAIR that shares
// every B tile (k_hamming_umma2, cta_group::2, M = 256; see "CTA pair" below).
// TMEM map (512 columns): accumulators [buffer 0..1][A tile 0..1] x 96 columns at 0..383, A tiles 2 x 64 columns at 384.
// Pipelines: smem stages (expanders <-> issuer) and TMEM accumulators (issuer <-> epilogue), all mbarrier based,
// running continuously across set boundaries (persistent CTAs).  Train-row ranges can be split across CTAs (small
// problems); partial results merge with atomicMax on the packed key.
// Pairwise batches (SETQ: query set s against train set s, e.g. frame i against frame i + 1) cannot keep one A operand
// across sets, so there a CTA owns ONE (set, query tile) unit: gridDim.z = number of sets, the A tile is expanded at setup
// as above, and CTAs whose query tile is empty for their set exit before any setup.  Few units keep the train-row split.
// One body serves every operation (MatchOp): match, knnMatch k = 2, cross-check, top-k and the two radius passes.
// knnMatch for k > 2 (TopK, KB = list capacity 4 / 8 / 16 / 32): the single-CTA body, shared-query or pairwise, whose epilogue
// keeps each query row's KB best keys in registers (see topk_tile); no CTA pair and no train-row split, as for knn2.
// radiusMatch (RadiusCount, RadiusEmit): the same single-CTA body, whose epilogue counts, then writes, each query row's columns
// at or above the radius threshold (see radius_tile); orbx_radius.cuh scans the counts and orders the lists.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "orbx_device.cuh"

namespace orbx {

constexpr int MT_QROWS = 256;          // query rows per CTA (two UMMA M=128 tiles)
constexpr int MT_BN = 96;              // train rows per B tile (UMMA N)
constexpr int MT_STAGES = 4;
constexpr int MT_EXP_GROUPS = 2;                  // expander groups take alternate B tiles, so a group has two tile periods per tile
constexpr int MT_EXP_WARPS = MT_EXP_GROUPS * MT_BN / 32;
// Warp ids: the SM's warp arbiter favours HIGHER warp ids, so the latency-critical roles sit on top:
//   0 .. 5 expanders (run ahead, not critical) | 6 MMA issuer of the odd tiles | 7 .. 14 epilogue | 15 MMA issuer of the even tiles
constexpr int MT_EPI_WARP0 = 7;
constexpr int MT_ISSUER_WARP = 15;
constexpr int MT_ISSUER2_WARP = 6;      // second issuer (odd tiles): its barrier waits / commits run under the other issuer's MMAs
constexpr int MT_THREADS = 16 * 32;
static_assert(MT_EXP_WARPS <= MT_EPI_WARP0, "role layout");
constexpr int MT_B_BYTES = MT_BN * 256;
constexpr int MT_SMEM_B = 0;
constexpr int MT_PREFETCH = 6;          // raw descriptor rows are fetched this many B tiles ahead (cp.async ring)
constexpr int MT_SMEM_RAW = MT_SMEM_B + MT_STAGES * MT_B_BYTES;
constexpr int MT_SMEM_CA = MT_SMEM_RAW + MT_EXP_GROUPS * MT_PREFETCH * MT_BN * 32;   // constant A tile of the bias k-step (128 rows x 128 B, SW128)
constexpr int MT_SMEM_CB = MT_SMEM_CA + 128 * 128;                  // constant B tile of the bias k-step (MT_BN rows x 128 B, SW128)
constexpr int MT_SMEM_BAR = MT_SMEM_CB + MT_BN * 128;
constexpr int MT_ASCALE = 127;         // query bits expand to +-127, train bits to +-1: accumulator = 127 * dot + bias
static_assert(MT_BN <= MT_ASCALE, "the per-tile index bias must stay below the dot-product quantum");
constexpr int MT_SMEM_BYTES = MT_SMEM_BAR + 128 + 1024;   // + barriers/tmem slot + 1 KB alignment slack
constexpr uint32_t MT_TMEM_COLS = 512;
constexpr uint32_t MT_TMEM_A = 4 * MT_BN;                  // first column of the A tiles
constexpr int MT_KEY_SHIFT = 20;
constexpr int MT_MAX_TRAIN = 1 << MT_KEY_SHIFT;            // train rows per set representable in the packed key
static_assert(4 * MT_BN + 128 <= 512, "TMEM budget");
// cross-check kernels only: every epilogue warp's column maxima of a tile, [accumulator buffer][epilogue warp][MT_BN] ints,
// behind the barrier block (the other kernels' layout and launch size stay as they are)
constexpr int MT_SMEM_XC = MT_SMEM_BAR + 128;
constexpr int MT_SMEM_BYTES_XC = MT_SMEM_XC + 2 * 8 * MT_BN * 4 + 1024;
constexpr int MT_MAX_QUERY_XC = 1 << MT_KEY_SHIFT;         // query rows representable in the column key dot << 20 | (0xFFFFF - q)

// ---- PTX wrappers ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// single non-blocking probe of an mbarrier phase
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
// A operand from tensor memory (TS form): D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void tc_mma_i8_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
                 "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
                 "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                   "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
                   "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
                   "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
                 : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
}
// .pack::16b: two adjacent 32-bit columns -> the low halves of both in one register (the accumulators fit in 16 bits);
// .xN counts destination registers, so N registers cover 2N columns
__device__ __forceinline__ void tc_ld32_pack16(uint32_t taddr, uint32_t* r) {     // 64 columns -> 32 registers
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.pack::16b.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld16_pack16(uint32_t taddr, uint32_t* r) {     // 32 columns -> 16 registers
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.pack::16b.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format: version 1 at bit 46, layout 2 at bit 61);
// 8-row groups are 1024 B apart (SBO = 64 x 16 B); LBO is unused for swizzled K-major (1 by convention).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor: D = S32 (c_format 2), A = B = signed int8 (format 1), both K-major, N = MT_BN, M = 128
constexpr uint32_t MT_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(MT_BN >> 3) << 17) | ((128u >> 4) << 24);

// 4 descriptor bits -> 4 int8 (+1 for a set bit, -1 otherwise): multiply-spread the nibble to one bit per byte, then
// 0xFF - 0xFE * bit.  No table, no shared-memory traffic.
__device__ __forceinline__ uint32_t pm1x4(uint32_t nibble) {
    const uint32_t spread = (nibble * 0x00204081u) & 0x01010101u;
    return 0xFFFFFFFFu - spread * 0xFEu;
}
__device__ __forceinline__ uint32_t pm127x4(uint32_t nibble) {          // +127 for a set bit, -127 otherwise
    const uint32_t spread = (nibble * 0x00204081u) & 0x01010101u;
    return 0x81818181u ^ (spread * 0xFEu);
}
// word i (0..63) of the expanded row = int8 values of descriptor bits 4i .. 4i+3
__device__ __forceinline__ uint32_t pm1_word(const uint32_t* w, int i) { return pm1x4((w[i >> 3] >> ((i & 7) * 4)) & 15u); }

// Expand one 32-byte descriptor row into 256 +-1 int8 in the canonical K-major SW128 layout of a `rows`-row tile:
//   byte k of row r  ->  tile + (k / 128) * rows * 128 + (r / 8) * 1024 + (r % 8) * 128 + (((k % 128) / 16) ^ (r % 8)) * 16 + k % 16
__device__ __forceinline__ void expand_row(uint8_t* tile, int rows, int r, const uint4 lo, const uint4 hi)
{
    const uint32_t w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    uint8_t* rbase = tile + (r >> 3) * 1024 + (r & 7) * 128;
#pragma unroll
    for (int c16 = 0; c16 < 16; ++c16) {                     // 16 descriptor bits -> 16 int8 -> one 16-byte chunk
        uint8_t* dst = rbase + (c16 >> 3) * rows * 128 + (((c16 & 7) ^ (r & 7)) << 4);
        *reinterpret_cast<uint4*>(dst) = make_uint4(pm1_word(w, 4 * c16), pm1_word(w, 4 * c16 + 1), pm1_word(w, 4 * c16 + 2), pm1_word(w, 4 * c16 + 3));
    }
}

// One K half (descriptor bytes 16h .. 16h+15 -> int8 columns 128h .. 128h+127) of row r.
__device__ __forceinline__ void expand_half_row(uint8_t* tile, int rows, int r, int h, const uint4 v)
{
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint8_t* rbase = tile + h * rows * 128 + (r >> 3) * 1024 + (r & 7) * 128;
#pragma unroll
    for (int c = 0; c < 8; ++c) {                            // 16 descriptor bits -> 16 int8 -> one 16-byte chunk
        const uint32_t two = w[c >> 1] >> ((c & 1) * 16);
        *reinterpret_cast<uint4*>(rbase + ((c ^ (r & 7)) << 4)) =
            make_uint4(pm1x4(two & 15u), pm1x4((two >> 4) & 15u), pm1x4((two >> 8) & 15u), pm1x4((two >> 12) & 15u));
    }
}

// Persistent over train sets: CTA (x = query tile, y = train-row split, z = set group) expands its 256 query rows
// ONCE and then walks sets z, z + gridDim.z, ... with all three pipelines running continuously across set
// boundaries (the map is shared by every frame, so the A operand never has to be rebuilt).
struct MatchSetRange { int n0, n1, ntiles; };
// rows present in a set (ragged sets: the raw count, clamped later) -- split from the range arithmetic so that a caller can
// issue the load a whole set ahead and only consume it at the next set boundary
__device__ __forceinline__ int match_set_count(const int* __restrict__ counts, int set, int nt)
{
    if (!counts) return nt;
    int v;                                                   // volatile: issued HERE, not sunk to the point of use
    asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(counts + set));
    return v;
}
__device__ __forceinline__ MatchSetRange match_set_range_n(int count, int nt, int split, int rows_per_split)
{
    const int nvalid = max(0, min(count, nt));
    MatchSetRange r;
    r.n0 = split * rows_per_split;
    r.n1 = min(nvalid, r.n0 + rows_per_split);
    r.ntiles = r.n1 > r.n0 ? (r.n1 - r.n0 + MT_BN - 1) / MT_BN : 0;
    return r;
}
__device__ __forceinline__ MatchSetRange match_set_range(const int* __restrict__ counts, int set, int nt, int split, int rows_per_split)
{
    return match_set_range_n(match_set_count(counts, set, nt), nt, split, rows_per_split);
}

// ---- CTA pair (tcgen05 cta_group::2): the same body with PAIR = true ---------------------------------------------
// Two CTAs on the SMs of one TPC share every B tile.  Each CTA still owns 256 query rows (two
// 128-row A tiles parked in its own tensor memory) and its own accumulators and epilogue; of a 96-row train tile each
// CTA expands only HALF (48 rows, two threads per row) into its own shared memory, and one UMMA of M = 256 issued by the
// leader feeds both SMs' tensor cores (the hardware exchanges the B halves).  Per SM that halves the bit expansion and the
// shared-memory operand reads of every MMA -- the two things that kept the single-CTA kernel at ~57 instead of 48 cycles
// per MMA.  Barriers: "stage full" and "accumulators free" live in the leader (the peer arrives on them through the
// cluster address space); "stage free" and "accumulators full" are signalled in BOTH CTAs by multicast tcgen05.commit.
// Row code of the bias k-step: local row i of CTA r carries 95 - (48 r + i); for a partial last tile issued with a smaller
// UMMA N the peer holds rows N/2 .. N-1, still in decreasing code order, and the epilogue maps the code back with N.
constexpr int MT2_HALF = MT_BN / 2;                          // train rows of a B tile held by each CTA of the pair
constexpr int MT2_GROUP_WARPS = MT_BN / 32;                  // expander warps per group (two threads per local row)
// instruction descriptor: as MT_IDESC but M = 256 (cta_group::2)
constexpr uint32_t MT2_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(MT_BN >> 3) << 17) | ((256u >> 4) << 24);

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t cta) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(cta)); return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");   // (default .release.cta, as CUTLASS' ClusterBarrier::arrive(cta_id): the cluster-scope form stalls the warp for ~1000 cycles)
}
__device__ __forceinline__ void tc_commit2(uint32_t bar) {   // arrives on the barrier at this offset in BOTH CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc_mma2_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_mma2_i8_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::i8 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}


// PAIR-generic pieces of the body
template <bool PAIR> __device__ __forceinline__ void group_sync() { if (PAIR) cluster_sync_all(); else __syncthreads(); }
template <bool PAIR> __device__ __forceinline__ void tmem_alloc_all(uint32_t slot_saddr) {
    if (PAIR) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_saddr), "r"(MT_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_saddr), "r"(MT_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
}
template <bool PAIR> __device__ __forceinline__ void tmem_dealloc_all(uint32_t base) {
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(MT_TMEM_COLS) : "memory");
    else      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(MT_TMEM_COLS) : "memory");
}
template <bool PAIR> __device__ __forceinline__ void bar_arrive_lead(uint32_t addr) { if (PAIR) mbar_arrive_cluster(addr); else mbar_arrive(addr); }
template <bool PAIR> __device__ __forceinline__ void umma_i8_ts(uint32_t d, uint32_t a, uint64_t db, uint32_t idesc, uint32_t acc) {
    if (PAIR) tc_mma2_i8_ts(d, a, db, idesc, acc); else tc_mma_i8_ts(d, a, db, idesc, acc);
}
template <bool PAIR> __device__ __forceinline__ void umma_i8(uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
    if (PAIR) tc_mma2_i8(d, da, db, idesc, acc); else tc_mma_i8(d, da, db, idesc, acc);
}
template <bool PAIR> __device__ __forceinline__ void umma_commit(uint32_t bar) { if (PAIR) tc_commit2(bar); else tc_commit(bar); }

// ---- what one launch computes -----------------------------------------------------------------------------------------
// The operations of the body.  Best, Knn2 and CrossCheck run on the single-CTA kernel and on the CTA pair; TopK and the
// two radius passes on the single-CTA kernel alone, without a train-row split (as Knn2).
enum class MatchOp : int {
    Best,           // cv match: each query row's nearest train row per set
    Knn2,           // cv knnMatch k = 2: best and second best
    CrossCheck,     // Best, plus every train row's nearest query (column keys) for BFMatcher crossCheck = true
    TopK,           // cv knnMatch for any k <= KB
    RadiusCount,    // cv radiusMatch, first pass: every list's length
    RadiusEmit,     // cv radiusMatch, second pass: the hits of every list that fits the output
};
__host__ __device__ constexpr bool match_op_pairs(MatchOp op) { return op == MatchOp::Best || op == MatchOp::Knn2 || op == MatchOp::CrossCheck; }

// The kernel parameters of one launch.  Record outputs are [nsets][nq] (list L = set * nq + query row).
struct MatchArgs {
    const uint8_t* query;        // nq rows, shared by every set; pairwise (SETQ): set s's own rows at query + s * nq * 32
    int nq;                      // query rows, or the query stride of a pairwise launch (and then the record pitch)
    const int* query_counts;     // pairwise: set s holds min(query_counts[s], nq) query rows; null otherwise
    const uint8_t* train;        // set s at train + s * train_stride_rows * 32
    int nt, train_stride_rows;   // rows per set, stride between sets
    const int* train_counts;     // ragged sets: set s holds min(train_counts[s], nt) rows; null: nt each
    int nsets, rows_per_split;   // train-row split: CTA y takes rows [y * rows_per_split, (y + 1) * rows_per_split) of a set
    int4* best;                  // records (TopK: [nsets][nq][knn_k]; RadiusEmit: the lists, at rad_offsets)
    int4* second;                // Knn2: the second-best records
    int* keys;                   // train-row split: packed row keys merged by atomicMax, made records by k_match_finalize
    int* col_keys;               // CrossCheck: [nsets][train_stride_rows] column keys, INT_MIN-initialised, merged by atomicMax
    int* status;                 // |= 2 when an mbarrier wait timed out
    int knn_k;                   // TopK: k
    int rad_thr;                 // radius: distance <= R  <=>  accumulator >= rad_thr = 127 * (256 - 2R)
    long long* rad_offsets;      // RadiusCount: list L's length to rad_offsets[1 + L]; RadiusEmit: the scanned offsets
    long long rad_cap;           // RadiusEmit: list L is written when rad_offsets[L + 1] <= rad_cap
};

// A DMatch record {queryIdx, trainIdx, imgIdx 0, distance = (256 - dot) / 2}
__device__ __forceinline__ int4 match_record(int qrow, int dot, int j)
{
    return make_int4(qrow, j, 0, __float_as_int((float)((256 - dot) >> 1)));
}
// packed row key  dot << 20 | (0xFFFFF - j)  (plain maximum = largest dot, lowest train index)
__device__ __forceinline__ int row_key(int dot, int j) { return dot * (1 << MT_KEY_SHIFT) + ((MT_MAX_TRAIN - 1) - j); }
// row key -> its record; INT_MIN (no train row) -> trainIdx -1
__device__ __forceinline__ int4 key_record(int qrow, int key)
{
    if (key == INT_MIN) return make_int4(qrow, -1, 0, 0);
    return match_record(qrow, key >> MT_KEY_SHIFT, (MT_MAX_TRAIN - 1) - (key & (MT_MAX_TRAIN - 1)));
}
// An accumulator 127 * dot + code of the tile at train row j0 -> dot and the global train row.  The code is MT_BN - 1 minus
// the row's place in the tile; in a CTA pair places 48 .. 95 are the peer's local rows, which hold tile rows N/2 .. N - 1
// (N: the tile's UMMA N, from the set's end n1).
struct AccRow { int dot, j; };
template <bool PAIR>
__device__ __forceinline__ AccRow acc_row(int v, int j0, int n1)
{
    const unsigned kk = (unsigned)(v + MT_ASCALE * 256);
    const unsigned q = kk / (unsigned)MT_ASCALE;             // dot + 256
    const int place = (MT_BN - 1) - (int)(kk - q * (unsigned)MT_ASCALE);
    const int nh = ((min(MT_BN, n1 - j0) + 31) & ~31) >> 1;
    return {(int)q - 256, j0 + (PAIR && place >= MT2_HALF ? nh + place - MT2_HALF : place)};
}

// ---- cross-check (CrossCheck): column maxima from the same accumulators ----------------------------------------------
// Every column of a tile holds one train row, and all its values carry that row's code, so the column maximum of the
// accumulator is the row's largest dot.  Widened to (v << 8) | (255 - row of the CTA), its plain maximum is "largest
// dot, lowest query row".  One PRMT widens a packed half (the selector's msb replicates the sign of the selected byte).
__device__ __forceinline__ int xc_widen(uint32_t packed, uint32_t c, uint32_t sel)
{
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(packed), "r"(c), "r"(sel));
    return (int)r;
}
// This warp's 96 column maxima over its 32 query rows -> xc[0 .. MT_BN) (slot 2u + h = half h of packed register u, the
// same slot in every warp).  A padded query row (q >= nq) counts as v = -32768, below every accumulator (>= -32512).
__device__ __forceinline__ void xc_warp_columns(const uint32_t* rp, bool valid, int row_cta, int* xc)
{
    const uint32_t c = 255u - (uint32_t)row_cta;
#pragma unroll
    for (int u = 0; u < MT_BN / 2; u += 2) {
        const uint32_t r0 = valid ? rp[u] : 0x80008000u, r1 = valid ? rp[u + 1] : 0x80008000u;
        int4 m;
        m.x = __reduce_max_sync(0xffffffffu, xc_widen(r0, c, 0x9104u));
        m.y = __reduce_max_sync(0xffffffffu, xc_widen(r0, c, 0xB324u));
        m.z = __reduce_max_sync(0xffffffffu, xc_widen(r1, c, 0x9104u));
        m.w = __reduce_max_sync(0xffffffffu, xc_widen(r1, c, 0xB324u));
        *reinterpret_cast<int4*>(xc + 2 * u) = m;
    }
}
__device__ __forceinline__ void xc_epilogue_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }   // the 8 epilogue warps only

// ---- top-k (TopK, KB > 0, BFMatcher knnMatch for any k <= KB): each epilogue thread keeps its query row's KB largest keys
// dot << 20 | (0xFFFFF - j) in registers, in descending order (INT_MIN = empty slot).  Keys are distinct per train row, so
// the first k of them are exactly cv's k nearest by (distance, trainIdx).  A tile's columns are tested against the list's
// last key in accumulator form (one compare per column; the whole tile is skipped when its packed maximum fails); only a
// column that enters the list is decoded and inserted by a branchless shift chain.
// The smallest accumulator of the tile at train row j0 whose key beats key t.  Every earlier tile holds lower train indices,
// so a row of such a tile is beaten by a strictly larger dot only; a row of this tile by a larger 127 * dot + code.
// An empty slot admits every column but the -32768 fill of chunks past the tile's UMMA N.
__device__ __forceinline__ int topk_threshold(int t, int j0)
{
    if (t == INT_MIN) return -32767;
    const int dot = t >> MT_KEY_SHIFT, j = (MT_MAX_TRAIN - 1) - (t & (MT_MAX_TRAIN - 1));
    return j < j0 ? MT_ASCALE * (dot + 1) : MT_ASCALE * dot + ((MT_BN - 1) - (j - j0)) + 1;
}
template <int KB>
__device__ __forceinline__ void topk_insert(int (&list)[KB], int x)   // x > list[KB - 1] or x == INT_MIN (no-op)
{
#pragma unroll
    for (int i = KB - 1; i > 0; --i) list[i] = x > list[i - 1] ? list[i - 1] : max(list[i], x);
    list[0] = max(list[0], x);
}
// One tile's packed accumulators (tmax: their maximum) of train rows j0 .. into the list; columns decoding to j >= n1 are the
// copies of the set's last row that pad a partial tile.
template <int KB>
__device__ __forceinline__ void topk_tile(const uint32_t* rp, int tmax, int j0, int n1, int (&list)[KB])
{
    int thr = topk_threshold(list[KB - 1], j0);
    if (tmax < thr) return;
#pragma unroll
    for (int u = 0; u < MT_BN / 2; ++u)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int v = h ? (int)rp[u] >> 16 : (int)(rp[u] << 16) >> 16;
            if (v >= thr) {
                const AccRow d = acc_row<false>(v, j0, n1);
                topk_insert<KB>(list, d.j < n1 ? row_key(d.dot, d.j) : INT_MIN);
                thr = topk_threshold(list[KB - 1], j0);
            }
        }
}

// ---- radius (RadiusCount and RadiusEmit passes; BFMatcher radiusMatch): distance h <= R  <=>  127 * dot + code >= thr =
// 127 * (256 - 2R), because the index code is below 127.  A tile whose packed maximum is below thr has no hit.  Count: n
// grows by the hits of train rows j < n1 (columns past the set's end are copies of its last row, with the same dot).  Emit
// (out != nullptr): the hits are also written to out[n], in ascending train row, the row decoded from the column's code.
template <bool EMIT>
__device__ __forceinline__ void radius_tile(const uint32_t* rp, int tmax, int thr, int j0, int n1, int qrow, int4* out, int& n)
{
    if (tmax < thr) return;
#pragma unroll
    for (int u = 0; u < MT_BN / 2; ++u) {
        if (__vcmpges2(rp[u], (uint32_t)(thr & 0xFFFF) * 0x10001u) == 0u) continue;   // neither column of the pair is a hit
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int v = h ? (int)rp[u] >> 16 : (int)(rp[u] << 16) >> 16;
            if (v >= thr) {
                const AccRow d = acc_row<false>(v, j0, n1);
                if (d.j < n1) {
                    if (EMIT && out) out[n] = match_record(qrow, d.dot, d.j);
                    ++n;
                }
            }
        }
    }
}

// The packed accumulators of one tile (chunks past its UMMA N hold -32768) -> their maximum, after the operation's consumers
// have seen the tile: the top-k list, the radius hits, the cross-check column maxima (xc_slots: this warp's).
template <MatchOp OP, int KB>
__device__ __forceinline__ int epilogue_tile(const uint32_t* rp, int j0, int n1, int qrow, int (&list)[KB > 0 ? KB : 1], int rad_thr,
                                             int4* rad_out, int& rad_n, bool qvalid, int row_cta, int* xc_slots)
{
    unsigned p[8];                                           // eight independent max chains (ILP), then a short tree
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        p[u] = __vimax3_s16x2(rp[u], rp[8 + u], rp[16 + u]);
        p[u] = __vimax3_s16x2(p[u], rp[24 + u], rp[32 + u]);
        p[u] = __vmaxs2(p[u], rp[40 + u]);
    }
    const unsigned pk = __vimax3_s16x2(__vimax3_s16x2(p[0], p[1], p[2]), __vimax3_s16x2(p[3], p[4], p[5]), __vmaxs2(p[6], p[7]));
    const int k1 = max((int)(pk << 16) >> 16, (int)pk >> 16);
    if constexpr (OP == MatchOp::TopK) topk_tile<KB>(rp, k1, j0, n1, list);
    if constexpr (OP == MatchOp::RadiusCount || OP == MatchOp::RadiusEmit)
        radius_tile<OP == MatchOp::RadiusEmit>(rp, k1, rad_thr, j0, n1, qrow, rad_out, rad_n);
    if constexpr (OP == MatchOp::CrossCheck) xc_warp_columns(rp, qvalid, row_cta, xc_slots);
    return k1;
}

// SETQ = false: one query set (the map) shared by every train set; nq is its row count.
// SETQ = true (pairwise): set s has its own query rows, min(query_counts[s], nq) of them at query + s * nq * 32, so nq is
// the query stride and the pitch of the outputs and of the split keys.  The A tile then belongs to ONE set: the grid has
// gridDim.z = nsets (one (set, query tile) unit per CTA), and a CTA whose query tile is empty for its set exits before
// any setup -- in a CTA pair only when the leader's (lower) tile is empty too, because the peer holds half of every B tile.
// Outputs: with keys (train-row split) atomicMax of the packed row key, finalised by k_match_finalize; else records directly.
// TopK (k = knn_k <= KB): best receives k records per (set, query row), [nsets][nq][k].
// RadiusCount: rad_offsets[1 + L] = list L's length.  RadiusEmit: rad_offsets holds the scanned offsets, and list L's hits
// go to best[rad_offsets[L] ..] in ascending train row when rad_offsets[L + 1] <= rad_cap.
template <MatchOp OP, bool PAIR, bool SETQ, int KB>
__device__ __forceinline__ void hamming_umma_body(const MatchArgs& args)
{
    static_assert(!PAIR || match_op_pairs(OP), "top-k and radius run on the single-CTA kernel alone");
    static_assert((OP == MatchOp::TopK) == (KB > 0), "KB is the top-k list capacity");
    constexpr bool KNN2 = OP == MatchOp::Knn2, XCHK = OP == MatchOp::CrossCheck;
    constexpr int RAD = OP == MatchOp::RadiusCount ? 1 : OP == MatchOp::RadiusEmit ? 2 : 0;
    const uint8_t* __restrict__ query = args.query;
    const uint8_t* __restrict__ train = args.train;
    const int* __restrict__ train_counts = args.train_counts;
    int4* __restrict__ best = args.best;
    int4* __restrict__ second = args.second;
    int* __restrict__ keys = args.keys;
    int* __restrict__ status = args.status;
    int* __restrict__ col_keys = args.col_keys;
    long long* __restrict__ rad_offsets = args.rad_offsets;
    const int nq = args.nq, nt = args.nt, train_stride_rows = args.train_stride_rows, nsets = args.nsets;
    const int rows_per_split = args.rows_per_split, knn_k = args.knn_k, rad_thr = args.rad_thr;
    const long long rad_cap = args.rad_cap;
    int nqv = nq;                                            // query rows present (padded rows q >= nqv are excluded)
    if constexpr (SETQ) {
        nqv = max(0, min(__ldg(args.query_counts + blockIdx.z), nq));
        if ((PAIR ? (int)(blockIdx.x & ~1u) : (int)blockIdx.x) * MT_QROWS >= nqv) return;
        query += (size_t)blockIdx.z * nq * 32;
    }
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bar0 = sbase + MT_SMEM_BAR;
    const uint32_t bar_full = bar0, bar_empty = bar0 + 8 * MT_STAGES, bar_tfull = bar0 + 16 * MT_STAGES, bar_tempty = bar_tfull + 16;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + MT_SMEM_BAR + 16 * MT_STAGES + 32);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int split = blockIdx.y;
    const int q0 = blockIdx.x * MT_QROWS;
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;     // pair: 0 = leader (issues the MMAs of the pair), 1 = peer
    constexpr int ROWS_CTA = PAIR ? MT2_HALF : MT_BN;        // rows of a B tile this CTA expands and holds
    constexpr uint32_t IDESC = PAIR ? MT2_IDESC : MT_IDESC;

    // ---- setup: barriers, TMEM, A tiles (expanded in registers and parked in tensor memory)
    if (tid == 0) {
        // one arrive per warp (same-address arrives serialise).  Pair: full / tempty are only used in the leader, the peer
        // arrives on them remotely, so they count both CTAs' warps
        for (int s = 0; s < MT_STAGES; ++s) { mbar_init(bar_full + 8 * s, (PAIR ? 2 : 1) * MT2_GROUP_WARPS); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, PAIR ? 16 : 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == MT_ISSUER_WARP) {
        tmem_alloc_all<PAIR>(smem_u32((const void*)tmem_slot));
    }
    for (int i = tid; i < (128 * 128 + MT_BN * 128) / 16; i += MT_THREADS) reinterpret_cast<uint4*>(smem + MT_SMEM_CA)[i] = make_uint4(0, 0, 0, 0);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // bias k-step operands: logical byte k = 0 of row r sits at (r / 8) * 1024 + (r % 8) * 128 + ((0 ^ (r % 8)) << 4)
    if (tid < 128) smem[MT_SMEM_CA + (tid >> 3) * 1024 + (tid & 7) * 128 + ((tid & 7) << 4)] = 1;
    else if (tid < 128 + ROWS_CTA) {                         // this CTA's rows of the bias B tile: local row i <-> code 95 - (ROWS_CTA * rank + i)
        const int i = tid - 128;
        smem[MT_SMEM_CB + (i >> 3) * 1024 + (i & 7) * 128 + ((i & 7) << 4)] = (uint8_t)(MT_BN - 1 - ((int)rank * ROWS_CTA + i));
    }
    const uint32_t tmem_base = *tmem_slot;
    bool ok = true;
    if (warp >= MT_EPI_WARP0 && warp < MT_EPI_WARP0 + 8) {   // thread <-> query row <-> TMEM lane (same mapping as the epilogue)
        const int q = q0 + ((warp - MT_EPI_WARP0) >> 2) * 128 + (warp & 3) * 32 + lane;
        uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
        if (q < nqv) {
            const uint4* p = reinterpret_cast<const uint4*>(query + (size_t)q * 32);
            lo = __ldg(p); hi = __ldg(p + 1);
        }
        const uint32_t w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
        const uint32_t ta = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + MT_TMEM_A + (uint32_t)((warp - MT_EPI_WARP0) >> 2) * 64u;
#pragma unroll
        for (int half = 0; half < 2; ++half) {               // 64 columns = K 256 int8, four per 32-bit column
            uint32_t r[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = pm127x4((w[(half * 32 + i) >> 3] >> (((half * 32 + i) & 7) * 4)) & 15u);
            tc_st32(ta + half * 32, r);
        }
        tc_wait_st();
    }
    fence_proxy_async_smem();                                // constant bias tiles (generic-proxy stores) -> visible to the tensor core
    tc_fence_before();
    group_sync<PAIR>();                                      // (pair: both CTAs) barriers initialised, TMEM allocated, A tiles parked
    tc_fence_after();
    // where "stage full" / "accumulators free" are signalled: the leader's barriers through the cluster address space, or simply the CTA's own
    const uint32_t lead_full = PAIR ? mapa_u32(bar_full, 0) : bar_full, lead_tempty = PAIR ? mapa_u32(bar_tempty, 0) : bar_tempty;

    if (warp < MT_EXP_WARPS) {
        // ================= expanders: one B-tile row per thread; raw rows arrive through a cp.async ring
        //                   MT_PREFETCH tiles ahead, so global-load latency never sits on the pipeline's critical path
        // 96 threads per group, two groups on alternate tiles.  Single CTA: one B-tile row (32 raw bytes) per thread.  Pair: a
        // tile of N rows is split between the CTAs -- rows [0, N/2) live in the leader's shared memory, [N/2, N) in the
        // peer's -- and two threads share a local row (one 16-byte K half each).
        const int grp = tid / MT_BN, tl = tid - grp * MT_BN;
        const int r = PAIR ? tl % MT2_HALF : tl, hk = PAIR ? tl / MT2_HALF : 0;      // local row, K half
        constexpr int PIECE = PAIR ? 16 : 32;                // raw bytes per thread and tile
        struct TileIter {
            int set, i; MatchSetRange rg;
        };
        auto seek = [&](TileIter& it) -> bool {              // make (set, i) name an existing tile, skipping empty sets
            while (it.set < nsets && it.i >= it.rg.ntiles) {
                it.set += gridDim.z; it.i = 0;
                if (it.set < nsets) it.rg = match_set_range(train_counts, it.set, nt, split, rows_per_split);
            }
            return it.set < nsets;
        };
        auto step = [&](TileIter& it) -> bool { if (it.set < nsets) ++it.i; return seek(it); };
        TileIter cur = {(int)blockIdx.z, 0, {0, 0, 0}};
        if (cur.set < nsets) cur.rg = match_set_range(train_counts, cur.set, nt, split, rows_per_split);
        seek(cur);
        for (int k = 0; k < grp; ++k) step(cur);             // group g owns tiles g, g + GROUPS, g + 2 GROUPS, ...
        TileIter ahead = cur;
        uint8_t* raw = smem + MT_SMEM_RAW + (grp * MT_PREFETCH * MT_BN + tl) * PIECE;
        auto fetch = [&](int slot) {                         // raw (half) row of the tile `ahead` names -> ring slot (own piece only)
            uint8_t* dst = raw + slot * (MT_BN * PIECE);
            if (ahead.set < nsets) {
                const int j0t = ahead.rg.n0 + ahead.i * MT_BN;
                const int nh = ((min(MT_BN, ahead.rg.n1 - j0t) + 31) & ~31) >> (PAIR ? 1 : 0);    // rows per CTA of this tile (UMMA N, halved for a pair)
                // rows past the set's end repeat the set's LAST row: a copy scores like the original but carries a smaller
                // index code, so it can never win -- and the epilogue needs no per-column masking
                const int j = min(j0t + (int)rank * nh + r, ahead.rg.n1 - 1);
                if (r < nh) {
                    const uint8_t* src = train + ((size_t)ahead.set * train_stride_rows + j) * 32 + hk * 16;
                    const uint32_t d = smem_u32(dst);
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
                    if (!PAIR) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + 16), "l"(src + 16) : "memory");
                } else {
                    reinterpret_cast<uint4*>(dst)[0] = make_uint4(0, 0, 0, 0);
                    if (!PAIR) reinterpret_cast<uint4*>(dst)[1] = make_uint4(0, 0, 0, 0);
                }
#pragma unroll 1
                for (int k = 0; k < MT_EXP_GROUPS; ++k) step(ahead);
            }
            asm volatile("cp.async.commit_group;" ::: "memory");   // one group per tile slot, empty or not
        };
#pragma unroll 1
        for (int k = 0; k < MT_PREFETCH; ++k) fetch(k);
        int t = grp, n = 0;                                  // global tile number (pipeline stage / phase), own tile count (ring slot)
        while (cur.set < nsets) {
            asm volatile("cp.async.wait_group %0;" ::"n"(MT_PREFETCH - 1) : "memory");
            const int slot = n % MT_PREFETCH;
            const uint4 cv = reinterpret_cast<const uint4*>(raw + slot * (MT_BN * PIECE))[0];
            uint4 cv2 = cv;
            if (!PAIR) cv2 = reinterpret_cast<const uint4*>(raw + slot * (MT_BN * PIECE))[1];
            fetch(slot);                                     // refill the slot just consumed
            const int s = t % MT_STAGES;
            const uint32_t ph = (uint32_t)(t / MT_STAGES) & 1u;
            if (!mbar_wait(bar_empty + 8 * s, ph ^ 1u)) { ok = false; break; }
            if (PAIR) expand_half_row(smem + MT_SMEM_B + s * MT_B_BYTES, MT2_HALF, r, hk, cv);
            else      expand_row(smem + MT_SMEM_B + s * MT_B_BYTES, MT_BN, r, cv, cv2);
            fence_proxy_async_smem();                        // every writer fences, then one lane arrives for the warp (on the leader's barrier)
            __syncwarp();
            if (lane == 0) bar_arrive_lead<PAIR>(lead_full + 8 * s);
#pragma unroll 1
            for (int k = 0; k < MT_EXP_GROUPS; ++k) step(cur);
            t += MT_EXP_GROUPS;
            ++n;
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else if ((warp == MT_ISSUER_WARP || warp == MT_ISSUER2_WARP) && rank == 0) {   // (pair: the leader issues for both CTAs)
        // ================= MMA issuers =================
        // The whole warp runs the loop so that every operand is computed in warp-uniform code (uniform registers, no
        // per-instruction ELECT / R2UR waterfall); one elected lane issues the tcgen05 instructions.
        // TWO issuer warps take alternate tiles (issuer g <-> tiles t = g mod 2 <-> accumulator buffer g): issuing blocks on
        // the short MMA queue for the whole tensor time of a tile, so a single issuer exposes its per-tile barrier waits,
        // commits and loop latency (~200 cycles of a ~1200-cycle tile period) as tensor-pipe idle time; with two, the next
        // tile's MMAs are already queued behind the current one's.
        const int issuer = warp == MT_ISSUER_WARP ? 0 : 1;
        const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
        const uint32_t sbu = __shfl_sync(0xffffffffu, sbase, 0);
        const uint64_t dca = umma_desc_sw128(sbu + MT_SMEM_CA), dcb = umma_desc_sw128(sbu + MT_SMEM_CB);
        int t = 0;
        bool ready_next = false;                             // barriers of tile t already observed complete (probed mid-tile)
        // (the row count of the NEXT set is loaded a whole set ahead: its global-load latency would otherwise stall the
        //  pipeline at every set boundary)
        int cnt_next = match_set_count(train_counts, min((int)blockIdx.z, nsets - 1), nt);
        for (int set = blockIdx.z; set < nsets && ok; set += gridDim.z) {
            const MatchSetRange rg = match_set_range_n(cnt_next, nt, split, rows_per_split);
            if (set + (int)gridDim.z < nsets) cnt_next = match_set_count(train_counts, set + (int)gridDim.z, nt);   // consumed at the next set boundary
            for (int i = 0; i < rg.ntiles; ++i, ++t) {
                if ((t & 1) != issuer) continue;              // the other issuer's tile
                const int s = t % MT_STAGES;
                const uint32_t ph = (uint32_t)(t / MT_STAGES) & 1u;
                const int b = t & 1;
                const uint32_t bph = (uint32_t)(t >> 1) & 1u;
                if (!ready_next) {
                    if (!mbar_wait(bar_tempty + 8 * b, bph ^ 1u)) { ok = false; break; }
                    if (!mbar_wait(bar_full + 8 * s, ph)) { ok = false; break; }
                }
                tc_fence_after();
                const uint32_t sb = sbu + MT_SMEM_B + s * MT_B_BYTES;
                const uint64_t db0 = umma_desc_sw128(sb);
                // A set's last tile usually holds fewer than MT_BN rows: issue it with the smallest UMMA N (multiple of 16)
                // that covers them -- tensor time is proportional to N.  Columns beyond keep stale values the epilogue
                // never reads (it bounds partial tiles by the row count).
                const int rows_here = min(MT_BN, rg.n1 - (rg.n0 + i * MT_BN));
                const uint32_t idesc = (IDESC & ~(0x3Fu << 17)) | ((uint32_t)(((rows_here + 31) & ~31) >> 3) << 17);
                // barriers of this issuer's NEXT tile, t + 2 (same pipelines, consecutive tile numbers even across set boundaries)
                const int s1 = (t + 2) % MT_STAGES, b1 = b;
                const uint32_t ph1 = (uint32_t)((t + 2) / MT_STAGES) & 1u, bph1 = (uint32_t)((t + 2) >> 1) & 1u;
#pragma unroll
                for (int a = 0; a < 2; ++a) {
                    if (elect_one()) {
                        const uint32_t d = tb + (uint32_t)((b * 2 + a) * MT_BN);
                        const uint32_t ta = tb + MT_TMEM_A + (uint32_t)a * 64u;
#pragma unroll
                        for (int ks = 0; ks < 8; ++ks) {      // K = 256 = 8 x UMMA_K(32 int8): 8 TMEM columns of A, 4 k-steps per 128-B swizzle atom of B
                            const uint64_t db = db0 + (uint64_t)(((ks >> 2) * (ROWS_CTA * 128) + (ks & 3) * 32) >> 4);   // start-address field, 16-byte units
                            umma_i8_ts<PAIR>(d, ta + (uint32_t)ks * 8u, db, idesc, ks > 0 ? 1u : 0u);
                        }
                        umma_i8<PAIR>(d, dca, dcb, idesc, 1u); // bias k-step: + row code in every row
                    }
                    // While the queued MMAs execute, probe the next tile's barriers so its issue can start without a wait.
                    // The probe sits AFTER the last MMA of the tile: issuing blocks on the MMA queue for most of the tile's
                    // tensor time, so by now the epilogue of tile t - 1 has usually handed its accumulators back.
                    if (a == 1) ready_next = mbar_test(bar_tempty + 8 * b1, bph1 ^ 1u) && mbar_test(bar_full + 8 * s1, ph1);
                }
                if (elect_one()) {
                    umma_commit<PAIR>(bar_empty + 8 * s);           // smem stage reusable once these MMAs retire (both CTAs' barriers)
                    umma_commit<PAIR>(bar_tfull + 8 * b);           // accumulators of this tile complete (both CTAs' barriers)
                }
                __syncwarp();
            }
        }
    } else if (warp >= MT_EPI_WARP0 && warp < MT_EPI_WARP0 + 8) {
        // ================= epilogue =================
        const int a = (warp - MT_EPI_WARP0) >> 2;            // A tile; the TMEM lane quarter is fixed by hardware to warp % 4
        const int qrow = q0 + a * 128 + (warp & 3) * 32 + lane;
        const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
        int t = 0;
        int cnt_next = match_set_count(train_counts, min((int)blockIdx.z, nsets - 1), nt);
        // XCHK: the epilogue warps meet at a named barrier once per tile, so after a timeout a warp keeps walking the tiles
        // (without waiting on the pipeline) and never leaves the others at that barrier
        for (int set = blockIdx.z; set < nsets && (XCHK || ok); set += gridDim.z) {
            const MatchSetRange rg = match_set_range_n(cnt_next, nt, split, rows_per_split);   // (next set's row count loaded a set ahead, as in the issuer)
            if (set + (int)gridDim.z < nsets) cnt_next = match_set_count(train_counts, set + (int)gridDim.z, nt);
            int m1 = INT_MIN, m2 = INT_MIN;
            int list[KB > 0 ? KB : 1];                       // top-k: this row's best keys, descending
#pragma unroll
            for (int r = 0; r < (KB > 0 ? KB : 1); ++r) list[r] = INT_MIN;
            int rad_n = 0;                                   // radius: this row's hits so far in the set
            int4* rad_out = nullptr;                         // emit pass: where they go (null: the list is past the cap)
            if constexpr (RAD == 2) {
                if (qrow < nqv) {
                    const size_t o = (size_t)set * nq + qrow;
                    if (rad_offsets[o + 1] <= rad_cap) rad_out = best + rad_offsets[o];
                }
            }
            for (int i = 0; i < rg.ntiles; ++i, ++t) {
                const int b = t & 1;
                const uint32_t bph = (uint32_t)(t >> 1) & 1u;
                if constexpr (XCHK) {
                    if (ok && !mbar_wait(bar_tfull + 8 * b, bph)) ok = false;
                    if (!ok) { xc_epilogue_sync(); continue; }
                } else {
                    if (!mbar_wait(bar_tfull + 8 * b, bph)) { ok = false; break; }
                }
                tc_fence_after();
                const int j0 = rg.n0 + i * MT_BN;
                const bool full = (j0 + MT_BN <= rg.n1);
                constexpr int NCH = MT_BN / 32;
                uint32_t r[NCH][32];
                const uint32_t tacc = tmem_base + lane_base + (uint32_t)((b * 2 + a) * MT_BN);
                int k1 = INT_MIN, k2 = INT_MIN;
                if (!KNN2 && full) {
                    // accumulator = 127 * dot + code lies in [-32512, 32607]: it fits in 16 bits, so the tile comes out of
                    // tensor memory packed two columns per register (half the registers, half the max operations), and every
                    // value of a row is distinct (distinct codes), so the packed maximum loses nothing
                    uint32_t rp[MT_BN / 2];
                    tc_ld32_pack16(tacc, rp);
                    tc_ld16_pack16(tacc + 64, rp + 32);
                    tc_wait_ld();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) bar_arrive_lead<PAIR>(lead_tempty + 8 * b);           // TMEM buffer back to the issuer BEFORE the reduction
                    k1 = epilogue_tile<OP, KB>(rp, j0, rg.n1, qrow, list, rad_thr, rad_out, rad_n, qrow < nqv, qrow - q0,
                                               reinterpret_cast<int*>(smem + MT_SMEM_XC) + (b * 8 + warp - MT_EPI_WARP0) * MT_BN);
                } else if (!KNN2) {
                    // a set's partial last tile was issued with N = 32, 64 (or 96) columns, its rows past the set's end are
                    // copies of the last row (never the maximum): same packed path, 32-column chunks as far as N goes
                    const int nch = (rg.n1 - j0 + 31) >> 5;
                    uint32_t rp[MT_BN / 2];
#pragma unroll
                    for (int ch = 0; ch < NCH; ++ch) {
                        if (ch < nch) tc_ld16_pack16(tacc + (uint32_t)(ch * 32), rp + ch * 16);
                        else {
#pragma unroll
                            for (int u = 0; u < 16; ++u) rp[ch * 16 + u] = 0x80008000u;
                        }
                    }
                    tc_wait_ld();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) bar_arrive_lead<PAIR>(lead_tempty + 8 * b);
                    k1 = epilogue_tile<OP, KB>(rp, j0, rg.n1, qrow, list, rad_thr, rad_out, rad_n, qrow < nqv, qrow - q0,
                                               reinterpret_cast<int*>(smem + MT_SMEM_XC) + (b * 8 + warp - MT_EPI_WARP0) * MT_BN);
                } else {
#pragma unroll
                    for (int ch = 0; ch < NCH; ++ch) tc_ld32(tacc + (uint32_t)(ch * 32), r[ch]);
                    tc_wait_ld();
                    // The accumulators now live in registers: hand the TMEM buffer back to the issuer BEFORE the max
                    // reduction, so the epilogue's arithmetic overlaps the MMAs of tile t + 2 instead of gating them.
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) bar_arrive_lead<PAIR>(lead_tempty + 8 * b);
#pragma unroll
                    for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
                        for (int c = 0; c < 32; ++c)
                            if (full || j0 + ch * 32 + c < rg.n1) {
                                const int k = (int)r[ch][c];
                                if (KNN2) k2 = max(k2, min(k1, k));
                                k1 = max(k1, k);
                            }
                }
                // decode the tile winner(s) into the global row key (top-k: already in the list; radius: nothing to keep)
#pragma unroll
                for (int w = 0; w < (KNN2 ? 2 : match_op_pairs(OP) ? 1 : 0); ++w) {
                    const int k = w == 0 ? k1 : k2;
                    if (k != INT_MIN) {
                        const AccRow d = acc_row<PAIR>(k, j0, rg.n1);
                        const int gk = row_key(d.dot, d.j);
                        if (KNN2) m2 = max(m2, min(m1, gk));
                        m1 = max(m1, gk);
                    }
                }
                if constexpr (XCHK) {
                    // the 8 warps' maxima of a column -> the CTA's, decoded like a row winner (the code names the train row,
                    // whatever the column's slot) into the column key  dot << 20 | (0xFFFFF - q); one atomicMax per column.
                    // Slots of buffer b are written again at tile t + 2, behind the next tile's barrier.
                    xc_epilogue_sync();
                    const int e = tid - MT_EPI_WARP0 * 32;
                    if (e < MT_BN) {
                        const int* xcs = reinterpret_cast<const int*>(smem + MT_SMEM_XC) + b * 8 * MT_BN + e;
                        int kx = xcs[0];
#pragma unroll
                        for (int w = 1; w < 8; ++w) kx = max(kx, xcs[w * MT_BN]);
                        const int v = kx >> 8;
                        if (v != -32768) {                   // (only padded query rows, or a chunk past the tile's N)
                            const AccRow d = acc_row<PAIR>(v, j0, rg.n1);
                            if (d.j < rg.n1)                 // columns past the set's end are copies of its last row
                                atomicMax(&col_keys[(size_t)set * train_stride_rows + d.j],
                                          d.dot * (1 << MT_KEY_SHIFT) + ((MT_MAX_QUERY_XC - 1) - (q0 + 255 - (kx & 255))));
                        }
                    }
                }
            }
            if (ok && qrow < nqv) {
                const size_t o = (size_t)set * nq + qrow;
                if constexpr (RAD > 0) {                    // count pass: the list's length (the emit pass has written its hits)
                    if constexpr (RAD == 1) rad_offsets[1 + o] = rad_n;
                } else if constexpr (KB > 0) {              // the k records of this row, once per set
                    int4* out = best + o * knn_k;
#pragma unroll
                    for (int r = 0; r < KB; ++r) {
                        if (r >= knn_k) break;
                        out[r] = key_record(qrow, list[r]);
                    }
                } else if (keys) {
                    if (m1 != INT_MIN) atomicMax(&keys[o], m1);
                } else {                                     // (an empty train set: trainIdx -1)
                    best[o] = key_record(qrow, m1);
                    if (KNN2) second[o] = key_record(qrow, m2);
                }
            }
        }
    }
    if (!ok) atomicOr(status, 2);
    tc_fence_before();
    group_sync<PAIR>();                                      // (pair: neither CTA may free tensor memory or exit while the other still works)
    if (warp == MT_ISSUER_WARP) {
        tc_fence_after();
        tmem_dealloc_all<PAIR>(tmem_base);
    }
}


// The matcher kernels: the body for one operation (see MatchOp; CrossCheck is launched with MT_SMEM_BYTES_XC), shared query
// or pairwise (SETQ: set s's own query rows against train set s, gridDim.z = nsets), and KB: TopK's list capacity.
// Single CTA per query tile (small problems: independent CTAs, train rows can be split across them): every operation.
template <MatchOp OP, bool SETQ, int KB = 0>
__global__ void __launch_bounds__(MT_THREADS, 1) k_hamming_umma(const __grid_constant__ MatchArgs args)
{
    hamming_umma_body<OP, false, SETQ, KB>(args);
}
// CTA pair on the two SMs of a TPC (tcgen05 cta_group::2): blockIdx.x = 2 * pair + rank; Best, Knn2 and CrossCheck
template <MatchOp OP, bool SETQ>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MT_THREADS, 1) k_hamming_umma2(const __grid_constant__ MatchArgs args)
{
    hamming_umma_body<OP, true, SETQ, 0>(args);
}

// ONE CTA per set: query i keeps its best match (i, j) iff column j's key names i, i.e. i is also train row j's nearest
// query (lowest index on ties); the kept records are compacted stably in query order to out[set][0 .. n_out[set]).
// best and out may be the same buffer: a record only moves to a lower or equal index, and a chunk is read before it is written.
// Sets are nq records apart; set s holds min(query_counts[s], nq) query rows (pairwise), or all nq (query_counts null).
constexpr int XC_NT = 1024;
__global__ void __launch_bounds__(XC_NT) k_crosscheck_compact(const int4* best, int nq, const int* __restrict__ query_counts,
                                                              const int* __restrict__ col_keys, int stride_rows, int4* out, int* __restrict__ n_out)
{
    __shared__ int s_warp[XC_NT / 32];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const size_t set = blockIdx.x;
    const int nrows = query_counts ? max(0, min(__ldg(query_counts + set), nq)) : nq;
    best += set * nq; out += set * nq; col_keys += set * stride_rows;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int base = 0; base < nrows; base += XC_NT) {
        const int i = base + tid;
        int4 r = make_int4(0, -1, 0, 0);
        if (i < nrows) r = best[i];
        const bool keep = r.y >= 0 && (MT_MAX_QUERY_XC - 1) - (col_keys[r.y] & (MT_MAX_QUERY_XC - 1)) == i;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[wid] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < XC_NT / 32; ++w) { const int c = s_warp[w]; if (w < wid) before += c; total += c; }
        const int out0 = s_base;
        if (keep) out[out0 + before + __popc(bal & ((1u << lane) - 1u))] = r;
        __syncthreads();
        if (tid == 0) s_base = out0 + total;
        __syncthreads();
    }
    if (tid == 0) n_out[set] = s_base;
}

__global__ void k_match_keys_init(int* __restrict__ keys, size_t n)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = INT_MIN;
}

// split keys -> DMatch record i of [n / nq][nq]; with query_counts (pairwise) only the min(query_counts[s], nq) rows of set
// s, the record slots past that count left as they are
__global__ void k_match_finalize(const int* __restrict__ keys, int nq, const int* __restrict__ query_counts, size_t n, int4* __restrict__ best)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || (query_counts && (int)(i % (size_t)nq) >= __ldg(query_counts + i / (size_t)nq))) return;
    best[i] = key_record((int)(i % (size_t)nq), keys[i]);
}

}  // namespace orbx
