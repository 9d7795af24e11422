// orbx_device.cuh -- device primitives shared by more than one stage header, sm_100a.  A helper that only one stage uses
// lives in that stage's header.
//
// One header per stage of cv::ORB::detectAndCompute (src/frontend.cpp:153) and one for the matcher:
//   orbx_pyr.cuh     A.1 gray, A.2 pyramid           orbx_select.cuh  A.4-6 retainBest(2n) -> Harris -> retainBest(n)
//   orbx_fast.cuh    A.3 FAST + NMS                  orbx_desc.cuh    A.8 blur, A.7 / A.9 / A.10 describe
//   orbx_match.cuh   A.11 brute-force Hamming matcher (tcgen05)
// Stage arithmetic follows SURVEY.md Appendix A and is bit-exact against OpenCV: integer stages in integer arithmetic, float
// stages with explicit round-to-nearest intrinsics (never contracted) and __fmaf_rn only where OpenCV's own build uses FMA (A.8).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace orbx {

__device__ __forceinline__ unsigned lanemask_lt() { unsigned m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }

// cp.async (LDGSTS): global -> shared copies that cost neither registers nor scoreboards while in flight (a warp has six
// scoreboards; a deep register-prefetch pipeline ends up sharing them and the oldest load waits for the youngest).
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }
__device__ __forceinline__ unsigned lds_u32(unsigned addr) { unsigned v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v; }
__device__ __forceinline__ unsigned lds_u8(unsigned addr) { unsigned v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v; }
__device__ __forceinline__ void sts_u8(unsigned addr, unsigned v) { asm volatile("st.shared.u8 [%0], %1;" :: "r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ uint4 lds_v4(unsigned addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}

// ---- mbarriers and TMA
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
// Bounded wait: returns false after ~0.25 s so that a protocol bug ends the kernel instead of hanging the GPU.
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity) {
    unsigned long long t0 = 0;
    for (uint32_t it = 0;; ++it) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return true;
        if ((it & 1023u) == 1023u) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t0 == 0) t0 = t;
            else if (t - t0 > 250000000ull) return false;
        }
    }
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar_s, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar_s), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_tile_3d(unsigned dst_s, const CUtensorMap* map, int x, int y, int z, unsigned bar_s)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 :: "r"(dst_s), "l"(map), "r"(x), "r"(y), "r"(z), "r"(bar_s) : "memory");
}

}  // namespace orbx
