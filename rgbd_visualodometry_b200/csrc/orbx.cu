// orbx.cu -- host side of liborbx.so: context, device-memory layout, kernel launches and the C-ABI of include/orbx.h.
//
// The two operator calls of the reference front-end that this library stands in for:
//   cv::ORB::detectAndCompute            src/frontend.cpp:153   -> orbx_detect_and_compute*
//   cv::DescriptorMatcher::match         src/frontend.cpp:187   -> orbx_match_hamming*
// There is no CPU fallback anywhere in this file: every entry point either runs the sm_100a kernels or fails.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <float.h>
#include <limits.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <memory>
#include <new>
#include <string>
#include <vector>

#include "../../include/orbx.h"
#include "orbx_geom.h"
#include "orbx_pyr.cuh"
#include "orbx_fast.cuh"
#include "orbx_select.cuh"
#include "orbx_desc.cuh"
#include "orbx_match.cuh"
#include "orbx_radius.cuh"
#include "orbx_map.cuh"
#include "orbx_stage.h"
#include <unordered_map>

using namespace orbx;

namespace {

const int8_t k_pattern_host[256 * 4] = {
#include "brief_pattern.inc"
};

constexpr int FAST_R = 16, FAST_NT = 256;
constexpr int FAST_NWARP = 4;             // warps per CTA of k_fast_warp (independent units; 7 CTAs per SM by shared memory)
static_assert(FAST_R == FW_R, "band height");
constexpr int HOST_LANES = 8;              // host-buffer calls: more, shorter ranges shrink the un-overlapped head (first upload) and tail
constexpr int HOST_LANE_MIN_FRAMES = 16;   // host-buffer batches: lanes mainly overlap PCIe copies with kernels
constexpr long SIDE_LEVEL_MAX_PX = 100000; // pyramid levels (from level 2 on) below this many pixels run on the side stream
constexpr size_t STAGE_WAKE_BYTES = (size_t)2 << 20;   // staged copies of at least this many bytes wake the copier threads
constexpr int N_STAGES = 7;
const char* const k_stage_names[N_STAGES] = {"gray", "pyramid", "fast_nms", "select_harris", "blur", "describe", "match"};
constexpr int MATCH_WORDS = 16;           // matcher status words (mstatus), one per slot: lane k of a host-buffer batch uses slot k

size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// NVTX ranges around every stage's launches and around the C-ABI calls (the reference's only timer is the wall clock around
// AddFrame, app/run_vo.cpp:104-109); header-only NVTX 3: free when no tool is attached.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};
struct NvtxStages {                      // one open range at a time: next() closes the previous stage's
    bool open = false;
    void next(const char* name) { if (open) nvtxRangePop(); nvtxRangePushA(name); open = true; }
    ~NvtxStages() { if (open) nvtxRangePop(); }
};

// The context's CUDA resources, each released by its owner's destructor (none of these throws).
template <class T, cudaError_t (*release)(void*)>
struct Mem {                                 // move-only, so that a grown table column can replace the old one
    T* p = nullptr;
    size_t bytes = 0;
    Mem() = default;
    Mem(Mem&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
    Mem& operator=(Mem&& o) noexcept { std::swap(p, o.p); std::swap(bytes, o.bytes); o.reset(); return *this; }
    ~Mem() { reset(); }
    void reset() { if (p) release(p); p = nullptr; bytes = 0; }
};
using Buf = Mem<void, cudaFree>;             // device memory
using HostBuf = Mem<uint8_t, cudaFreeHost>;  // pinned host memory

template <class H, cudaError_t (*destroy)(H)>
struct Handle {                              // a stream or an event
    H h = nullptr;
    Handle() = default;
    Handle(const Handle&) = delete;
    Handle& operator=(const Handle&) = delete;
    ~Handle() { if (h) destroy(h); }
    operator H() const { return h; }
};
using Stream = Handle<cudaStream_t, cudaStreamDestroy>;
using Event = Handle<cudaEvent_t, cudaEventDestroy>;

}  // namespace

// Members are released in reverse order of declaration, after orbx_destroy has synchronized every stream: the stager
// goes first, so its threads are joined before the pinned staging they copy into is freed, and the streams go last.
struct orbx_ctx {
    Stream stream;
    Stream lane[HOST_LANES];                 // extra frame-range pipelines (lane 0 is `stream`)
    Stream side[HOST_LANES];                 // per lane: high-priority stream of the small pyramid levels + their FAST bands
    Event ev[N_STAGES + 2];                  // 0..6 bracket the six extraction stages, 7..8 the matcher
    Event ev_sfork[HOST_LANES], ev_sjoin[HOST_LANES];
    Event ev_fork, ev_join[HOST_LANES];

    int device = 0, nfeatures = 0, nlevels = 0, max_w = 0, max_h = 0, max_batch = 0;
    float scale_factor = 1.2f;
    std::string err;
    uint64_t launches = 0;

    Geom geom{};             // geometry of the current frame size
    FastMaps fmaps{};        // TMA tensor maps (x, y, frame) of the pyramid levels for the current geometry
    PyrMaps pmaps{};         // ... of every level as the SOURCE of the next one (k_pyr_tma boxes)
    DescMaps dmaps{};        // ... of every pyramid / blurred level with k_describe_tma's window boxes
    Geom geom_max{};         // geometry of (max_w, max_h): sizes the buffers
    int geom_w = 0, geom_h = 0;
    size_t tabs_len = 0;

    Buf pyr, blur, rowcnt, rowent, work, selpos, fincnt, selcnt, status, tabs, pattern;
    Buf in, kps, desc, counts;               // host-path staging on the device
    int out_cap = 0;
    const uint8_t* view_desc = nullptr;      // device descriptors / counts of the frames the last host call (or collect) produced
    const int* view_counts = nullptr;
    int view_frames = 0;
    Buf mq, mt, mbest, msecond, mkeys, mstatus, mcounts;
    Buf mcolkeys, mxcount;                   // cross-check: column keys [nsets][stride_rows], the host form's pair count
    Buf mradoff, mradsums;                   // radius: the host form's offsets, the offsets scan's tile sums
    int last_batch = 0;

    // device-resident map-point table (SURVEY 8(f).1): slot-addressed columns + the host's id -> slot index
    Buf t_desc, t_pos, t_nrm, t_outl, t_slots, t_cand, t_ncand, t_q, t_in, t_best, t_filtered, t_minmax, t_aux;
    int map_capacity = 0;
    std::unordered_map<long long, int> map_slot;
    std::vector<int> map_free;
    int map_next = 0;

    // asynchronous single-frame pipeline (orbx_submit_frame / orbx_collect_frame): two slots of pinned host staging and
    // device outputs, so the host can prepare / consume one frame while the GPU works on the other
    struct AsyncSlot {
        Event done;
        Buf d_kps, d_desc, d_counts;
        HostBuf h_in;
        HostBuf h_out;                       // [counts 16 B][status 16 B][kps cap*28][desc cap*32]
        int cap = 0;
        bool busy = false;
    } aslot[2];
    int a_head = 0, a_inflight = 0;          // oldest in-flight slot, number in flight

    bool profiling = false;
    int force_kernels = -1;                   // orbx_debug_force_kernels: -1 by launch size, 0 warp-private TMA kernels, 1 CTA-cooperative kernels
    float stage_ms[N_STAGES] = {};
    bool stage_valid[N_STAGES] = {};

    // Pinned words the synchronous entry points read back, in ints: [counts][status][match]
    //   counts  max(max_batch, 3)  per-frame keypoint counts; orbx_track_match's candidate / match count and distance bounds
    //   status  max_batch          per-frame device status
    //   match   MATCH_WORDS        copies of the matcher status words
    HostBuf h_small;
    size_t h_small_bytes() const { return sizeof(int) * (std::max(max_batch, 3) + max_batch + MATCH_WORDS); }
    int* h_counts() const { return (int*)h_small.p; }
    int* h_status() const { return h_counts() + std::max(max_batch, 3); }
    int* h_match() const { return h_status() + max_batch; }
    HostBuf h_stage_in;                      // pinned staging of pageable caller frames (device layout)
    HostBuf h_stage_out;                     // ... of results bound for pageable caller buffers
    std::unique_ptr<HostStager> stager;      // copier threads, created by the first call that needs them

    void synchronize_streams() const
    {
        cudaStreamSynchronize(stream);
        for (int k = 1; k < HOST_LANES; ++k) cudaStreamSynchronize(lane[k]);
        for (const Stream& s : side) cudaStreamSynchronize(s);
    }
};

namespace {

int fail(orbx_ctx* c, int code, const char* fmt, const char* a = "", const char* b = "")
{
    if (c) {
        char buf[512];
        snprintf(buf, sizeof buf, fmt, a, b);
        c->err = buf;
    }
    return code;
}

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) return fail(c, ORBX_E_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

int ensure(orbx_ctx* c, Buf& b, size_t bytes)
{
    if (b.bytes >= bytes && b.p) return ORBX_OK;
    b.reset();
    bytes = std::max<size_t>(bytes, 256);
    cudaError_t e = cudaMalloc(&b.p, bytes);
    if (e != cudaSuccess) return fail(c, ORBX_E_NOMEM, "cudaMalloc failed: %s", cudaGetErrorString(e));
    b.bytes = bytes;
    return ORBX_OK;
}

int ensure(orbx_ctx* c, HostBuf& b, size_t bytes, const char* what)
{
    if (b.bytes >= bytes && b.p) return ORBX_OK;
    b.reset();
    bytes = std::max<size_t>(bytes, 4096);
    if (cudaMallocHost((void**)&b.p, bytes) != cudaSuccess) { cudaGetLastError(); return fail(c, ORBX_E_NOMEM, "%s", what); }
    b.bytes = bytes;
    return ORBX_OK;
}

// ---- geometry (SURVEY A.2 / A.4), identical arithmetic to OpenCV: float scale chain, cvRound sizes, float quotas
void level_sizes(int w, int h, int nlevels, float sf, int* ws, int* hs, float* sc)
{
    for (int l = 0; l < nlevels; ++l) {
        const float s = (float)pow((double)sf, (double)l);
        const float inv = 1.0f / s;
        sc[l] = s;
        ws[l] = (int)lrintf((float)w * inv);
        hs[l] = (int)lrintf((float)h * inv);
    }
}

void level_quotas(int nfeatures, float sf, int nlevels, int* q)
{
    const float factor = (float)(1.0 / (double)sf);
    const float one_minus = 1.0f - factor;
    const float num = (float)nfeatures * one_minus;
    const float den = 1.0f - (float)pow((double)factor, (double)nlevels);
    float nd = num / den;
    int sum = 0;
    for (int l = 0; l < nlevels - 1; ++l) {
        q[l] = (int)lrintf(nd);
        sum += q[l];
        nd = nd * factor;
    }
    q[nlevels - 1] = std::max(nfeatures - sum, 0);
}

// INTER_LINEAR_EXACT taps of one axis, packed i0 | c1 << 16 (c1 in 8.8 fixed point, c0 = 256 - c1)
void resize_taps(int s, int d, uint32_t* out)
{
    const double inv_scale = (double)d / (double)s;
    const double scale = 1.0 / inv_scale;
    for (int x = 0; x < d; ++x) {
        const double f = scale * ((double)x + 0.5) - 0.5;
        const int i = (int)floor(f);
        uint32_t i0, c1;
        if (i < 0 || s <= 1) { i0 = 0; c1 = 0; }
        else if (i >= s - 1) { i0 = (uint32_t)(s - 1); c1 = 0; }
        else { i0 = (uint32_t)i; c1 = (uint32_t)lrint((f - (double)i) * 256.0); }
        out[x] = i0 | (c1 << 16);
    }
}

void build_geom(const orbx_ctx* c, int w, int h, Geom* g, std::vector<uint32_t>* tabs)
{
    memset(g, 0, sizeof *g);
    int ws[ORBX_LEVELS_MAX], hs[ORBX_LEVELS_MAX], q[ORBX_LEVELS_MAX];
    float sc[ORBX_LEVELS_MAX];
    level_sizes(w, h, c->nlevels, c->scale_factor, ws, hs, sc);
    level_quotas(c->nfeatures, c->scale_factor, c->nlevels, q);
    g->nlevels = c->nlevels; g->w = w; g->h = h; g->band_rows = FAST_R;
    size_t pyr = 0, cnt = 0, ent = 0, wsz = 0, tab = 0;
    int bands = 0, blurs = 0, hblks = 0, selh = 64;
    for (int l = 0; l < c->nlevels; ++l) {
        LevelGeom& L = g->L[l];
        L.w = std::max(ws[l], 0); L.h = std::max(hs[l], 0);
        L.pitch = (int)round_up((size_t)std::max(L.w, 1), 16);
        L.quota = q[l]; L.scale = sc[l];
        L.in_w = std::max(L.w - 2 * ORBX_EDGE, 0); L.in_h = std::max(L.h - 2 * ORBX_EDGE, 0);
        if (L.in_w == 0 || L.in_h == 0) { L.in_w = 0; L.in_h = 0; }
        L.ent_pitch = (int)round_up((size_t)(L.in_w + 1) / 2 + 1, 8);
        L.ws_cap = std::max(((L.in_w + 1) / 2) * ((L.in_h + 1) / 2), 1);
        L.band0 = bands; L.nbands = (L.in_h + FAST_R - 1) / FAST_R; bands += L.nbands;
        if (L.in_w > 0) {                                    // blur work items: 8-column groups x strips of blur_rh rows, BLUR_NT per CTA
            L.blur_cgs = (L.w - 13 - BLUR_LO + 7) / 8;
            // strip height: a multiple of 7 (the kernel's unrolled row window) that wastes the fewest rows on this level
            const int rows = L.h - 26;
            long best = -1;
            for (int rh = 35; rh <= 84; rh += 7) {
                const long cost = (long)((rows + rh - 1) / rh) * (rh + 6);
                if (best < 0 || cost < best) { best = cost; L.blur_rh = rh; }
            }
            L.nblur = (L.blur_cgs * ((rows + L.blur_rh - 1) / L.blur_rh) + BLUR_NT - 1) / BLUR_NT;
        }
        L.blur0 = blurs; blurs += L.nblur;
        L.hblk0 = hblks; L.hblk = (2 * L.quota * 5 / 4 + 32 + HARRIS_NT - 1) / HARRIS_NT; hblks += L.hblk;
        selh = std::max(selh, 2 * L.quota * 5 / 4 + 64);
        L.img_off = pyr; pyr += round_up((size_t)L.pitch * std::max(L.h, 1), 256);
        L.cnt_off = cnt; cnt += round_up((size_t)std::max(L.in_h, 1), 8);
        L.ent_off = ent; ent += (size_t)L.ent_pitch * std::max(L.in_h, 1);
        L.ws_off = wsz; wsz += round_up((size_t)L.ws_cap, 4);
        if (l > 0) { L.xtab = (uint32_t)tab; tab += L.w; L.ytab = (uint32_t)tab; tab += L.h; }
    }
    g->total_bands = bands; g->total_blur = blurs; g->total_hblk = hblks;
    g->selh_elems = std::min((selh + 63) / 64 * 64, 16384);
    g->pyr_frame = round_up(pyr, 256); g->cnt_frame = cnt; g->ent_frame = ent; g->ws_frame = wsz;
    if (tabs) {
        tabs->assign(std::max<size_t>(tab, 1), 0);
        for (int l = 1; l < c->nlevels; ++l) {
            const LevelGeom& L = g->L[l];
            const LevelGeom& S = g->L[l - 1];
            if (L.w > 0 && L.h > 0 && S.w > 0 && S.h > 0) {
                resize_taps(S.w, L.w, tabs->data() + L.xtab);
                resize_taps(S.h, L.h, tabs->data() + L.ytab);
                int span = 0;                                // how far a thread's 4 outputs reach from its aligned first source byte
                for (int x = 0; x < L.w; x += 4) {
                    const int a = (int)((*tabs)[L.xtab + x] & 0xffffu) & ~3;
                    const int xl = std::min(x + 3, L.w - 1);
                    span = std::max(span, (int)((*tabs)[L.xtab + xl] & 0xffffu) - a);
                }
                g->L[l].xspan = span;
                // k_pyr_tma: a lane's 4 outputs must read at most 7 consecutive source bytes, and the source box of a
                // (128-column tile, 16-row strip) must fit a TMA box (<= 256 per dimension, 16-byte aligned first column)
                LevelGeom& D = g->L[l];
                const uint32_t* xt = tabs->data() + D.xtab;
                const uint32_t* yt = tabs->data() + D.ytab;
                int quad_span = 0, bw = 0, bh = 0;
                for (int x = 0; x < D.w; x += 4)
                    quad_span = std::max(quad_span, (int)(xt[std::min(x + 3, D.w - 1)] & 0xffffu) - (int)(xt[x] & 0xffffu));
                D.pt_ncx = (D.pitch + PT_CW - 1) / PT_CW;
                for (int cx = 0; cx < D.pt_ncx; ++cx) {
                    const int xl = std::min(cx * PT_CW + PT_CW - 1, D.w - 1);
                    const int X0 = (int)(xt[cx * PT_CW] & 0xffffu) & ~15;
                    bw = std::max(bw, (int)(xt[xl] & 0xffffu) + 2 - X0);
                }
                const int nstrips = (D.h + PT_RH - 1) / PT_RH;
                for (int st = 0; st < nstrips; ++st) {
                    const int ye = std::min(st * PT_RH + PT_RH, D.h);
                    bh = std::max(bh, std::min((int)(yt[ye - 1] & 0xffffu) + 1, S.h - 1) - (int)(yt[st * PT_RH] & 0xffffu) + 1);
                }
                D.pt_bw = (int)round_up((size_t)bw, 16); D.pt_bh = bh;
                D.pt_k = 4;
                D.pt_ntask = D.pt_ncx * ((nstrips + D.pt_k - 1) / D.pt_k);
                D.pt_ok = quad_span <= 6 && D.pt_bw <= 256 && D.pt_bh <= 256 && PT_NWARP * pt_warp_bytes(D.pt_bw, D.pt_bh) + 128 <= 160 * 1024;
            }
        }
    }
}

typedef CUresult (*enc_t)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                          CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// A 3-D u8 tensor map (x = pitch, y = rows, z = frame) over level L of `base` (the pyramid or the blurred pyramid, one
// frame every g.pyr_frame bytes) with boxes of bw x bh x 1; the hardware zero-fills the parts of a box outside the level.
bool encode_level(enc_t enc, const orbx_ctx* c, CUtensorMap* m, const Buf& base, const LevelGeom& L, int bw, int bh)
{
    const cuuint64_t dims[3] = {(cuuint64_t)L.pitch, (cuuint64_t)L.h, (cuuint64_t)c->max_batch};
    const cuuint64_t strides[2] = {(cuuint64_t)L.pitch, (cuuint64_t)c->geom.pyr_frame};
    const cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, 1}, es[3] = {1, 1, 1};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (uint8_t*)base.p + L.img_off, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// The tensor maps of the current geometry: k_fast_warp's image tiles (FW_TP x FW_TR boxes of every pyramid level),
// k_pyr_tma's source boxes (each level as the source of the next) and k_describe_tma's windows (pyramid and blurred levels).
int build_fast_maps(orbx_ctx* c)
{
    static enc_t enc = nullptr;
    if (!enc) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) != cudaSuccess || !fn)
            return fail(c, ORBX_E_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
        enc = (enc_t)fn;
    }
    const Geom& g = c->geom;
    memset(&c->fmaps, 0, sizeof c->fmaps);
    for (int l = 0; l < g.nlevels; ++l) {
        const LevelGeom& L = g.L[l];
        if (L.nbands <= 0 || L.in_w <= 0) continue;
        if (!encode_level(enc, c, &c->fmaps.m[l], c->pyr, L, FW_TP, FW_TR)) return fail(c, ORBX_E_CUDA, "cuTensorMapEncodeTiled failed for a pyramid level");
    }
    memset(&c->pmaps, 0, sizeof c->pmaps);
    for (int l = 1; l < g.nlevels; ++l) {
        const LevelGeom& D = g.L[l];
        if (D.pt_ok && !encode_level(enc, c, &c->pmaps.m[l], c->pyr, g.L[l - 1], D.pt_bw, D.pt_bh))
            return fail(c, ORBX_E_CUDA, "cuTensorMapEncodeTiled failed for a pyramid source level");
    }
    memset(&c->dmaps, 0, sizeof c->dmaps);
    for (int l = 0; l < g.nlevels; ++l) {
        const LevelGeom& L = g.L[l];
        if (L.in_w <= 0) continue;
        if (!encode_level(enc, c, &c->dmaps.ic[l], c->pyr, L, DS_ICW, DS_ICH) || !encode_level(enc, c, &c->dmaps.bl[l], c->blur, L, DS_BLW, DS_BLH))
            return fail(c, ORBX_E_CUDA, "cuTensorMapEncodeTiled failed for a descriptor window map");
    }
    return ORBX_OK;
}

// The cached size (geom_w, geom_h) is cleared first and stored last, so a failure anywhere in between leaves a context
// that rebuilds its geometry, tap table and tensor maps on the next call.
int set_geometry(orbx_ctx* c, int w, int h)
{
    if (c->geom_w == w && c->geom_h == h) return ORBX_OK;
    c->geom_w = c->geom_h = -1;
    std::vector<uint32_t> tabs;
    build_geom(c, w, h, &c->geom, &tabs);
    for (int l = 1; l < c->nlevels; ++l)
        if (c->geom.L[l].xspan > 11) return fail(c, ORBX_E_UNSUPPORTED, "scale_factor too large for the pyramid kernels (4 outputs must span <= 12 source bytes: about 2.6)");
    int rc = ensure(c, c->tabs, tabs.size() * 4);
    if (rc) return rc;
    CU(cudaMemcpyAsync(c->tabs.p, tabs.data(), tabs.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));       // `tabs` is a local
    if ((rc = build_fast_maps(c))) return rc;
    c->geom_w = w; c->geom_h = h;
    return ORBX_OK;
}

void stage_mark(orbx_ctx* c, int i)
{
    if (c->profiling) cudaEventRecord(c->ev[i], c->stream);
}

// The extraction pipeline on device-resident frames; everything asynchronous on c->stream.
// Frame range of host-buffer lane k.  The ranges taper towards both ends (weights 1, 2, 4, 4, ..., 4, 2, 1): the first
// upload has nothing to hide under and the last range's kernels + download have nothing left to hide, so both are short.
static void host_lane_range(int batch, int lanes, int k, int* f0, int* f1)
{
    auto wgt = [&](int i) { return 1 << std::min(2, std::min(i, lanes - 1 - i)); };
    long tot = 0, before = 0;
    for (int i = 0; i < lanes; ++i) { tot += wgt(i); if (i < k) before += wgt(i); }
    *f0 = (int)((long)batch * before / tot);
    *f1 = (int)((long)batch * (before + wgt(k)) / tot);
}

// The kernel sequence for frames [f0, f0 + nb) on stream `st`.  Every buffer is frame-major, so a frame range is
// just a base-pointer offset.
int run_extract_range(orbx_ctx* c, cudaStream_t st, int lane_id, bool marks, int f0, int nb,
                      const uint8_t* d_imgs, size_t step, size_t frame_stride, int channels, float* d_kps, uint8_t* d_desc, int cap,
                      int* d_counts)
{
    const Geom& g = c->geom;
    const size_t F = (size_t)f0;
    d_imgs += F * frame_stride;
    uint8_t* pyr = (uint8_t*)c->pyr.p + F * g.pyr_frame;
    uint8_t* blur = (uint8_t*)c->blur.p + F * g.pyr_frame;
    uint32_t* rowcnt = (uint32_t*)c->rowcnt.p + F * g.cnt_frame;
    uint32_t* rowent = (uint32_t*)c->rowent.p + F * g.ent_frame;
    Elem* work = (Elem*)c->work.p + F * g.ws_frame;
    uint32_t* selpos = (uint32_t*)c->selpos.p + 2 * F * g.ws_frame;
    int* fincnt = (int*)c->fincnt.p + F * g.nlevels;
    int* selcnt = (int*)c->selcnt.p + F * g.nlevels;
    int* status = (int*)c->status.p + F;
    d_kps += F * cap * 7; d_desc += F * cap * 32; d_counts += F;
    const uint32_t* tabs = (const uint32_t*)c->tabs.p;
    const unsigned B = (unsigned)nb;
    cudaStream_t side = c->side[lane_id];
    cudaEvent_t side_fork = c->ev_sfork[lane_id], side_join = c->ev_sjoin[lane_id];

    // ---- kernel choice for this call (orbx_debug_force_kernels: 0 pins the warp kernels, 1 the CTA-cooperative ones)
    // Pyramid / FAST by the size of the launch: the warp-private TMA kernels (one warp walks a whole band / a stack of strips)
    // win once there are enough warps to fill the GPU; below about 26 VGA frames' worth of pixels the CTA-cooperative
    // kernels have the shorter critical path (one 640x480 frame: pyramid + FAST 0.077 ms against 0.115 ms), which is what the
    // sequential VO loop (one frame per call, src/frontend.cpp:98-108) feels.
    const bool cta_family = c->force_kernels >= 0 ? c->force_kernels != 0 : (long)nb * g.w * g.h < 8000000L;
    // Selection by problem size: one WARP per (frame, level) when the candidate lists are short and there are thousands of
    // them (256 VGA frames: 0.116 ms against 0.17 ms), one CTA per (frame, level) when the lists are long -- 512 threads wide
    // there (64 frames of 1920x1080: 0.30 ms against 0.43 ms with 128 threads and 0.65 ms with warps; 3840x2160: 1.21
    // against 1.88 and 2.57 ms).  cta_select = false: the warp trio k_select_fast, k_harris, k_select_harris.
    const bool cta_select = c->force_kernels >= 0 ? c->force_kernels != 0 : (long)g.w * g.h > 600000L;
    // The small upper levels are a chain of short, latency-bound launches (at 640x480 levels 4..7 take as long as levels 1..3
    // for a fifth of the pixels).  They leave the critical path: from level `lt` on, the pyramid chain and the FAST bands of
    // those levels run on a HIGH-PRIORITY side stream (their few CTAs take the next free slots) underneath the FAST launch of the
    // large levels, which is issue-bound and has slots to spare for them only in time, not in space.
    int lt = g.nlevels;                                      // first level of the side chain
    for (int l = g.nlevels - 1; l >= 2 && (long)g.L[l].w * g.L[l].h < SIDE_LEVEL_MAX_PX; --l) lt = l;
    if (cta_family || g.total_bands <= 0 || marks) lt = g.nlevels;   // (stage timers on: one stream, clean per-stage times)
    // Describe groups of 4 slots per warp: four per warp when the batch is large (the warp's set-up is shared, and there are
    // still enough CTAs for several waves), one group per warp (lowest latency) when it is a single frame.
    const long groups = (long)nb * ((std::min(std::max(cap, 1), std::max(c->nfeatures, 1)) + DS_G - 1) / DS_G);
    const int gpw = groups >= 148L * 24 * 8 ? 4 : 1;   // measured at 256 VGA frames: 1 / 2 / 4 / 8 / 16 -> 0.192 / 0.192 / 0.185 / 0.205 / 0.259 ms

    NvtxStages nv;
    nv.next("orbx:gray");
    if (marks) stage_mark(c, 0);
    {
        const int aligned16 = ((reinterpret_cast<uintptr_t>(d_imgs) | step | frame_stride) & 15) == 0;
        const dim3 blk(32, 8);
        const dim3 grd((unsigned)((g.L[0].pitch / 16 + 31) / 32), (unsigned)((g.L[0].h + 7) / 8), B);
        if (channels == 3) k_gray<3><<<grd, blk, 0, st>>>(d_imgs, frame_stride, step, aligned16, g, pyr);
        else               k_gray<1><<<grd, blk, 0, st>>>(d_imgs, frame_stride, step, aligned16, g, pyr);
        ++c->launches;
    }
    if (marks) stage_mark(c, 1);
    auto launch_pyr = [&](int l, cudaStream_t s) {
        if (g.L[l].w <= 0 || g.L[l].h <= 0) return;
        const int nitems = (g.L[l].pitch / 8) * ((g.L[l].h + PYR_RH - 1) / PYR_RH);     // (column octet, row strip) work items
        const dim3 grd((unsigned)((nitems + PYR_NT - 1) / PYR_NT), B);
        if (g.L[l].pt_ok && !cta_family)
            k_pyr_tma<<<dim3((unsigned)((g.L[l].pt_ntask + PT_NWARP - 1) / PT_NWARP), B), PT_NWARP * 32,
                        PT_NWARP * pt_warp_bytes(g.L[l].pt_bw, g.L[l].pt_bh) + 128, s>>>(g, c->pmaps.m[l], l, f0, (uint8_t*)c->pyr.p, tabs, status);
        else if (g.L[l].xspan <= 7) k_pyr_down<false><<<grd, PYR_NT, 0, s>>>(g, l, pyr, tabs);
        else                   k_pyr_down<true><<<grd, PYR_NT, 0, s>>>(g, l, pyr, tabs);
        ++c->launches;
    };
    // The blur (FMA-pipe-bound, needs only the pyramid) follows the small levels on the side stream, i.e. it also runs under the
    // large levels' FAST launch (ALU-pipe-bound): 0.959 -> 0.944 ms per 256 VGA frames.  Capping the occupancy of either kernel
    // so that both are resident in fixed proportions was measured and loses (FAST needs its 7 CTAs per SM).
    bool blur_done = false;
    auto launch_fast = [&](int band_lo, int band_hi, cudaStream_t s) {
        if (band_hi <= band_lo) return;
        if (cta_family) {
            if (band_lo == 0) k_fast_bands<FAST_R, FAST_NT><<<dim3((unsigned)g.total_bands, B), FAST_NT, 0, s>>>(g, pyr, rowcnt, rowent);
        } else
            k_fast_warp<FAST_NWARP><<<dim3((unsigned)((band_hi - band_lo + FAST_NWARP - 1) / FAST_NWARP), B), FAST_NWARP * 32, FAST_NWARP * FW_WARP_BYTES + 128, s>>>(
                g, c->fmaps, f0, band_lo, band_hi, rowcnt, rowent, status);
        ++c->launches;
    };
    nv.next("orbx:pyramid");
    for (int l = 1; l < lt; ++l) launch_pyr(l, st);
    if (marks) stage_mark(c, 2);
    nv.next("orbx:fast_nms (+ small pyramid levels and blur on the side stream)");
    if (lt < g.nlevels) {
        CU(cudaEventRecord(side_fork, st));
        CU(cudaStreamWaitEvent(side, side_fork, 0));
        for (int l = lt; l < g.nlevels; ++l) launch_pyr(l, side);
        launch_fast(g.L[lt].band0, g.total_bands, side);
        if (g.total_blur > 0) {
            k_blur<<<dim3((unsigned)g.total_blur, B), BLUR_NT, 0, side>>>(g, pyr, blur);
            ++c->launches; blur_done = true;
        }
        CU(cudaEventRecord(side_join, side));
        launch_fast(0, g.L[lt].band0, st);
        CU(cudaStreamWaitEvent(st, side_join, 0));
    } else if (g.total_bands > 0) launch_fast(0, g.total_bands, st);
    nv.next("orbx:select_harris");
    if (marks) stage_mark(c, 3);
    if (cta_select) {
        k_select<<<dim3(B, (unsigned)g.nlevels), SEL_NT, 0, st>>>(g, pyr, rowcnt, rowent, work, selpos, fincnt);
        ++c->launches;
    } else {
        // (the warp going straight on to Harris and the second retainBest -- one launch instead of three -- was measured: 0.1435 ms
        //  against 0.1159 ms per 256 VGA frames; the 14 serial Harris evaluations per lane cost the level-0 warps more than the
        //  two launch gaps and the Harris kernel's tail)
        k_select_fast<<<dim3(B, (unsigned)g.nlevels), 32, 0, st>>>(g, rowcnt, rowent, work, selpos, selcnt, fincnt);
        if (g.total_hblk > 0) k_harris<<<dim3((unsigned)g.total_hblk, B), HARRIS_NT, 0, st>>>(g, pyr, work, selcnt);
        k_select_harris<<<dim3(B, (unsigned)g.nlevels), 32, (size_t)g.selh_elems * 12, st>>>(g, work, selpos, selcnt, fincnt, g.selh_elems);
        c->launches += 3;
    }
    nv.next("orbx:blur");
    if (marks) stage_mark(c, 4);
    if (g.total_blur > 0 && !blur_done) {
        k_blur<<<dim3((unsigned)g.total_blur, B), BLUR_NT, 0, st>>>(g, pyr, blur);
        ++c->launches;
    }
    nv.next("orbx:describe");
    if (marks) stage_mark(c, 5);
    const int gcap = (std::max(cap, 1) + DS_G - 1) / DS_G;
    k_describe_tma<<<dim3((unsigned)((gcap + DS_NW * gpw - 1) / (DS_NW * gpw)), B), DS_NW * 32, DS_NW * DS_WARP_BYTES + 128, st>>>(
        g, c->dmaps, f0, work, fincnt, (const float4*)c->pattern.p, d_kps, d_desc, d_counts, cap, gpw, status);
    ++c->launches;
    if (marks) stage_mark(c, 6);
    return ORBX_OK;
}

// The extraction pipeline on device-resident frames; everything asynchronous, ordered on c->stream.  One frame range:
// every kernel fills the GPU on its own (cutting the batch into concurrent frame ranges measured 4 % slower with 3 ranges).
int run_extract(orbx_ctx* c, const uint8_t* d_imgs, int batch, int w, int h, size_t step, size_t frame_stride, int channels,
                float* d_kps, uint8_t* d_desc, int cap, int* d_counts)
{
    int rc = set_geometry(c, w, h);
    if (rc) return rc;
    CU(cudaMemsetAsync(c->status.p, 0, sizeof(int) * (size_t)batch, c->stream));
    if ((rc = run_extract_range(c, c->stream, 0, c->profiling, 0, batch, d_imgs, step, frame_stride, channels, d_kps, d_desc, cap, d_counts)))
        return rc;
    CU(cudaGetLastError());
    c->last_batch = batch;
    if (c->profiling) for (int i = 0; i < 6; ++i) c->stage_valid[i] = true;
    return ORBX_OK;
}

// Host frames [f0, f1) -> the context's staging buffer on stream `st`.  Tightly packed rows go as plain 1-D copies, and
// frames that are also contiguous in host memory (a video buffer, a numpy batch) as ONE copy per range: large linear
// transfers are what PCIe moves fastest.
int upload_frames(orbx_ctx* c, cudaStream_t st, const uint8_t* const* imgs, int f0, int f1, size_t step, size_t row, int h, size_t dstep, size_t fstride)
{
    if (step == row && dstep == row) {
        int i = f0;
        while (i < f1) {
            int j = i + 1;
            while (j < f1 && imgs[j] == imgs[j - 1] + fstride) ++j;
            CU(cudaMemcpyAsync((uint8_t*)c->in.p + fstride * i, imgs[i], fstride * (size_t)(j - i), cudaMemcpyHostToDevice, st));
            i = j;
        }
        return ORBX_OK;
    }
    for (int i = f0; i < f1; ++i)
        CU(cudaMemcpy2DAsync((uint8_t*)c->in.p + fstride * i, dstep, imgs[i], step, row, (size_t)h, cudaMemcpyHostToDevice, st));
    return ORBX_OK;
}

int check_args_extract(orbx_ctx* c, int batch, int w, int h, int channels, int cap)
{
    if (!c) return ORBX_E_ARG;
    if (batch < 0 || batch > c->max_batch) return fail(c, ORBX_E_ARG, "batch outside [0, max_batch]");
    if (w < 0 || h < 0 || w > c->max_w || h > c->max_h) return fail(c, ORBX_E_ARG, "frame larger than the context maximum");
    if (channels != 1 && channels != 3) return fail(c, ORBX_E_UNSUPPORTED, "channels must be 1 (gray) or 3 (BGR)");
    if (cap < 0) return fail(c, ORBX_E_ARG, "negative capacity");
    return ORBX_OK;
}

// A matcher status word was found set (an mbarrier wait timed out on the device): clear all of them, so that the next
// call starts clean without a per-call memset on the matcher's critical path, and report.
int match_timed_out(orbx_ctx* c)
{
    cudaMemset(c->mstatus.p, 0, sizeof(int) * MATCH_WORDS);
    return fail(c, ORBX_E_INTERNAL, "matcher pipeline timed out on an mbarrier (device status set)");
}

// Matcher status words [slot, slot + n) -> h_match(), behind everything queued on the context's stream; then wait for
// that stream and report a timeout if any of the words is set.
int sync_match_words(orbx_ctx* c, int slot, int n)
{
    int* h = c->h_match() + slot;
    if (n > 0) CU(cudaMemcpyAsync(h, (int*)c->mstatus.p + slot, sizeof(int) * n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < n; ++i) if (h[i]) return match_timed_out(c);
    return ORBX_OK;
}

// One matcher job on device-resident operands: nq query rows (shared by every set, or pairwise: set s's own
// min(query_counts[s], nq) rows at query + s * nq * 32, nq being the query stride and the record pitch) against nsets train
// sets of min(train_counts[s], train_stride) rows (null train_counts: all) at train + s * train_stride * 32.
struct MatchJob {
    MatchOp op = MatchOp::Best;
    const uint8_t* query = nullptr;
    int nq = 0;
    const int* query_counts = nullptr;       // pairwise; one CTA per (set, query tile), record slots past a set's count untouched
    const uint8_t* train = nullptr;
    int train_stride = 0;                    // rows per set
    const int* train_counts = nullptr;
    int nsets = 1;
    int4* best = nullptr;                    // [nsets][nq] records; TopK: [nsets][nq][k]; CrossCheck: set s's mutual pairs
                                             // compacted in place to best + s * nq; RadiusEmit: the lists
    int4* second = nullptr;                  // Knn2
    int* xc_count = nullptr;                 // CrossCheck: set s's pair count
    int k = 0;                               // TopK: k >= 2 (the single-CTA kernel of the smallest list bucket that holds k)
    int rad_thr = 0;                         // radius passes: see radius_pass
    long long* rad_offsets = nullptr;
    long long rad_cap = 0;
    // a lane of host_batch: its own stream and status word (concurrent lanes never reset each other's), no train-row split
    // (its key scratch is shared) and no stage marks; otherwise the context's stream and status word 0
    bool lane = false;
    cudaStream_t lane_stream = nullptr;
    int lane_slot = 0;
};
// The job of an operation on nsets train sets of train_stride rows each, train_counts[s] of them present (null: all), and
// one query set of nq rows; the other fields keep their defaults
MatchJob match_job(MatchOp op, const uint8_t* query, int nq, const uint8_t* train, int train_stride, const int* train_counts, int nsets, void* best)
{
    MatchJob job;
    job.op = op;
    job.query = query; job.nq = nq;
    job.train = train; job.train_stride = train_stride; job.train_counts = train_counts; job.nsets = nsets;
    job.best = (int4*)best;
    return job;
}

// The kernel of an operation: CTA pair or not, shared query or pairwise (SETQ), TopK's list bucket (4, 8, 16 or 32 keys).
using MatchKernel = void (*)(MatchArgs);
template <bool SETQ>
MatchKernel match_kernel(MatchOp op, bool pair, int k)
{
    static_assert(ORBX_MAX_KNN <= 32, "the largest list bucket holds 32 keys");
    switch (op) {
    case MatchOp::Best:       return pair ? k_hamming_umma2<MatchOp::Best, SETQ> : k_hamming_umma<MatchOp::Best, SETQ>;
    case MatchOp::Knn2:       return pair ? k_hamming_umma2<MatchOp::Knn2, SETQ> : k_hamming_umma<MatchOp::Knn2, SETQ>;
    case MatchOp::CrossCheck: return pair ? k_hamming_umma2<MatchOp::CrossCheck, SETQ> : k_hamming_umma<MatchOp::CrossCheck, SETQ>;
    case MatchOp::TopK:       return k <= 4 ? k_hamming_umma<MatchOp::TopK, SETQ, 4> : k <= 8 ? k_hamming_umma<MatchOp::TopK, SETQ, 8>
                                   : k <= 16 ? k_hamming_umma<MatchOp::TopK, SETQ, 16> : k_hamming_umma<MatchOp::TopK, SETQ, 32>;
    case MatchOp::RadiusCount: return k_hamming_umma<MatchOp::RadiusCount, SETQ>;
    case MatchOp::RadiusEmit:  return k_hamming_umma<MatchOp::RadiusEmit, SETQ>;
    }
    return nullptr;
}
MatchKernel match_kernel(MatchOp op, bool pair, bool pairwise, int k)
{
    return pairwise ? match_kernel<true>(op, pair, k) : match_kernel<false>(op, pair, k);
}
int match_smem(MatchOp op) { return op == MatchOp::CrossCheck ? MT_SMEM_BYTES_XC : MT_SMEM_BYTES; }

// Every matcher kernel may use its dynamic shared memory (once per context)
bool match_kernels_allow_smem()
{
    constexpr MatchOp ops[] = {MatchOp::Best, MatchOp::Knn2, MatchOp::CrossCheck, MatchOp::TopK, MatchOp::RadiusCount, MatchOp::RadiusEmit};
    for (MatchOp op : ops)
        for (int pairwise = 0; pairwise < 2; ++pairwise)
            for (int pair = 0; pair < 2; ++pair)
                for (int k : {4, 8, 16, 32})
                    if (cudaFuncSetAttribute(match_kernel(op, pair, pairwise, k), cudaFuncAttributeMaxDynamicSharedMemorySize, match_smem(op)) != cudaSuccess)
                        return false;
    return true;
}

// Runs a job, asynchronous on its stream.
int run_match(orbx_ctx* c, const MatchJob& job)
{
    NvtxRange nvr("orbx:match_hamming");
    const int nq = job.nq, nt = job.train_stride, nsets = job.nsets;
    const cudaStream_t st = job.lane ? job.lane_stream : c->stream;
    if (nt >= MT_MAX_TRAIN) return fail(c, ORBX_E_UNSUPPORTED, "train set larger than 2^20 - 1 rows");
    const bool xchk = job.op == MatchOp::CrossCheck;
    if (xchk && nq >= MT_MAX_QUERY_XC) return fail(c, ORBX_E_UNSUPPORTED, "cross-check query set larger than 2^20 - 1 rows");
    const bool knn2 = job.op == MatchOp::Knn2;
    const bool unsplit = !match_op_pairs(job.op);            // top-k and radius: single-CTA kernels, no train-row split
    // CTA-pair kernel (tcgen05 cta_group::2, query tiles in twos) whenever the (query tile, set) pairs alone fill the GPU;
    // small problems keep the single-CTA kernel, whose CTAs are independent units for the train-row split.
    const int tiles_1 = (nq + MT_QROWS - 1) / MT_QROWS, tiles_2 = (tiles_1 + 1) & ~1;
    const bool pair = !unsplit && tiles_1 >= 2 && (long)tiles_2 * nsets >= 148;
    const int tiles_m = pair ? tiles_2 : tiles_1;
    const int ntile_n = (nt + MT_BN - 1) / MT_BN;
    constexpr int kSMs = 148;                                // one CTA per SM (163 KB of shared memory each)
    // Few (query tile, set) pairs: split the train rows across CTAs and merge with atomicMax on the packed key.
    int nsplit = 1;
    if (!knn2 && !unsplit && !job.lane) {
        const long base = (long)tiles_m * nsets;
        if (base < kSMs) nsplit = (int)std::min<long>(ntile_n, std::max<long>(1, (kSMs + base - 1) / base));
    }
    const int tiles_per_split = (ntile_n + nsplit - 1) / nsplit;
    const int rows_per_split = tiles_per_split * MT_BN;
    nsplit = (nt + rows_per_split - 1) / rows_per_split;
    // Many sets: each CTA keeps its expanded query tile and walks sets z, z + zgroups, ... (persistent pipelines).
    // zgroups: waves(z) * sets-per-CTA(z) is the time in units of one (query tile, set) pass; a CTA's setup (TMEM
    // allocation, query expansion, pipeline fill) costs about a third of such a pass for ~1000-row sets, less for longer ones.
    // Pairwise: every set has its own query tile, so every set gets its own CTAs.
    const bool pairwise = job.query_counts != nullptr;
    int zgroups = nsets;
    if (!pairwise) {
        zgroups = 1;
        const long per_z = (long)tiles_m * nsplit;
        const long setup20 = std::max<long>(1, std::min<long>(20, 20L * 4 / std::max(1, tiles_per_split)));   // in 1/20 passes
        long best_cost = -1;
        for (int z = 1; z <= nsets; ++z) {
            const long waves = (per_z * z + kSMs - 1) / kSMs;
            const long cost = waves * (20L * ((nsets + z - 1) / z) + setup20);
            if (best_cost < 0 || cost < best_cost) { best_cost = cost; zgroups = z; }
        }
    }
    // (status words: zero since orbx_create; re-zeroed by match_timed_out() after a failure)
    MatchArgs a = {job.query, nq, job.query_counts, job.train, nt, nt, job.train_counts, nsets, rows_per_split, job.best,
                   job.second, nullptr, nullptr, (int*)c->mstatus.p + (job.lane ? job.lane_slot : 0), job.k, job.rad_thr, job.rad_offsets,
                   job.rad_cap};
    const size_t nout = (size_t)nq * nsets;
    int rc;
    if (!job.lane) stage_mark(c, 7);
    if (nsplit > 1) {
        if ((rc = ensure(c, c->mkeys, nout * sizeof(int)))) return rc;
        a.keys = (int*)c->mkeys.p;
        k_match_keys_init<<<(unsigned)((nout + 255) / 256), 256, 0, st>>>(a.keys, nout);
        ++c->launches;
    }
    if (xchk) {
        const size_t ncol = (size_t)nsets * job.train_stride;
        if ((rc = ensure(c, c->mcolkeys, ncol * sizeof(int)))) return rc;
        a.col_keys = (int*)c->mcolkeys.p;
        k_match_keys_init<<<(unsigned)((ncol + 255) / 256), 256, 0, st>>>(a.col_keys, ncol);
        ++c->launches;
    }
    const dim3 grd((unsigned)tiles_m, (unsigned)nsplit, (unsigned)zgroups);
    const MatchKernel kernel = match_kernel(job.op, pair, pairwise, job.k);
    kernel<<<grd, MT_THREADS, match_smem(job.op), st>>>(a);
    ++c->launches;
    if (nsplit > 1) {
        k_match_finalize<<<(unsigned)((nout + 255) / 256), 256, 0, st>>>(a.keys, nq, job.query_counts, nout, job.best);
        ++c->launches;
    }
    if (xchk) {                                              // reads the finalised row winners
        k_crosscheck_compact<<<(unsigned)nsets, XC_NT, 0, st>>>(job.best, nq, job.query_counts, a.col_keys, job.train_stride, job.best,
                                                               job.xc_count);
        ++c->launches;
    }
    if (!job.lane) { stage_mark(c, 8); if (c->profiling) c->stage_valid[6] = true; }
    CU(cudaGetLastError());
    return ORBX_OK;
}

// One pass of radiusMatch (job.op RadiusCount or RadiusEmit, rad_thr and rad_offsets set), list L = set * nq + query row,
// asynchronous on the context's stream.  The count pass writes every list's length to rad_offsets[1 + L], and the scan turns
// rad_offsets[0 .. nsets * nq] into the 64-bit CSR offsets.  The emit pass (behind it) writes every list that ends at or below
// rad_cap to job.best in ascending trainIdx, and k_radius_order puts each into std::sort's order.
int radius_pass(orbx_ctx* c, const MatchJob& job)
{
    const long long nlists = (long long)job.nsets * job.nq;
    long long* d_offsets = job.rad_offsets;
    int rc;
    if (job.op == MatchOp::RadiusCount) {
        const long long ntiles = (nlists + RS_SCAN_TILE - 1) / RS_SCAN_TILE;
        if ((rc = ensure(c, c->mradsums, sizeof(long long) * (size_t)ntiles))) return rc;
        CU(cudaMemsetAsync(d_offsets, 0, sizeof(long long) * (size_t)(nlists + 1), c->stream));   // (pairwise: rows past a count stay 0)
        if ((rc = run_match(c, job))) return rc;
        long long* sums = (long long*)c->mradsums.p;
        k_radius_tile_sums<<<(unsigned)ntiles, RS_SCAN_NT, 0, c->stream>>>(d_offsets + 1, nlists, sums);
        k_radius_scan_sums<<<1, RS_SCAN_NT, 0, c->stream>>>(sums, ntiles);
        k_radius_scan_tiles<<<(unsigned)ntiles, RS_SCAN_NT, 0, c->stream>>>(d_offsets + 1, nlists, sums);
        c->launches += 3;
    } else {
        if ((rc = run_match(c, job))) return rc;
        k_radius_order<<<(unsigned)((nlists + RS_WARPS - 1) / RS_WARPS), RS_WARPS * 32, 0, c->stream>>>(job.best, d_offsets, nlists, job.nq,
                                                                                                        job.rad_cap);
        ++c->launches;
    }
    CU(cudaGetLastError());
    return ORBX_OK;
}

// The matcher's threshold of the integer radius R = min(256, floor(max_distance)): distance <= R <=> accumulator >= thr
int radius_threshold(float max_distance)
{
    const int r = max_distance >= 256.0f ? 256 : (int)floorf(max_distance);
    return MT_ASCALE * (256 - 2 * r);
}

// cv's CV_Assert(maxDistance > FLT_EPSILON) (false for NaN too)
bool bad_radius(float max_distance) { return !(max_distance > FLT_EPSILON); }

// One matcher request, on host buffers (match_on_host) or device memory (match_on_device).
// in: nq query rows shared by every set, or pairwise (query_counts set) set s's own min(query_counts[s], nq) rows at
//     query + s * nq * 32; against nsets train sets of min(train_counts[s], train_stride) rows (null: all) at
//     train + s * train_stride * 32.
// what: k for TopK; max_distance and cap (the records `best` holds) for radius.  RadiusEmit is radiusMatch: the count
//     pass, then the lists (the emit pass alone once `counted`, the offsets holding the count); RadiusCount the count alone.
// out: best [nsets][nq] records (TopK [nsets][nq][k]; CrossCheck set s's mutual pairs at best + s * nq; radius the lists);
//     second for Knn2 (on the host without it, best receives [nq][2] {best, second}); n_out each set's CrossCheck pair count
//     (on the host: the pairs, radius's records, otherwise nq); offsets radius's nsets * nq + 1 CSR offsets.
struct MatchRequest {
    struct { const uint8_t* query; int nq; const int* query_counts; const uint8_t* train; int train_stride; const int* train_counts; int nsets; } in;
    struct { MatchOp op; int k; float max_distance; long long cap; bool counted; } what;
    struct { orbx_match* best; orbx_match* second; int* n_out; int64_t* offsets; } out;
};

// A request on device memory, asynchronous on the context's stream.  An empty input (no query row, train row or set)
// launches nothing: CrossCheck zeroes every set's pair count and radius every list's offset.
int match_on_device(orbx_ctx* c, const MatchRequest& r)
{
    CU(cudaSetDevice(c->device));
    const MatchOp op = r.what.op;
    const bool radius = op == MatchOp::RadiusCount || op == MatchOp::RadiusEmit;
    if (r.in.nq == 0 || r.in.train_stride == 0 || r.in.nsets == 0) {
        if (op == MatchOp::CrossCheck) CU(cudaMemsetAsync(r.out.n_out, 0, sizeof(int) * (size_t)r.in.nsets, c->stream));
        if (radius) CU(cudaMemsetAsync(r.out.offsets, 0, sizeof(int64_t) * ((size_t)r.in.nsets * r.in.nq + 1), c->stream));
        return ORBX_OK;
    }
    MatchJob job = match_job(op, r.in.query, r.in.nq, r.in.train, r.in.train_stride, r.in.train_counts, r.in.nsets, r.out.best);
    job.query_counts = r.in.query_counts; job.second = (int4*)r.out.second; job.k = r.what.k;
    job.xc_count = op == MatchOp::CrossCheck ? r.out.n_out : nullptr;
    if (!radius) return run_match(c, job);
    job.rad_thr = radius_threshold(r.what.max_distance); job.rad_offsets = (long long*)r.out.offsets; job.rad_cap = r.what.cap;
    if (op == MatchOp::RadiusEmit && !r.what.counted) {      // the count pass first
        job.op = MatchOp::RadiusCount;
        const int rc = radius_pass(c, job);
        if (rc) return rc;
        job.op = MatchOp::RadiusEmit;
    }
    return radius_pass(c, job);
}

// A request on host buffers (not empty), synchronous on the context's stream: the operands go to the context's staging
// buffers, match_on_device runs there (radius: the count pass, the capacity check, then the lists), and the results come
// back.
int match_on_host(orbx_ctx* c, const MatchRequest& r)
{
    CU(cudaSetDevice(c->device));
    const MatchOp op = r.what.op;
    const bool knn2 = op == MatchOp::Knn2, xchk = op == MatchOp::CrossCheck, radius = op == MatchOp::RadiusEmit;
    const int nq = r.in.nq, nsets = r.in.nsets;
    const size_t tbytes = (size_t)nsets * r.in.train_stride * 32, nlists = (size_t)nsets * nq;
    const size_t obytes = nlists * 16 * (size_t)(op == MatchOp::TopK ? r.what.k : 1);
    int rc;
    if ((rc = ensure(c, c->mq, (size_t)nq * 32)) || (rc = ensure(c, c->mt, tbytes)) ||
        (r.in.train_counts && (rc = ensure(c, c->mcounts, sizeof(int) * (size_t)nsets))) ||
        (radius && (rc = ensure(c, c->mradoff, sizeof(long long) * (nlists + 1)))) || (!radius && (rc = ensure(c, c->mbest, obytes))) ||
        (knn2 && (rc = ensure(c, c->msecond, obytes))) || (xchk && (rc = ensure(c, c->mxcount, sizeof(int) * (size_t)nsets))))
        return rc;
    CU(cudaMemcpyAsync(c->mq.p, r.in.query, (size_t)nq * 32, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->mt.p, r.in.train, tbytes, cudaMemcpyHostToDevice, c->stream));
    if (r.in.train_counts)
        CU(cudaMemcpyAsync(c->mcounts.p, r.in.train_counts, sizeof(int) * (size_t)nsets, cudaMemcpyHostToDevice, c->stream));
    MatchRequest d = r;                                      // the same request on the staging buffers
    d.in.query = (const uint8_t*)c->mq.p;
    d.in.train = (const uint8_t*)c->mt.p;
    d.in.train_counts = r.in.train_counts ? (const int*)c->mcounts.p : nullptr;
    d.out = {(orbx_match*)c->mbest.p, knn2 ? (orbx_match*)c->msecond.p : nullptr, xchk ? (int*)c->mxcount.p : nullptr,
             radius ? (int64_t*)c->mradoff.p : nullptr};
    if (radius) {                                            // the lists are made only once they are known to fit
        d.what.op = MatchOp::RadiusCount;
        if ((rc = match_on_device(c, d))) return rc;
        long long total = 0;
        CU(cudaMemcpyAsync(&total, d.out.offsets + nlists, sizeof total, cudaMemcpyDeviceToHost, c->stream));
        if ((rc = sync_match_words(c, 0, 1))) return rc;
        if (total > INT_MAX) return fail(c, ORBX_E_UNSUPPORTED, "more than 2^31 - 1 records");
        *r.out.n_out = (int)total;
        if (total > r.what.cap) return fail(c, ORBX_E_CAPACITY, "output capacity below the number of records");
        if ((rc = ensure(c, c->mbest, 16 * (size_t)total))) return rc;
        d.what = {MatchOp::RadiusEmit, 0, r.what.max_distance, total, true};
        d.out.best = (orbx_match*)c->mbest.p;
    }
    if ((rc = match_on_device(c, d))) return rc;
    int pairs = 0;
    if (xchk) CU(cudaMemcpyAsync(&pairs, d.out.n_out, sizeof(int), cudaMemcpyDeviceToHost, c->stream));   // (one set)
    if (radius) {
        CU(cudaMemcpyAsync(r.out.best, d.out.best, 16 * (size_t)d.what.cap, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(r.out.offsets, d.out.offsets, sizeof(int64_t) * (nlists + 1), cudaMemcpyDeviceToHost, c->stream));
    } else if (knn2 && !r.out.second) {
        CU(cudaMemcpy2DAsync(r.out.best, 32, d.out.best, 16, 16, (size_t)nq, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpy2DAsync(r.out.best + 1, 32, d.out.second, 16, 16, (size_t)nq, cudaMemcpyDeviceToHost, c->stream));
    } else {
        CU(cudaMemcpyAsync(r.out.best, d.out.best, obytes, cudaMemcpyDeviceToHost, c->stream));
        if (r.out.second) CU(cudaMemcpyAsync(r.out.second, d.out.second, obytes, cudaMemcpyDeviceToHost, c->stream));
    }
    if ((rc = sync_match_words(c, 0, 1))) return rc;
    if (r.out.n_out && !radius) *r.out.n_out = xchk ? pairs : nq;
    return ORBX_OK;
}

}  // namespace

// =================================================================================================== C-ABI
extern "C" {

const char* orbx_version(void) { return "orbx 0.1 (sm_100a; tcgen05 int8 matcher)"; }

int orbx_create(orbx_ctx** out, int device, int nfeatures, float scale_factor, int nlevels, int max_w, int max_h, int max_batch)
{
    if (!out) return ORBX_E_ARG;
    *out = nullptr;
    if (nfeatures < 0 || nlevels < 1 || nlevels > ORBX_LEVELS_MAX || !(scale_factor > 1.0f) || max_w < 1 || max_h < 1 ||
        max_w > 65535 || max_h > 65535 || max_batch < 1 || max_batch > 65535)
        return ORBX_E_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return ORBX_E_CUDA;
    std::unique_ptr<orbx_ctx> owner(new (std::nothrow) orbx_ctx());   // a failure below deletes the partly built context
    orbx_ctx* c = owner.get();
    if (!c) return ORBX_E_NOMEM;
    c->device = device; c->nfeatures = nfeatures; c->scale_factor = scale_factor; c->nlevels = nlevels;
    c->max_w = max_w; c->max_h = max_h; c->max_batch = max_batch;
    if (cudaSetDevice(device) != cudaSuccess) return ORBX_E_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return ORBX_E_CUDA;
    if (prop.major != 10) return ORBX_E_CUDA;                // sm_100a only: no other code path exists
    int prio_lo = 0, prio_hi = 0;
    if (cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi) != cudaSuccess) return ORBX_E_CUDA;
    if (cudaStreamCreateWithFlags(&c->stream.h, cudaStreamNonBlocking) != cudaSuccess) return ORBX_E_CUDA;
    for (int k = 0; k < HOST_LANES; ++k)
        if ((k > 0 && cudaStreamCreateWithFlags(&c->lane[k].h, cudaStreamNonBlocking) != cudaSuccess) ||
            cudaStreamCreateWithPriority(&c->side[k].h, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_join[k].h, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_sfork[k].h, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_sjoin[k].h, cudaEventDisableTiming) != cudaSuccess)
            return ORBX_E_CUDA;
    if (cudaEventCreateWithFlags(&c->ev_fork.h, cudaEventDisableTiming) != cudaSuccess) return ORBX_E_CUDA;
    for (auto& a : c->aslot) if (cudaEventCreateWithFlags(&a.done.h, cudaEventDisableTiming) != cudaSuccess) return ORBX_E_CUDA;
    for (Event& e : c->ev) if (cudaEventCreate(&e.h) != cudaSuccess) return ORBX_E_CUDA;
    build_geom(c, max_w, max_h, &c->geom_max, nullptr);
    const Geom& g = c->geom_max;
    const size_t B = (size_t)max_batch;
    if (ensure(c, c->pyr, g.pyr_frame * B + (size_t)(96 + 8) * g.L[0].pitch) ||   // + slack: the blur streams up to ~100 rows past a level's end (masked outputs)
        ensure(c, c->blur, g.pyr_frame * B) || ensure(c, c->rowcnt, g.cnt_frame * 4 * B) || ensure(c, c->rowent, g.ent_frame * 4 * B) ||
        ensure(c, c->work, g.ws_frame * sizeof(Elem) * B) || ensure(c, c->selpos, g.ws_frame * 8 * B) || ensure(c, c->fincnt, sizeof(int) * ORBX_LEVELS_MAX * B) || ensure(c, c->selcnt, sizeof(int) * ORBX_LEVELS_MAX * B) ||
        ensure(c, c->status, sizeof(int) * B) || ensure(c, c->pattern, sizeof(float) * 1024) || ensure(c, c->mstatus, sizeof(int) * MATCH_WORDS) ||
        ensure(c, c->h_small, c->h_small_bytes(), "cudaMallocHost failed"))
        return ORBX_E_NOMEM;
    if (cudaMemset(c->mstatus.p, 0, sizeof(int) * MATCH_WORDS) != cudaSuccess) return ORBX_E_CUDA;
    {
        float pat[1024];                                     // the rBRIEF pattern as float4 (x0, y0, x1, y1) per test,
        for (int t = 0; t < 8; ++t)                          // transposed to [t][lane]: test lane * 8 + t  (k_describe_tma)
            for (int lane = 0; lane < 32; ++lane)
                for (int k = 0; k < 4; ++k) pat[(t * 32 + lane) * 4 + k] = (float)k_pattern_host[(lane * 8 + t) * 4 + k];
        if (cudaMemcpy(c->pattern.p, pat, sizeof pat, cudaMemcpyHostToDevice) != cudaSuccess) return ORBX_E_CUDA;
    }
    if (cudaMemset(c->status.p, 0, sizeof(int) * B) != cudaSuccess) return ORBX_E_CUDA;
    if (!match_kernels_allow_smem() ||
        cudaFuncSetAttribute(k_fast_warp<FAST_NWARP>, cudaFuncAttributeMaxDynamicSharedMemorySize, FAST_NWARP * FW_WARP_BYTES + 128) != cudaSuccess ||
        cudaFuncSetAttribute(k_pyr_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(k_describe_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, DS_NW * DS_WARP_BYTES + 128) != cudaSuccess ||
        cudaFuncSetAttribute(k_select_harris, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 12) != cudaSuccess)
        return ORBX_E_CUDA;
    *out = owner.release();
    return ORBX_OK;
}

void orbx_destroy(orbx_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    c->synchronize_streams();
    delete c;
}

const char* orbx_last_error(const orbx_ctx* c) { return c ? c->err.c_str() : "null context"; }
void* orbx_stream(orbx_ctx* c) { return c ? (void*)c->stream : nullptr; }
uint64_t orbx_launch_count(const orbx_ctx* c) { return c ? c->launches : 0; }

int orbx_synchronize(orbx_ctx* c)
{
    if (!c) return ORBX_E_ARG;
    CU(cudaSetDevice(c->device));
    const int b = c->last_batch;
    if (b > 0) CU(cudaMemcpyAsync(c->h_status(), c->status.p, sizeof(int) * (size_t)b, cudaMemcpyDeviceToHost, c->stream));
    const int rc = sync_match_words(c, 0, MATCH_WORDS);     // the asynchronous matcher entry points defer their status words to this call
    if (rc) return rc;
    for (int i = 0; i < b; ++i)
        if (c->h_status()[i]) return fail(c, ORBX_E_INTERNAL, "device-side status set for a frame");
    return ORBX_OK;
}

int orbx_detect_and_compute_device(orbx_ctx* c, const uint8_t* d_imgs, int batch, int w, int h, size_t step, size_t frame_stride,
                                   int channels, orbx_keypoint* d_kps, uint8_t* d_desc, int cap, int* d_counts)
{
    int rc = check_args_extract(c, batch, w, h, channels, cap);
    if (rc) return rc;
    if (batch == 0) return ORBX_OK;
    if (!d_imgs || !d_kps || !d_desc || !d_counts) return fail(c, ORBX_E_ARG, "null pointer");
    if (w == 0 || h == 0) return fail(c, ORBX_E_ARG, "empty frames are only accepted by the host entry points");
    if (step < (size_t)w * channels) return fail(c, ORBX_E_ARG, "step smaller than a row");
    CU(cudaSetDevice(c->device));
    return run_extract(c, d_imgs, batch, w, h, step, frame_stride, channels, (float*)d_kps, d_desc, cap, d_counts);
}

// ---- host-buffer batches: one core for orbx_detect_and_compute_batch (nmaps = 0) and orbx_extract_match_batch.
// Frame ranges ("lanes") on their own streams: upload -> kernels -> (matches) -> download per lane, so the H2D copy of lane
// k+1 runs under the kernels of lane k and the D2H of lane k under the kernels of lane k+1 (PCIe is the bound here).
// Caller buffers that are NOT page-locked (the reference's cv::Mat frames and std::vector results) go through the context's
// pinned staging, copied by the HostStager threads (orbx_stage.h), so the lanes overlap for them as well.
static bool host_ptr_is_pinned(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

static HostStager* stager_of(orbx_ctx* c)
{
    if (!c->stager) {
        int n = getenv("ORBX_STAGE_THREADS") ? atoi(getenv("ORBX_STAGE_THREADS")) : (int)std::min(8u, std::max(2u, std::thread::hardware_concurrency() / 2));
        c->stager.reset(new HostStager(std::max(0, std::min(n, 32))));
    }
    return c->stager.get();
}

static int host_batch(orbx_ctx* c, const uint8_t* const* imgs, int batch, int w, int h, size_t step, int channels,
                      orbx_keypoint* kps, uint8_t* desc, int cap, int* n_out, const uint8_t* const* queries, const int* nq,
                      int nmaps, orbx_match* const* best)
{
    int rc;
    NvtxRange nvr("orbx:host_batch (stage / upload / extract / match / download)");
    CU(cudaSetDevice(c->device));
    const size_t row = (size_t)w * channels, dstep = round_up(row, 16), fstride = dstep * h;   // 16: k_gray takes 128-bit loads
    const size_t capz = (size_t)std::max(cap, 1);
    size_t qrows = 0, mrows = 0;
    for (int j = 0; j < nmaps; ++j) { qrows += (size_t)nq[j]; mrows += (size_t)nq[j] * batch; }
    if ((rc = ensure(c, c->in, fstride * batch)) || (rc = ensure(c, c->kps, sizeof(orbx_keypoint) * capz * batch)) ||
        (rc = ensure(c, c->desc, (size_t)32 * capz * batch)) || (rc = ensure(c, c->counts, sizeof(int) * (size_t)batch)))
        return rc;
    if (nmaps > 0 && ((rc = ensure(c, c->mq, std::max<size_t>(qrows, 1) * 32)) || (rc = ensure(c, c->mbest, std::max<size_t>(mrows, 1) * 16))))
        return rc;
    for (int i = 0; i < batch; ++i) if (!imgs[i]) return fail(c, ORBX_E_ARG, "null frame pointer");
    if ((rc = set_geometry(c, w, h))) return rc;

    // ---- which caller buffers need staging
    const bool stage_in = !(host_ptr_is_pinned(imgs[0]) && host_ptr_is_pinned(imgs[batch - 1] + (size_t)(h - 1) * step + row - 1));
    bool stage_out = false;
    if (cap > 0) stage_out = !(host_ptr_is_pinned(kps) && host_ptr_is_pinned(desc));
    for (int j = 0; j < nmaps && !stage_out; ++j) if (nq[j] > 0 && !host_ptr_is_pinned(best[j])) stage_out = true;
    const size_t o_kps = 0, o_desc = round_up(sizeof(orbx_keypoint) * capz * batch, 256), o_best = o_desc + round_up((size_t)32 * capz * batch, 256);
    const char* no_pinned = "cudaMallocHost failed for the pinned staging buffer";
    if (stage_in && (rc = ensure(c, c->h_stage_in, fstride * batch, no_pinned))) return rc;
    if (stage_out && (rc = ensure(c, c->h_stage_out, o_best + mrows * 16, no_pinned))) return rc;
    HostStager* hs = (stage_in || stage_out) ? stager_of(c) : nullptr;
    const bool wake_in = fstride * batch >= STAGE_WAKE_BYTES, wake_out = (size_t)60 * capz * batch + mrows * 16 >= STAGE_WAKE_BYTES;
    orbx_keypoint* kps_dl = stage_out ? (orbx_keypoint*)(c->h_stage_out.p + o_kps) : kps;       // where the D2H copies land
    uint8_t* desc_dl = stage_out ? c->h_stage_out.p + o_desc : desc;

    CU(cudaMemsetAsync(c->status.p, 0, sizeof(int) * (size_t)batch, c->stream));
    {
        size_t off = 0;
        for (int j = 0; j < nmaps; ++j) {
            if (nq[j] > 0) CU(cudaMemcpyAsync((uint8_t*)c->mq.p + off * 32, queries[j], (size_t)nq[j] * 32, cudaMemcpyHostToDevice, c->stream));
            off += (size_t)nq[j];
        }
    }
    int* h_counts = c->h_counts();
    int* h_status = c->h_status();
    const int lanes = c->profiling ? 1 : std::max(1, std::min(HOST_LANES, batch / HOST_LANE_MIN_FRAMES));
    // staged inputs: all pieces are queued up front, lane by lane, so the copier threads run ahead of the lane loop
    std::atomic<int> in_done[HOST_LANES], out_done(0);
    int in_target[HOST_LANES] = {}, out_target = 0;
    struct Drain {                                           // no queued piece may outlive the counters above, whichever way this call ends
        HostStager* hs; std::atomic<int>* in; int* in_t; int n; std::atomic<int>* out; int* out_t;
        ~Drain() { if (hs) { for (int k = 0; k < n; ++k) hs->help_until(in[k], in_t[k]); hs->help_until(*out, *out_t); } }
    } drain{hs, in_done, in_target, stage_in ? lanes : 0, &out_done, &out_target};
    if (stage_in)
        for (int k = 0; k < lanes; ++k) {
            int f0, f1;
            host_lane_range(batch, lanes, k, &f0, &f1);
            in_done[k].store(0, std::memory_order_relaxed);
            for (int i = f0; i < f1; ++i) in_target[k] += hs->submit(c->h_stage_in.p + fstride * i, dstep, imgs[i], step, row, (size_t)h, &in_done[k], wake_in, true);
        }
    CU(cudaEventRecord(c->ev_fork, c->stream));
    for (int k = 0; k < lanes; ++k) {
        int f0, f1;
        host_lane_range(batch, lanes, k, &f0, &f1);
        const size_t n = (size_t)(f1 - f0);
        cudaStream_t st = k == 0 ? c->stream : c->lane[k];
        if (k > 0) CU(cudaStreamWaitEvent(st, c->ev_fork, 0));
        if (stage_in) {
            hs->help_until(in_done[k], in_target[k]);        // (the pinned image has the device layout: one copy per lane)
            CU(cudaMemcpyAsync((uint8_t*)c->in.p + fstride * f0, c->h_stage_in.p + fstride * f0, fstride * n, cudaMemcpyHostToDevice, st));
        } else if ((rc = upload_frames(c, st, imgs, f0, f1, step, row, h, dstep, fstride))) return rc;
        if ((rc = run_extract_range(c, st, k, c->profiling, f0, f1 - f0, (const uint8_t*)c->in.p, dstep,
                                    fstride, channels, (float*)c->kps.p, (uint8_t*)c->desc.p, cap, (int*)c->counts.p)))
            return rc;
        CU(cudaMemcpyAsync(h_counts + f0, (int*)c->counts.p + f0, sizeof(int) * n, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(h_status + f0, (int*)c->status.p + f0, sizeof(int) * n, cudaMemcpyDeviceToHost, st));
        if (cap > 0) {
            // outputs are [batch][cap] on both sides: bulk copies per lane (records past n_out[i] are unspecified)
            CU(cudaMemcpyAsync(kps_dl + (size_t)f0 * cap, (orbx_keypoint*)c->kps.p + (size_t)f0 * cap, sizeof(orbx_keypoint) * (size_t)cap * n, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(desc_dl + (size_t)f0 * cap * 32, (uint8_t*)c->desc.p + (size_t)f0 * cap * 32, (size_t)32 * cap * n, cudaMemcpyDeviceToHost, st));
        }
        size_t qoff = 0, moff = 0;
        for (int j = 0; j < nmaps; ++j) {
            if (nq[j] > 0) {
                int4* d_best = (int4*)c->mbest.p + moff + (size_t)f0 * nq[j];
                // train sets = this lane's frames, straight from the extraction outputs ([frame][cap][32] + counts)
                MatchJob job = match_job(MatchOp::Best, (const uint8_t*)c->mq.p + qoff * 32, nq[j], (const uint8_t*)c->desc.p + (size_t)f0 * cap * 32,
                                         cap, (const int*)c->counts.p + f0, (int)n, d_best);
                job.lane = true; job.lane_stream = st; job.lane_slot = k;
                if ((rc = run_match(c, job))) return rc;
                orbx_match* dl = stage_out ? (orbx_match*)(c->h_stage_out.p + o_best) + moff + (size_t)f0 * nq[j] : best[j] + (size_t)f0 * nq[j];
                CU(cudaMemcpyAsync(dl, d_best, (size_t)16 * nq[j] * n, cudaMemcpyDeviceToHost, st));
            }
            qoff += (size_t)nq[j]; moff += (size_t)nq[j] * batch;
        }
        if (k > 0 || stage_out) CU(cudaEventRecord(c->ev_join[k], st));
        if (k > 0) CU(cudaStreamWaitEvent(c->stream, c->ev_join[k], 0));
    }
    CU(cudaGetLastError());
    c->last_batch = batch;
    c->out_cap = cap;
    c->view_desc = (const uint8_t*)c->desc.p; c->view_counts = (const int*)c->counts.p; c->view_frames = batch;
    if (c->profiling) for (int i = 0; i < 6; ++i) c->stage_valid[i] = true;
    if (stage_out) {
        // results leave the pinned staging lane by lane, as soon as a lane's downloads have landed, under the later lanes' work:
        // only the records a frame really has are copied (the caller's records past n_out[i] stay untouched)
        for (int k = 0; k < lanes; ++k) {
            int f0, f1;
            host_lane_range(batch, lanes, k, &f0, &f1);
            CU(cudaEventSynchronize(c->ev_join[k]));
            for (int i = f0; i < f1; ++i) {
                const size_t ni = (size_t)std::max(0, std::min(h_counts[i], cap));
                if (ni > 0) {
                    out_target += hs->submit(kps + (size_t)i * cap, 0, kps_dl + (size_t)i * cap, 0, sizeof(orbx_keypoint) * ni, 1, &out_done, wake_out);
                    out_target += hs->submit(desc + (size_t)i * cap * 32, 0, desc_dl + (size_t)i * cap * 32, 0, 32 * ni, 1, &out_done, wake_out);
                }
            }
            size_t moff = 0;
            for (int j = 0; j < nmaps; ++j) {
                if (nq[j] > 0)
                    out_target += hs->submit(best[j] + (size_t)f0 * nq[j], 0, (orbx_match*)(c->h_stage_out.p + o_best) + moff + (size_t)f0 * nq[j], 0,
                                             (size_t)16 * nq[j] * (size_t)(f1 - f0), 1, &out_done, wake_out);
                moff += (size_t)nq[j] * batch;
            }
        }
        hs->help_until(out_done, out_target);
    }
    if ((rc = sync_match_words(c, 0, nmaps > 0 ? lanes : 0))) return rc;      // lane k's matches report in slot k
    bool over = false;
    for (int i = 0; i < batch; ++i) {
        if (h_status[i]) return fail(c, ORBX_E_INTERNAL, "device-side status set for a frame");
        n_out[i] = h_counts[i];
        if (h_counts[i] > cap) over = true;
    }
    if (over) return fail(c, ORBX_E_CAPACITY, "output capacity too small; n_out holds the needed counts");
    return ORBX_OK;
}

int orbx_detect_and_compute_batch(orbx_ctx* c, const uint8_t* const* imgs, int batch, int w, int h, size_t step, int channels,
                                  orbx_keypoint* kps, uint8_t* desc, int cap, int* n_out)
{
    int rc = check_args_extract(c, batch, w, h, channels, cap);
    if (rc) return rc;
    if (n_out) for (int i = 0; i < batch; ++i) n_out[i] = 0;
    if (batch == 0 || w == 0 || h == 0) return ORBX_OK;     // cv: empty image -> silent return, no keypoints
    if (!imgs || !n_out || (cap > 0 && (!kps || !desc))) return fail(c, ORBX_E_ARG, "null pointer");
    if (step < (size_t)w * channels) return fail(c, ORBX_E_ARG, "step smaller than a row");
    return host_batch(c, imgs, batch, w, h, step, channels, kps, desc, cap, n_out, nullptr, nullptr, 0, nullptr);
}

int orbx_extract_match_batch(orbx_ctx* c, const uint8_t* const* imgs, int batch, int w, int h, size_t step, int channels,
                             orbx_keypoint* kps, uint8_t* desc, int cap, int* n_out, const uint8_t* const* queries, const int* nq,
                             int nmaps, orbx_match* const* best)
{
    int rc = check_args_extract(c, batch, w, h, channels, cap);
    if (rc) return rc;
    if (nmaps < 0 || nmaps > 8) return fail(c, ORBX_E_ARG, "nmaps outside [0, 8]");
    if (n_out) for (int i = 0; i < batch; ++i) n_out[i] = 0;
    if (batch == 0) return ORBX_OK;
    if (!imgs || !n_out || cap <= 0 || !kps || !desc) return fail(c, ORBX_E_ARG, "null pointer / zero capacity");
    if (nmaps > 0 && (!queries || !nq || !best)) return fail(c, ORBX_E_ARG, "null map arguments");
    for (int j = 0; j < nmaps; ++j) if (nq[j] < 0 || (nq[j] > 0 && (!queries[j] || !best[j]))) return fail(c, ORBX_E_ARG, "bad map");
    if (w == 0 || h == 0) {                                  // cv: empty image -> no keypoints; a query against an empty train set -> no matches
        return ORBX_OK;
    }
    if (step < (size_t)w * channels) return fail(c, ORBX_E_ARG, "step smaller than a row");
    if (cap >= MT_MAX_TRAIN) return fail(c, ORBX_E_UNSUPPORTED, "capacity larger than 2^20 - 1 rows");
    return host_batch(c, imgs, batch, w, h, step, channels, kps, desc, cap, n_out, queries, nq, nmaps, best);
}

int orbx_host_register(orbx_ctx* c, void* ptr, size_t bytes)
{
    if (!c) return ORBX_E_ARG;
    if (!ptr || bytes == 0) return fail(c, ORBX_E_ARG, "null pointer / empty range");
    CU(cudaSetDevice(c->device));
    CU(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
    return ORBX_OK;
}

int orbx_host_unregister(orbx_ctx* c, void* ptr)
{
    if (!c) return ORBX_E_ARG;
    if (!ptr) return fail(c, ORBX_E_ARG, "null pointer");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));                    // nothing of this context may still be copying from / into it
    CU(cudaHostUnregister(ptr));
    return ORBX_OK;
}

int orbx_detect_and_compute(orbx_ctx* c, const uint8_t* img, int w, int h, size_t step, int channels, orbx_keypoint* kps,
                            uint8_t* desc, int cap, int* n_out)
{
    if (!c) return ORBX_E_ARG;
    if (!n_out) return fail(c, ORBX_E_ARG, "null n_out");
    *n_out = 0;
    if (w == 0 || h == 0 || !img) { if (!img && w > 0 && h > 0) return fail(c, ORBX_E_ARG, "null image"); return ORBX_OK; }
    const uint8_t* one[1] = {img};
    return orbx_detect_and_compute_batch(c, one, 1, w, h, step, channels, kps, desc, cap, n_out);
}

// Argument checks of the one-set host forms (orbx_match_hamming, _knn2, _knn, _crosscheck, _radius), after their own: the
// row counts and the caller's other invalid arguments (`bad`) -> E_ARG; the caller's unsupported case (`unsupported`: its
// message, or null) -> E_UNSUPPORTED; an empty input (no query or train row) -> *empty, before the pointers -> E_ARG.
static int check_args_one_set(orbx_ctx* c, const void* q, int nq, const void* t, int nt, const void* out, bool bad, const char* unsupported,
                              bool* empty)
{
    if (bad || nq < 0 || nt < 0) return fail(c, ORBX_E_ARG, "bad sizes");
    if (unsupported) return fail(c, ORBX_E_UNSUPPORTED, unsupported);
    if ((*empty = nq == 0 || nt == 0)) return ORBX_OK;       // cv: empty query or train -> no matches, no throw
    if (!q || !t || !out) return fail(c, ORBX_E_ARG, "null pointer");
    return ORBX_OK;
}

int orbx_match_hamming(orbx_ctx* c, const uint8_t* q, int nq, const uint8_t* t, int nt, orbx_match* out, int* n_out)
{
    return orbx_match_hamming_knn(c, q, nq, t, nt, 1, out, n_out);
}
int orbx_match_hamming_knn2(orbx_ctx* c, const uint8_t* q, int nq, const uint8_t* t, int nt, orbx_match* out, int* n_out)
{
    return orbx_match_hamming_knn(c, q, nq, t, nt, 2, out, n_out);
}
int orbx_match_hamming_knn(orbx_ctx* c, const uint8_t* q, int nq, const uint8_t* t, int nt, int k, orbx_match* out, int* n_out)
{
    if (!c) return ORBX_E_ARG;
    if (n_out) *n_out = 0;
    if (k < 1) return fail(c, ORBX_E_ARG, "k < 1");
    if (k > ORBX_MAX_KNN) return fail(c, ORBX_E_UNSUPPORTED, "k larger than ORBX_MAX_KNN");
    bool empty;
    const int rc = check_args_one_set(c, q, nq, t, nt, out, false, nullptr, &empty);
    if (rc || empty) return rc;
    // k records per query row ([nq][k]): k = 1 the plain matcher, k = 2 the knn2 one (interleaved {best, second})
    const MatchOp op = k == 1 ? MatchOp::Best : k == 2 ? MatchOp::Knn2 : MatchOp::TopK;
    return match_on_host(c, {{q, nq, nullptr, t, nt, nullptr, 1}, {op, k}, {out, nullptr, n_out}});
}

int orbx_match_hamming_device(orbx_ctx* c, const uint8_t* d_query, int nq, const uint8_t* d_train, int nt, int nsets,
                              orbx_match* d_best, orbx_match* d_second)
{
    if (!c) return ORBX_E_ARG;
    if (nq < 0 || nt < 0 || nsets < 0 || nsets > 65535) return fail(c, ORBX_E_ARG, "bad sizes");
    if (nq == 0 || nt == 0 || nsets == 0) return ORBX_OK;
    if (!d_query || !d_train || !d_best) return fail(c, ORBX_E_ARG, "null pointer");
    return match_on_device(c, {{d_query, nq, nullptr, d_train, nt, nullptr, nsets}, {d_second ? MatchOp::Knn2 : MatchOp::Best}, {d_best, d_second}});
}

// Argument checks of the shared-query ragged family (_device_ragged, _sets, _device_crosscheck, _device_knn, _device_radius):
// nq query rows against nsets train sets of train_stride_rows rows.  In order: the sizes and the caller's other invalid
// arguments (`bad`) -> E_ARG; the caller's unsupported case (`unsupported`: its message, or null) -> E_UNSUPPORTED; the
// pointers -> E_ARG.  With `empty`, an empty input (no query row, train row or set) is reported there, before the pointers
// are checked; without it the pointers are checked whatever the sizes.
static int check_args_ragged(orbx_ctx* c, const void* query, int nq, const void* train, int train_stride_rows, const int* train_counts,
                             int nsets, const void* out, bool bad, const char* unsupported, bool* empty)
{
    if (bad || nq < 0 || train_stride_rows < 0 || nsets < 0 || nsets > 65535) return fail(c, ORBX_E_ARG, "bad sizes");
    if (unsupported) return fail(c, ORBX_E_UNSUPPORTED, unsupported);
    if (empty && (*empty = nq == 0 || train_stride_rows == 0 || nsets == 0)) return ORBX_OK;
    if (!query || !train || !train_counts || !out) return fail(c, ORBX_E_ARG, "null pointer");
    return ORBX_OK;
}

int orbx_match_hamming_device_ragged(orbx_ctx* c, const uint8_t* d_query, int nq, const uint8_t* d_train, int train_stride_rows,
                                     const int* d_train_counts, int nsets, orbx_match* d_best, orbx_match* d_second)
{
    if (!c) return ORBX_E_ARG;
    bool empty;
    const int rc = check_args_ragged(c, d_query, nq, d_train, train_stride_rows, d_train_counts, nsets, d_best, false, nullptr, &empty);
    if (rc || empty) return rc;
    return match_on_device(c, {{d_query, nq, nullptr, d_train, train_stride_rows, d_train_counts, nsets},
                               {d_second ? MatchOp::Knn2 : MatchOp::Best}, {d_best, d_second}});
}

int orbx_match_hamming_sets(orbx_ctx* c, const uint8_t* query, int nq, const uint8_t* train, int train_stride_rows,
                            const int* train_counts, int nsets, orbx_match* best, orbx_match* second)
{
    if (!c) return ORBX_E_ARG;
    bool empty;
    const int rc = check_args_ragged(c, query, nq, train, train_stride_rows, train_counts, nsets, best, false, nullptr, &empty);
    if (rc || empty) return rc;
    return match_on_host(c, {{query, nq, nullptr, train, train_stride_rows, train_counts, nsets}, {second ? MatchOp::Knn2 : MatchOp::Best},
                             {best, second}});
}

int orbx_match_hamming_crosscheck(orbx_ctx* c, const uint8_t* q, int nq, const uint8_t* t, int nt, orbx_match* out, int* n_out)
{
    if (!c) return ORBX_E_ARG;
    if (!n_out) return fail(c, ORBX_E_ARG, "null n_out");
    *n_out = 0;
    bool empty;                                              // empty query or train -> no pairs (cv2 raises on an empty train)
    const int rc = check_args_one_set(c, q, nq, t, nt, out, false,
                                      nq >= MT_MAX_QUERY_XC ? "cross-check query set larger than 2^20 - 1 rows" : nullptr, &empty);
    if (rc || empty) return rc;
    return match_on_host(c, {{q, nq, nullptr, t, nt, nullptr, 1}, {MatchOp::CrossCheck}, {out, nullptr, n_out}});
}

int orbx_match_hamming_device_crosscheck(orbx_ctx* c, const uint8_t* d_query, int nq, const uint8_t* d_train, int train_stride_rows,
                                         const int* d_train_counts, int nsets, orbx_match* d_out, int* d_n_out)
{
    if (!c) return ORBX_E_ARG;
    bool empty;
    const int rc = check_args_ragged(c, d_query, nq, d_train, train_stride_rows, d_train_counts, nsets, d_out, false,
                                     nq >= MT_MAX_QUERY_XC ? "cross-check query set larger than 2^20 - 1 rows" : nullptr, &empty);
    if (rc || nsets == 0) return rc;
    if (!d_n_out) return fail(c, ORBX_E_ARG, "null pointer");
    return match_on_device(c, {{d_query, nq, nullptr, d_train, train_stride_rows, d_train_counts, nsets}, {MatchOp::CrossCheck},
                               {d_out, nullptr, d_n_out}});
}

int orbx_match_hamming_device_knn(orbx_ctx* c, const uint8_t* d_query, int nq, const uint8_t* d_train, int train_stride_rows,
                                  const int* d_train_counts, int nsets, int k, orbx_match* d_out)
{
    if (!c) return ORBX_E_ARG;
    bool empty;
    const int rc = check_args_ragged(c, d_query, nq, d_train, train_stride_rows, d_train_counts, nsets, d_out, k < 1,
                                     k > ORBX_MAX_KNN ? "k larger than ORBX_MAX_KNN" : nullptr, &empty);
    if (rc || empty) return rc;
    // k = 1: the plain matcher's [nsets][nq] records are the [nsets][nq][1] layout
    return match_on_device(c, {{d_query, nq, nullptr, d_train, train_stride_rows, d_train_counts, nsets}, {k > 1 ? MatchOp::TopK : MatchOp::Best, k},
                               {d_out}});
}

// orbx_match_hamming_device_pairwise[_crosscheck|_knn|_radius]: pair p = query set p against train set p.  Argument checks
// common to all.
static int check_args_pairwise(orbx_ctx* c, const uint8_t* d_query, int query_stride_rows, const int* d_query_counts, const uint8_t* d_train,
                               int train_stride_rows, const int* d_train_counts, int npairs, const void* d_out)
{
    if (query_stride_rows < 0 || train_stride_rows < 0 || npairs < 0 || npairs > 65535) return fail(c, ORBX_E_ARG, "bad sizes");
    if (query_stride_rows >= MT_MAX_TRAIN || train_stride_rows >= MT_MAX_TRAIN)
        return fail(c, ORBX_E_UNSUPPORTED, "pairwise set stride of 2^20 rows or more");
    if (!d_query || !d_query_counts || !d_train || !d_train_counts || !d_out) return fail(c, ORBX_E_ARG, "null pointer");
    return ORBX_OK;
}

int orbx_match_hamming_device_pairwise(orbx_ctx* c, const uint8_t* d_query, int query_stride_rows, const int* d_query_counts,
                                       const uint8_t* d_train, int train_stride_rows, const int* d_train_counts, int npairs,
                                       orbx_match* d_best, orbx_match* d_second)
{
    if (!c) return ORBX_E_ARG;
    int rc = check_args_pairwise(c, d_query, query_stride_rows, d_query_counts, d_train, train_stride_rows, d_train_counts, npairs, d_best);
    if (rc) return rc;
    return match_on_device(c, {{d_query, query_stride_rows, d_query_counts, d_train, train_stride_rows, d_train_counts, npairs},
                               {d_second ? MatchOp::Knn2 : MatchOp::Best}, {d_best, d_second}});
}

int orbx_match_hamming_device_pairwise_crosscheck(orbx_ctx* c, const uint8_t* d_query, int query_stride_rows, const int* d_query_counts,
                                                  const uint8_t* d_train, int train_stride_rows, const int* d_train_counts, int npairs,
                                                  orbx_match* d_out, int* d_n_out)
{
    if (!c) return ORBX_E_ARG;
    int rc = check_args_pairwise(c, d_query, query_stride_rows, d_query_counts, d_train, train_stride_rows, d_train_counts, npairs, d_out);
    if (rc) return rc;
    if (!d_n_out) return fail(c, ORBX_E_ARG, "null pointer");
    return match_on_device(c, {{d_query, query_stride_rows, d_query_counts, d_train, train_stride_rows, d_train_counts, npairs},
                               {MatchOp::CrossCheck}, {d_out, nullptr, d_n_out}});
}

int orbx_match_hamming_device_pairwise_knn(orbx_ctx* c, const uint8_t* d_query, int query_stride_rows, const int* d_query_counts,
                                           const uint8_t* d_train, int train_stride_rows, const int* d_train_counts, int npairs, int k,
                                           orbx_match* d_out)
{
    if (!c) return ORBX_E_ARG;
    if (k < 1) return fail(c, ORBX_E_ARG, "k < 1");
    int rc = check_args_pairwise(c, d_query, query_stride_rows, d_query_counts, d_train, train_stride_rows, d_train_counts, npairs, d_out);
    if (rc) return rc;
    if (k > ORBX_MAX_KNN) return fail(c, ORBX_E_UNSUPPORTED, "k larger than ORBX_MAX_KNN");
    return match_on_device(c, {{d_query, query_stride_rows, d_query_counts, d_train, train_stride_rows, d_train_counts, npairs},
                               {k > 1 ? MatchOp::TopK : MatchOp::Best, k}, {d_out}});
}

int orbx_match_hamming_radius(orbx_ctx* c, const uint8_t* q, int nq, const uint8_t* t, int nt, float max_distance, orbx_match* out, int cap,
                              int64_t* offsets, int* n_out)
{
    if (!c) return ORBX_E_ARG;
    if (!n_out || !offsets) return fail(c, ORBX_E_ARG, "null pointer");
    *n_out = 0;
    bool empty;
    const int rc = check_args_one_set(c, q, nq, t, nt, out, cap < 0 || bad_radius(max_distance),
                                      nt >= MT_MAX_TRAIN ? "train set larger than 2^20 - 1 rows" : nullptr, &empty);
    if (rc) return rc;
    if (empty) {                                             // one empty list per query (cv), or none
        memset(offsets, 0, sizeof(int64_t) * ((size_t)nq + 1));
        return ORBX_OK;
    }
    return match_on_host(c, {{q, nq, nullptr, t, nt, nullptr, 1}, {MatchOp::RadiusEmit, 0, max_distance, cap}, {out, nullptr, n_out, offsets}});
}

int orbx_match_hamming_device_radius(orbx_ctx* c, const uint8_t* d_query, int nq, const uint8_t* d_train, int train_stride_rows,
                                     const int* d_train_counts, int nsets, float max_distance, orbx_match* d_out, int64_t cap, int64_t* d_offsets)
{
    if (!c) return ORBX_E_ARG;
    const int rc = check_args_ragged(c, d_query, nq, d_train, train_stride_rows, d_train_counts, nsets, d_out, cap < 0, nullptr, nullptr);
    if (rc) return rc;
    if (bad_radius(max_distance)) return fail(c, ORBX_E_ARG, "maxDistance must be larger than FLT_EPSILON");
    if (!d_offsets) return fail(c, ORBX_E_ARG, "null pointer");
    if (train_stride_rows >= MT_MAX_TRAIN) return fail(c, ORBX_E_UNSUPPORTED, "train set stride of 2^20 rows or more");
    return match_on_device(c, {{d_query, nq, nullptr, d_train, train_stride_rows, d_train_counts, nsets}, {MatchOp::RadiusEmit, 0, max_distance, cap},
                               {d_out, nullptr, nullptr, d_offsets}});
}

int orbx_match_hamming_device_pairwise_radius(orbx_ctx* c, const uint8_t* d_query, int query_stride_rows, const int* d_query_counts,
                                              const uint8_t* d_train, int train_stride_rows, const int* d_train_counts, int npairs,
                                              float max_distance, orbx_match* d_out, int64_t cap, int64_t* d_offsets)
{
    if (!c) return ORBX_E_ARG;
    if (cap < 0) return fail(c, ORBX_E_ARG, "bad sizes");
    if (bad_radius(max_distance)) return fail(c, ORBX_E_ARG, "maxDistance must be larger than FLT_EPSILON");
    if (!d_offsets) return fail(c, ORBX_E_ARG, "null pointer");
    int rc = check_args_pairwise(c, d_query, query_stride_rows, d_query_counts, d_train, train_stride_rows, d_train_counts, npairs, d_out);
    if (rc) return rc;
    return match_on_device(c, {{d_query, query_stride_rows, d_query_counts, d_train, train_stride_rows, d_train_counts, npairs},
                               {MatchOp::RadiusEmit, 0, max_distance, cap}, {d_out, nullptr, nullptr, d_offsets}});
}

int orbx_filter_matches(orbx_match* m, int n, float ratio)
{
    if (!m || n <= 0) return 0;
    // records with trainIdx < 0 are the "empty train set" placeholders of the batched matchers (distance 0): they are neither
    // matches nor candidates for the minimum -- same rule as the device filter k_filter_matches
    bool any = false;
    float mn = 0.0f;
    for (int i = 0; i < n; ++i) if (m[i].trainIdx >= 0 && (!any || m[i].distance < mn)) { mn = m[i].distance; any = true; }
    if (!any) return 0;
    const float mx = std::max(mn * ratio, 30.0f);
    int k = 0;
    for (int i = 0; i < n; ++i) if (m[i].trainIdx >= 0 && m[i].distance <= mx) m[k++] = m[i];
    return k;
}

int orbx_level_geometry(const orbx_ctx* c, int w, int h, int* ws, int* hs, float* scales, int* quotas)
{
    if (!c || w < 0 || h < 0) return ORBX_E_ARG;
    int a[ORBX_LEVELS_MAX], b[ORBX_LEVELS_MAX], q[ORBX_LEVELS_MAX];
    float s[ORBX_LEVELS_MAX];
    level_sizes(w, h, c->nlevels, c->scale_factor, a, b, s);
    level_quotas(c->nfeatures, c->scale_factor, c->nlevels, q);
    for (int l = 0; l < c->nlevels; ++l) {
        if (ws) ws[l] = a[l];
        if (hs) hs[l] = b[l];
        if (scales) scales[l] = s[l];
        if (quotas) quotas[l] = q[l];
    }
    return ORBX_OK;
}

int orbx_debug_read_level(orbx_ctx* c, int frame, int level, uint8_t* out, size_t out_bytes)
{
    if (!c || !out) return ORBX_E_ARG;
    if (frame < 0 || frame >= c->last_batch || level < 0 || level >= c->geom.nlevels) return fail(c, ORBX_E_ARG, "frame/level out of range");
    const LevelGeom& L = c->geom.L[level];
    if (out_bytes < (size_t)L.w * L.h) return fail(c, ORBX_E_CAPACITY, "buffer too small");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    if (L.w > 0 && L.h > 0)
        CU(cudaMemcpy2D(out, (size_t)L.w, (const uint8_t*)c->pyr.p + (size_t)frame * c->geom.pyr_frame + L.img_off, (size_t)L.pitch,
                        (size_t)L.w, (size_t)L.h, cudaMemcpyDeviceToHost));
    return ORBX_OK;
}

int orbx_debug_read_fast(orbx_ctx* c, int frame, int level, int32_t* x, int32_t* y, int32_t* score, int cap, int* n_out)
{
    if (!c || !n_out) return ORBX_E_ARG;
    *n_out = 0;
    if (frame < 0 || frame >= c->last_batch || level < 0 || level >= c->geom.nlevels) return fail(c, ORBX_E_ARG, "frame/level out of range");
    const Geom& g = c->geom;
    const LevelGeom& L = g.L[level];
    if (L.in_h <= 0) return ORBX_OK;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    std::vector<uint32_t> cnt((size_t)L.in_h), ent((size_t)L.in_h * L.ent_pitch);
    CU(cudaMemcpy(cnt.data(), (const uint32_t*)c->rowcnt.p + (size_t)frame * g.cnt_frame + L.cnt_off, cnt.size() * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(ent.data(), (const uint32_t*)c->rowent.p + (size_t)frame * g.ent_frame + L.ent_off, ent.size() * 4, cudaMemcpyDeviceToHost));
    int n = 0;
    for (int r = 0; r < L.in_h; ++r)
        for (uint32_t i = 0; i < cnt[r]; ++i, ++n)
            if (n < cap) {
                const uint32_t e = ent[(size_t)r * L.ent_pitch + i];
                if (x) x[n] = (int)(e & 0xffffu);
                if (y) y[n] = r + ORBX_EDGE;
                if (score) score[n] = (int)(e >> 16);
            }
    *n_out = n;
    return n > cap ? ORBX_E_CAPACITY : ORBX_OK;
}

int orbx_debug_force_kernels(orbx_ctx* c, int mode)
{
    if (!c || mode < -1 || mode > 1) return ORBX_E_ARG;
    c->force_kernels = mode;
    return ORBX_OK;
}

int orbx_set_profiling(orbx_ctx* c, int enable)
{
    if (!c) return ORBX_E_ARG;
    c->profiling = enable != 0;
    for (int i = 0; i < N_STAGES; ++i) c->stage_valid[i] = false;
    return ORBX_OK;
}

int orbx_debug_stage_times(orbx_ctx* c, const char** names, float* ms, int cap)
{
    if (!c) return ORBX_E_ARG;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    int n = 0;
    for (int i = 0; i < N_STAGES && n < cap; ++i) {
        if (!c->stage_valid[i]) continue;
        float t = 0.f;
        const int e0 = i < 6 ? i : 7;
        if (cudaEventElapsedTime(&t, c->ev[e0], c->ev[e0 + 1]) != cudaSuccess) continue;
        if (names) names[n] = k_stage_names[i];
        if (ms) ms[n] = t;
        ++n;
    }
    return n;
}

}  // extern "C"

// =================================================================================================== map table / tracking
namespace {

// grow a table column, keeping its contents
int grow_keep(orbx_ctx* c, Buf& b, size_t old_bytes, size_t new_bytes)
{
    if (b.bytes >= new_bytes && b.p) return ORBX_OK;
    Buf nb;                                                  // freed here if anything below fails
    const size_t bytes = std::max<size_t>(new_bytes, 256);
    if (cudaMalloc(&nb.p, bytes) != cudaSuccess) return fail(c, ORBX_E_NOMEM, "cudaMalloc failed (map table)");
    nb.bytes = bytes;
    if (cudaMemsetAsync(nb.p, 0, bytes, c->stream) != cudaSuccess) return fail(c, ORBX_E_CUDA, "memset failed");
    if (b.p && old_bytes && cudaMemcpyAsync(nb.p, b.p, old_bytes, cudaMemcpyDeviceToDevice, c->stream) != cudaSuccess)
        return fail(c, ORBX_E_CUDA, "copy failed");
    cudaStreamSynchronize(c->stream);
    b = std::move(nb);
    return ORBX_OK;
}

int map_reserve(orbx_ctx* c, int capacity)
{
    if (capacity <= c->map_capacity) return ORBX_OK;
    int ncap = std::max(capacity, std::max(1024, c->map_capacity * 2));
    const size_t o = (size_t)c->map_capacity, n = (size_t)ncap;
    int rc;
    if ((rc = grow_keep(c, c->t_desc, o * 32, n * 32)) || (rc = grow_keep(c, c->t_pos, o * 24, n * 24)) || (rc = grow_keep(c, c->t_nrm, o * 24, n * 24)) ||
        (rc = grow_keep(c, c->t_outl, o, n)))
        return rc;
    c->map_capacity = ncap;
    return ORBX_OK;
}

// ids -> slots (allocating new slots when `create`); the slot list is left in c->t_slots on the device
int map_slots(orbx_ctx* c, const int64_t* ids, int n, bool create, std::vector<int>* slots)
{
    slots->resize((size_t)n);
    if (create) {
        int fresh = 0;
        for (int i = 0; i < n; ++i) if (!c->map_slot.count((long long)ids[i])) ++fresh;     // duplicates inside one call over-count: harmless
        const int need = c->map_next - (int)c->map_free.size() + fresh;
        int rc = map_reserve(c, std::max(need, c->map_next));
        if (rc) return rc;
    }
    for (int i = 0; i < n; ++i) {
        auto it = c->map_slot.find((long long)ids[i]);
        if (it != c->map_slot.end()) { (*slots)[i] = it->second; continue; }
        if (!create) return fail(c, ORBX_E_ARG, "unknown map-point id");
        int s;
        if (!c->map_free.empty()) { s = c->map_free.back(); c->map_free.pop_back(); }
        else {
            s = c->map_next++;
            if (s >= c->map_capacity) { int rc = map_reserve(c, s + 1); if (rc) return rc; }
        }
        c->map_slot.emplace((long long)ids[i], s);
        (*slots)[i] = s;
    }
    int rc = ensure(c, c->t_slots, sizeof(int) * (size_t)std::max(n, 1));
    if (rc) return rc;
    CU(cudaMemcpyAsync(c->t_slots.p, slots->data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    return ORBX_OK;
}

}  // namespace

extern "C" {

int orbx_map_reserve(orbx_ctx* c, int capacity)
{
    if (!c || capacity < 0) return ORBX_E_ARG;
    CU(cudaSetDevice(c->device));
    return map_reserve(c, capacity);
}

int orbx_map_size(const orbx_ctx* c) { return c ? (int)c->map_slot.size() : 0; }

int orbx_map_clear(orbx_ctx* c)
{
    if (!c) return ORBX_E_ARG;
    c->map_slot.clear(); c->map_free.clear(); c->map_next = 0;
    return ORBX_OK;
}

int orbx_map_upsert(orbx_ctx* c, const int64_t* ids, int n, const uint8_t* desc, const double* pos, const double* norm, const uint8_t* outlier)
{
    if (!c || n < 0) return ORBX_E_ARG;
    if (n == 0) return ORBX_OK;
    if (!ids) return fail(c, ORBX_E_ARG, "null ids");
    CU(cudaSetDevice(c->device));
    std::vector<int> slots;
    std::vector<char> is_new((size_t)n);
    for (int i = 0; i < n; ++i) is_new[i] = !c->map_slot.count((long long)ids[i]);
    int rc = map_slots(c, ids, n, true, &slots);
    if (rc) return rc;
    // staging: [desc n*32][pos n*24][norm n*24][outlier n]; a column the caller leaves NULL keeps its value for existing
    // points and starts as zero for new ones (outlier_ = false, norm_ = 0: src/mappoint.cpp:35)
    const size_t N = (size_t)n, o_pos = N * 32, o_nrm = o_pos + N * 24, o_out = o_nrm + N * 24, total = o_out + N;
    if ((rc = ensure(c, c->t_in, total))) return rc;
    uint8_t* st = (uint8_t*)c->t_in.p;
    if (desc) CU(cudaMemcpyAsync(st, desc, N * 32, cudaMemcpyHostToDevice, c->stream));
    if (pos) CU(cudaMemcpyAsync(st + o_pos, pos, N * 24, cudaMemcpyHostToDevice, c->stream));
    if (norm) CU(cudaMemcpyAsync(st + o_nrm, norm, N * 24, cudaMemcpyHostToDevice, c->stream));
    if (outlier) CU(cudaMemcpyAsync(st + o_out, outlier, N, cudaMemcpyHostToDevice, c->stream));
    if (!desc || !pos || !norm || !outlier) {
        // zero the columns of NEW points that were not supplied: one scatter of zeros for those slots
        std::vector<int> ns;
        for (int i = 0; i < n; ++i) if (is_new[i]) ns.push_back(slots[i]);
        if (!ns.empty()) {
            const size_t Z = ns.size();
            const size_t zoff = round_up(Z * 4, 16);        // the zero block is read as uint4 / double: keep it 16-byte aligned
            if ((rc = ensure(c, c->t_aux, zoff + Z * 32))) return rc;
            CU(cudaMemcpyAsync(c->t_aux.p, ns.data(), Z * 4, cudaMemcpyHostToDevice, c->stream));
            uint8_t* z = (uint8_t*)c->t_aux.p + zoff;
            CU(cudaMemsetAsync(z, 0, Z * 32, c->stream));
            k_map_scatter<<<(unsigned)((Z + 255) / 256), 256, 0, c->stream>>>((const int*)c->t_aux.p, (int)Z, desc ? nullptr : z, pos ? nullptr : (const double*)z,
                                                                              norm ? nullptr : (const double*)z, outlier ? nullptr : z, (uint8_t*)c->t_desc.p,
                                                                              (double*)c->t_pos.p, (double*)c->t_nrm.p, (uint8_t*)c->t_outl.p);
            ++c->launches;
            CU(cudaStreamSynchronize(c->stream));            // `ns` is a local
        }
    }
    k_map_scatter<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>((const int*)c->t_slots.p, n, desc ? st : nullptr, pos ? (const double*)(st + o_pos) : nullptr,
                                                                      norm ? (const double*)(st + o_nrm) : nullptr, outlier ? st + o_out : nullptr,
                                                                      (uint8_t*)c->t_desc.p, (double*)c->t_pos.p, (double*)c->t_nrm.p, (uint8_t*)c->t_outl.p);
    ++c->launches;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));                    // host sources are borrowed only for the duration of the call
    return ORBX_OK;
}

int orbx_map_upsert_from_frame(orbx_ctx* c, const int64_t* ids, int n, int frame, const int32_t* kp_index, const double* pos, const double* norm)
{
    if (!c || n < 0) return ORBX_E_ARG;
    if (n == 0) return ORBX_OK;
    if (!ids || !kp_index) return fail(c, ORBX_E_ARG, "null pointer");
    if (!c->view_desc || c->out_cap <= 0 || frame < 0 || frame >= c->view_frames) return fail(c, ORBX_E_ARG, "no host-API extraction holds that frame");
    for (int i = 0; i < n; ++i) if (kp_index[i] < 0 || kp_index[i] >= c->out_cap) return fail(c, ORBX_E_ARG, "keypoint index out of range");
    int rc = orbx_map_upsert(c, ids, n, nullptr, pos, norm, nullptr);
    if (rc) return rc;
    std::vector<int> slots;
    if ((rc = map_slots(c, ids, n, false, &slots))) return rc;
    if ((rc = ensure(c, c->t_aux, sizeof(int) * (size_t)n))) return rc;
    CU(cudaMemcpyAsync(c->t_aux.p, kp_index, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    k_map_scatter_desc<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>((const int*)c->t_slots.p, (const int*)c->t_aux.p, n,
                                                                           c->view_desc + (size_t)frame * c->out_cap * 32, (uint8_t*)c->t_desc.p);
    ++c->launches;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    return ORBX_OK;
}

int orbx_map_erase(orbx_ctx* c, const int64_t* ids, int n)
{
    if (!c || n < 0 || (n > 0 && !ids)) return ORBX_E_ARG;
    for (int i = 0; i < n; ++i) {
        auto it = c->map_slot.find((long long)ids[i]);
        if (it == c->map_slot.end()) continue;
        c->map_free.push_back(it->second);
        c->map_slot.erase(it);
    }
    return ORBX_OK;
}

int orbx_track_match(orbx_ctx* c, const int64_t* ids, int m, const double* pose_Tcw, const double* cam, int cols, int rows,
                     const uint8_t* train, int nt_or_frame, float match_ratio, int32_t* cand, int* n_cand, orbx_match* matches, int* n_matches,
                     float* min_dis, float* max_dis)
{
    if (!c) return ORBX_E_ARG;
    if (n_cand) *n_cand = 0;
    if (n_matches) *n_matches = 0;
    if (m < 0 || !pose_Tcw || !cam || !n_cand || !n_matches) return fail(c, ORBX_E_ARG, "bad arguments");
    if (m == 0) return ORBX_OK;
    if (!ids || !cand || !matches) return fail(c, ORBX_E_ARG, "null pointer");
    CU(cudaSetDevice(c->device));
    // train set: host rows, or frame `nt_or_frame` of the last host-API extraction (still on the device)
    const uint8_t* d_train = nullptr;
    const int* d_tcount = nullptr;
    int nt = 0;
    int rc;
    if (train) {
        nt = nt_or_frame;
        if (nt < 0) return fail(c, ORBX_E_ARG, "negative train count");
        if (nt > 0) {
            if ((rc = ensure(c, c->mt, (size_t)nt * 32))) return rc;
            CU(cudaMemcpyAsync(c->mt.p, train, (size_t)nt * 32, cudaMemcpyHostToDevice, c->stream));
            d_train = (const uint8_t*)c->mt.p;
        }
    } else {
        const int f = nt_or_frame;
        if (!c->view_desc || c->out_cap <= 0 || f < 0 || f >= c->view_frames) return fail(c, ORBX_E_ARG, "no host-API extraction holds that frame");
        d_train = c->view_desc + (size_t)f * c->out_cap * 32;
        d_tcount = c->view_counts + f;
        nt = c->out_cap;
    }
    std::vector<int> slots;
    if ((rc = map_slots(c, ids, m, false, &slots))) return rc;
    if ((rc = ensure(c, c->t_cand, sizeof(int) * (size_t)m)) || (rc = ensure(c, c->t_ncand, 16)) || (rc = ensure(c, c->t_q, (size_t)m * 32)) ||
        (rc = ensure(c, c->t_best, (size_t)m * 16)) || (rc = ensure(c, c->t_filtered, (size_t)m * 16)) || (rc = ensure(c, c->t_minmax, 16)))
        return rc;
    Pose T; Cam K;
    for (int i = 0; i < 12; ++i) T.m[i] = pose_Tcw[i];
    K.fx = cam[0]; K.fy = cam[1]; K.cx = cam[2]; K.cy = cam[3];
    k_visibility<<<1, VIS_NT, 0, c->stream>>>((const int*)c->t_slots.p, m, T, K, cols, rows, (const double*)c->t_pos.p, (const double*)c->t_nrm.p,
                                              (const uint8_t*)c->t_outl.p, (int*)c->t_cand.p, (int*)c->t_ncand.p);
    ++c->launches;
    int* h = c->h_counts();
    CU(cudaMemcpyAsync(h, c->t_ncand.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));                    // the candidate count sizes the matcher's grid
    const int nc = h[0];
    *n_cand = nc;
    if (nc > 0) CU(cudaMemcpyAsync(cand, c->t_cand.p, sizeof(int) * (size_t)nc, cudaMemcpyDeviceToHost, c->stream));
    if (nc == 0 || nt == 0) { CU(cudaStreamSynchronize(c->stream)); return ORBX_OK; }   // cv: empty query or train -> no matches
    k_gather_desc<<<(unsigned)((nc + 255) / 256), 256, 0, c->stream>>>((const int*)c->t_slots.p, (const int*)c->t_cand.p, nc, (const uint8_t*)c->t_desc.p,
                                                                       (uint8_t*)c->t_q.p);
    ++c->launches;
    const MatchJob job = match_job(MatchOp::Best, (const uint8_t*)c->t_q.p, nc, d_train, nt, d_tcount, 1, c->t_best.p);
    if ((rc = run_match(c, job))) return rc;
    k_filter_matches<<<1, VIS_NT, 0, c->stream>>>((const int4*)c->t_best.p, nc, match_ratio, (int4*)c->t_filtered.p, (int*)c->t_ncand.p + 1,
                                                  (float*)c->t_minmax.p);
    ++c->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h, (int*)c->t_ncand.p + 1, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(h + 1, c->t_minmax.p, 2 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if ((rc = sync_match_words(c, 0, 1))) return rc;
    const int nm = h[0];
    if (nm > 0) CU(cudaMemcpy(matches, c->t_filtered.p, (size_t)nm * 16, cudaMemcpyDeviceToHost));
    *n_matches = nm;
    if (min_dis) memcpy(min_dis, h + 1, sizeof(float));
    if (max_dis) memcpy(max_dis, h + 2, sizeof(float));
    return ORBX_OK;
}

int orbx_backproject(orbx_ctx* c, const orbx_keypoint* kps, int n, const uint16_t* depth, int w, int h, size_t step_bytes, float depth_scale,
                     const double* cam, const double* pose_Tcw, double* pos_w, uint8_t* valid)
{
    if (!c || n < 0) return ORBX_E_ARG;
    if (n == 0) return ORBX_OK;
    if (!kps || !depth || !cam || !pose_Tcw || !pos_w || !valid || w <= 0 || h <= 0 || step_bytes < (size_t)w * 2 || (step_bytes & 1))
        return fail(c, ORBX_E_ARG, "bad arguments");
    CU(cudaSetDevice(c->device));
    const size_t N = (size_t)n, dbytes = step_bytes * (size_t)h;
    const size_t o_depth = round_up(N * 28, 256), o_pos = round_up(o_depth + dbytes, 256), o_valid = o_pos + N * 24, total = o_valid + N;
    int rc = ensure(c, c->t_in, total);
    if (rc) return rc;
    uint8_t* st = (uint8_t*)c->t_in.p;
    CU(cudaMemcpyAsync(st, kps, N * 28, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(st + o_depth, depth, dbytes, cudaMemcpyHostToDevice, c->stream));
    Pose T; Cam K;
    for (int i = 0; i < 12; ++i) T.m[i] = pose_Tcw[i];
    K.fx = cam[0]; K.fy = cam[1]; K.cx = cam[2]; K.cy = cam[3];
    k_backproject<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>((const float*)st, n, (const uint16_t*)(st + o_depth), w, h, step_bytes / 2,
                                                                      (double)depth_scale, K, T, (double*)(st + o_pos), st + o_valid);
    ++c->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(pos_w, st + o_pos, N * 24, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(valid, st + o_valid, N, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return ORBX_OK;
}

}  // extern "C"

// =================================================================================================== async single-frame pipeline
extern "C" {

int orbx_submit_frame(orbx_ctx* c, const uint8_t* img, int w, int h, size_t step, int channels)
{
    if (!c) return ORBX_E_ARG;
    if (!img || w <= 0 || h <= 0) return fail(c, ORBX_E_ARG, "empty or null image (use the synchronous call for empty frames)");
    int rc = check_args_extract(c, 1, w, h, channels, 0);
    if (rc) return rc;
    if (step < (size_t)w * channels) return fail(c, ORBX_E_ARG, "step smaller than a row");
    if (c->a_inflight >= 2) return fail(c, ORBX_E_BUSY, "two frames already in flight: collect one first");
    CU(cudaSetDevice(c->device));
    orbx_ctx::AsyncSlot& a = c->aslot[(c->a_head + c->a_inflight) & 1];
    const int cap = std::max(2 * c->nfeatures, 64);
    const size_t row = (size_t)w * channels, dstep = round_up(row, 16), fstride = dstep * h;
    if ((rc = ensure(c, a.h_in, fstride, "pinned allocation failed")) || (rc = ensure(c, a.h_out, 32 + (size_t)cap * 60, "pinned allocation failed")) ||
        (rc = ensure(c, c->in, fstride)) || (rc = ensure(c, a.d_kps, sizeof(orbx_keypoint) * (size_t)cap)) || (rc = ensure(c, a.d_desc, (size_t)32 * cap)) ||
        (rc = ensure(c, a.d_counts, 32)))
        return rc;
    a.cap = cap;
    if (c->view_desc == (const uint8_t*)a.d_desc.p) {         // the last collected frame lives in this slot: its descriptors are about to be
        c->view_desc = nullptr; c->view_counts = nullptr; c->view_frames = 0;   // overwritten, so "frame 0 of the last extraction" no longer exists
    }
    if ((rc = set_geometry(c, w, h))) return rc;
    for (int y = 0; y < h; ++y) memcpy(a.h_in.p + (size_t)y * dstep, img + (size_t)y * step, row);     // the caller's buffer is free on return
    // everything below is stream-ordered behind the previous frame: the shared per-frame workspace is reused safely
    CU(cudaMemcpyAsync(c->in.p, a.h_in.p, fstride, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemsetAsync(c->status.p, 0, sizeof(int), c->stream));
    if ((rc = run_extract_range(c, c->stream, 0, false, 0, 1, (const uint8_t*)c->in.p, dstep, fstride, channels, (float*)a.d_kps.p,
                                (uint8_t*)a.d_desc.p, cap, (int*)a.d_counts.p)))
        return rc;
    CU(cudaMemcpyAsync(a.h_out.p, a.d_counts.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(a.h_out.p + 16, c->status.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(a.h_out.p + 32, a.d_kps.p, sizeof(orbx_keypoint) * (size_t)cap, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(a.h_out.p + 32 + (size_t)cap * 28, a.d_desc.p, (size_t)32 * cap, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaEventRecord(a.done, c->stream));
    CU(cudaGetLastError());
    a.busy = true;
    ++c->a_inflight;
    return ORBX_OK;
}

int orbx_collect_frame(orbx_ctx* c, orbx_keypoint* kps, uint8_t* desc, int cap, int* n_out)
{
    if (!c || !n_out) return ORBX_E_ARG;
    *n_out = 0;
    if (c->a_inflight <= 0) return fail(c, ORBX_E_ARG, "no frame in flight");
    if (cap < 0 || (cap > 0 && (!kps || !desc))) return fail(c, ORBX_E_ARG, "null output");
    CU(cudaSetDevice(c->device));
    orbx_ctx::AsyncSlot& a = c->aslot[c->a_head];
    CU(cudaEventSynchronize(a.done));
    int n, status;
    memcpy(&n, a.h_out.p, sizeof n);
    memcpy(&status, a.h_out.p + 16, sizeof status);
    *n_out = n;
    if (n > a.cap) {                                          // more ties than the internal capacity: redo synchronously is the caller's fallback
        a.busy = false; c->a_head ^= 1; --c->a_inflight;
        return fail(c, ORBX_E_CAPACITY, "internal capacity exceeded; use orbx_detect_and_compute for this frame");
    }
    if (status) {                                             // device-side flag (selection fallback bound / TMA timeout): never hand out a possibly wrong frame
        a.busy = false; c->a_head ^= 1; --c->a_inflight;
        *n_out = 0;
        return fail(c, ORBX_E_INTERNAL, "device-side status set for the collected frame");
    }
    if (n > cap) return fail(c, ORBX_E_CAPACITY, "output capacity too small; n_out holds the needed count (frame still in flight)");
    memcpy(kps, a.h_out.p + 32, sizeof(orbx_keypoint) * (size_t)n);
    memcpy(desc, a.h_out.p + 32 + (size_t)a.cap * 28, (size_t)32 * n);
    // the collected frame becomes "frame 0 of the last extraction" for orbx_track_match / orbx_map_upsert_from_frame
    c->view_desc = (const uint8_t*)a.d_desc.p; c->view_counts = (const int*)a.d_counts.p; c->view_frames = 1; c->out_cap = a.cap;
    a.busy = false;
    c->a_head ^= 1;
    --c->a_inflight;
    return ORBX_OK;
}

}  // extern "C"
