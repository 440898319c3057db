// spgroup.cu -- C ABI (include/spgroup.h) over the sm_100a grouping kernels.
//
// Host-side runtime of the path: handle/workspace management, launch configuration, the chunked
// host-buffer pipeline (H2D copy of chunk c+1 overlapped with the kernels of chunk c on two streams) and
// the state transfer used by the stage-wise drop-in functions.  No torch, no CPU implementation: if the
// device or a launch fails the call fails.
#include "../../include/spgroup.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "assemble.cuh"
#include "common.cuh"
#include "limb_match.cuh"
#include "limb_score.cuh"
#include "limb_score_persist.cuh"
#include "match_assemble.cuh"
#include "nms_peaks.cuh"
#include "nms_peaks_persist.cuh"
#include "nms_peaks_banded.cuh"
#include "postnet.cuh"
#include "postnet_rot.cuh"
#include "prenet.cuh"

using namespace spg;

static_assert(sizeof(spg_params) == sizeof(spg::Params), "spg_params layout");

static thread_local std::string g_create_error;

struct spg_handle {
    spg_config cfg{};
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    Workspace ws{};
    std::vector<void *> allocs;
    // staging for spg_group_host
    void *in_heat = nullptr, *in_paf = nullptr;
    size_t in_heat_bytes = 0, in_paf_bytes = 0;
    unsigned int *done_counter = nullptr;          // "last CTA done" counter of the in-kernel wire signal
    unsigned long long *armed_flag = nullptr;      // spg_arm_wire_signal: consumed by the next assemble launch
    unsigned long long armed_value = 0;
    double *heat_acc = nullptr;  // postnet: float64 accumulator of the keypoint maps over the scale loop
    size_t heat_acc_elems = 0;
    unsigned char *pre_img = nullptr;  // prenet: imageToTest_padded of the current scale, uint8 [Hp][Wp][3]
    size_t pre_img_bytes = 0;
    cudaStream_t streams[2] = {nullptr, nullptr};
    int64_t launches = 0;
    const char *stage_kernel[5] = {"", "", "", "", ""};  // nms_peaks, limb_score, limb_match, assemble, post-network
    // tuning / A-B switches, read from the environment ONCE in spg_create (never per launch); none changes a result
    int persist = 1;      // persistent warp-specialised nms_peaks / limb_score when they apply (SPG_PERSIST=0 turns them off)
    int screen = 1;       // limb_score phase A on (SPG_NO_SCREEN=1 turns it off: every pair is evaluated exactly)
    int exact_warps = 12; // scorer warps of the persistent limb_score (SPG_EXACT_WARPS)
    int post_generic_ident = 0;  // SPG_POST_IDENT=0: single-scale identity configurations take postnet_kernel<true,true,*> (A/B timing)
    int ma_warps = kMAMatchWarps;  // matcher warps of the fused kernel (SPG_MA_WARPS, tuning)
    int fuse_ma = 1;      // whole-path calls run the fused match+assemble kernel (SPG_FUSE_MA=0: the two kernels back to back)
    int cand_dtype = SPG_F32;  // dtype of the planes the current candidates were scored on
    int stage = 0;  // 0 none, 1 peaks, 2 candidates, 3 connections, 4 people
    std::string err;
};

namespace {

int fail(spg_handle *h, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define SPG_CUDA(h, call)                                                                              \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail((h), SPG_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

template <typename T>
int dalloc(spg_handle *h, T **p, size_t count) {
    void *q = nullptr;
    SPG_CUDA(h, cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T)));
    h->allocs.push_back(q);
    *p = static_cast<T *>(q);
    return SPG_OK;
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int cur = -1;
        cudaGetDevice(&cur);
        if (prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};

int check_dims(spg_handle *h, int n, int H, int W) {
    if (n < 0 || n > h->cfg.max_batch) return fail(h, SPG_E_INVALID, "n_images %d outside [0, max_batch=%d]", n, h->cfg.max_batch);
    if (H < 2 || W < 2 || H > h->cfg.max_h || W > h->cfg.max_w || H > 32767 || W > 32767)
        return fail(h, SPG_E_INVALID, "map %dx%d outside [2, %dx%d]", H, W, h->cfg.max_h, h->cfg.max_w);
    return SPG_OK;
}

int check_params(spg_handle *h, const spg_params *p) {
    if (!p) return fail(h, SPG_E_INVALID, "params is NULL");
    if (p->offset_radius < 0 || p->offset_radius > kMaxRefineRadius)
        return fail(h, SPG_E_INVALID, "offset_radius %d outside [0, %d]", p->offset_radius, kMaxRefineRadius);
    if (p->mid_num < 1) return fail(h, SPG_E_INVALID, "mid_num must be >= 1");
    return SPG_OK;
}

// ---- stage launchers on absolute image range [base, base+n) with chunk-local input pointers ----
int launch_nms(spg_handle *h, const float *heat, int64_t img_stride, int64_t chan_stride, int base, int n, int H, int W,
               const spg_params *p, cudaStream_t st) {
    if (n == 0) return SPG_OK;
    NmsArgs a{};
    a.heat = heat;
    a.img_stride = img_stride;
    a.chan_stride = chan_stride;
    a.H = H;
    a.W = W;
    // bands of ~16 KB through a ring of 3 buffers: two bands in flight per CTA while one is scanned, 4 CTAs per SM
    // (measured on B200 at 256 x 18 planes of 128x128: 94 us; whole-plane-resident and 512-thread variants: 97-108 us)
    a.band_rows = std::max(4, std::min(H, 4096 / W));
    a.radius = p->offset_radius;
    a.use_bulk = (W % 4 == 0) && (img_stride % 4 == 0) && (chan_stride % 4 == 0) && ((reinterpret_cast<uintptr_t>(heat) & 15) == 0);
    a.image_base = base;
    a.thr = (float)p->thre1;
    a.ws = h->ws;
    if (h->persist && a.use_bulk && nms_persist_smem_bytes(H, W, h->ws.capP) <= h->smem_optin && (size_t)H * W / 4 < 65536 &&
        (size_t)H * W * sizeof(float) < (1u << 20) &&
        ((size_t)H * W / 4 + kNmsPScanners - 1) / kNmsPScanners <= (size_t)32 * kNmsPMaxIter) {
        // one resident CTA per SM: loader, 28 scanners, 3 finishers over a ring of 3 plane slots
        const size_t psm = nms_persist_smem_bytes(H, W, h->ws.capP);
        const int items = n * h->ws.K;
        SPG_CUDA(h, cudaFuncSetAttribute(nms_peaks_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psm));
        nms_peaks_persist_kernel<<<std::min(items, h->sm_count), kNmsPThreads, psm, st>>>(a, items);
        h->stage_kernel[0] = "nms_peaks_persist_kernel";
        h->launches++;
        SPG_CUDA(h, cudaGetLastError());
        return SPG_OK;
    }
    const NmsBanding bg = (h->persist && a.use_bulk) ? nms_banding(H, W, h->ws.capP, h->smem_optin - 1024) : NmsBanding{};
    if (bg.slots >= kNmsBTeams) {
        // planes that do not fit three times: the same roles over a ring of ~17 KB band slots, four scanner teams
        const int items = n * h->ws.K;
        a.band_rows = bg.band_rows;
        SPG_CUDA(h, cudaFuncSetAttribute(nms_peaks_banded_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bg.smem));
        nms_peaks_banded_kernel<<<std::min(items, h->sm_count), kNmsBThreads, bg.smem, st>>>(a, items, bg.slots, bg.n_bands);
        h->stage_kernel[0] = "nms_peaks_banded_kernel";
        h->launches++;
        SPG_CUDA(h, cudaGetLastError());
        return SPG_OK;
    }
    a.band_rows = std::max(4, std::min(H, 4096 / W));
    const size_t smem = nms_smem_bytes(a.band_rows, H, W, h->ws.capP);
    if (smem > h->smem_optin) return fail(h, SPG_E_INVALID, "map width %d needs %zu B of shared memory per band", W, smem);
    SPG_CUDA(h, cudaFuncSetAttribute(nms_peaks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nms_peaks_kernel<<<n * h->ws.K, kNmsThreads, smem, st>>>(a);
    h->stage_kernel[0] = "nms_peaks_kernel";
    h->launches++;
    SPG_CUDA(h, cudaGetLastError());
    return SPG_OK;
}

template <typename T, typename TA = T>
int launch_score_t(spg_handle *h, const ScoreArgs &a, int n, cudaStream_t st) {
    const size_t plane_bytes = (size_t)a.H * a.W * sizeof(T);
    const size_t staged = score_smem_bytes(plane_bytes, h->ws.capP);
    const bool aligned = (plane_bytes % 16 == 0) && ((a.img_stride * sizeof(T)) % 16 == 0) && ((a.chan_stride * sizeof(T)) % 16 == 0) &&
                         ((reinterpret_cast<uintptr_t>(a.paf) & 15) == 0) && plane_bytes < (1u << 20);
    const int grid = n * h->ws.L;
    if (sizeof(T) == 4 && h->persist && aligned && h->ws.capP <= kPersistMaxCapP &&
        persist_smem_bytes(plane_bytes, h->ws.capP) <= h->smem_optin) {
        // one resident CTA per SM walking a ring of 3 plane slots (loader / screeners / scorers)
        const size_t smem = persist_smem_bytes(plane_bytes, h->ws.capP);
        SPG_CUDA(h, cudaFuncSetAttribute(limb_score_persist_kernel<TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        limb_score_persist_kernel<TA><<<std::min(grid, h->sm_count), kPersistThreads, smem, st>>>(a, grid);
        h->stage_kernel[1] = sizeof(TA) == 4 ? "limb_score_persist_kernel<float>" : "limb_score_persist_kernel<double>";
    } else if (aligned && staged <= h->smem_optin) {
        SPG_CUDA(h, (cudaFuncSetAttribute(limb_score_kernel<T, true, TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)staged)));
        limb_score_kernel<T, true, TA><<<grid, kScoreThreads, staged, st>>>(a);
        h->stage_kernel[1] = sizeof(T) == 8 ? "limb_score_kernel<double,true>" : sizeof(TA) == 4 ? "limb_score_kernel<float,true>" : "limb_score_kernel<float,true,double>";
    } else {  // plane larger than shared memory (or unaligned): sample through L2
        const size_t smem = score_smem_bytes(0, h->ws.capP);
        limb_score_kernel<T, false, TA><<<grid, kScoreThreads, smem, st>>>(a);
        h->stage_kernel[1] = sizeof(T) == 8 ? "limb_score_kernel<double,false>" : sizeof(TA) == 4 ? "limb_score_kernel<float,false>" : "limb_score_kernel<float,false,double>";
    }
    h->launches++;
    SPG_CUDA(h, cudaGetLastError());
    return SPG_OK;
}

int launch_score(spg_handle *h, const void *paf, int dtype, int64_t img_stride, int64_t chan_stride, int base, int n, int H,
                 int W, double extent, const spg_params *p, cudaStream_t st) {
    if (n == 0) return SPG_OK;
    ScoreArgs a{};
    a.paf = paf;
    a.img_stride = img_stride;
    a.chan_stride = chan_stride;
    a.H = H;
    a.W = W;
    a.image_base = base;
    a.mid_num = p->mid_num;
    a.image_extent = extent;
    a.thre2 = p->thre2;
    a.connect_ration = p->connect_ration;
    a.screen = h->screen;
    a.crit1_strict = p->crit1_strict != 0;
    a.debug = 0;
#ifdef SPG_DEBUG  // timing-only knobs that change results exist only in -DSPG_DEBUG builds (never in the shipped library)
    if (const char *e = getenv("SPG_DEBUG_PERSIST")) a.debug = atoi(e);
#endif
    a.exact_warps = h->exact_warps;
    a.ws = h->ws;
    h->cand_dtype = dtype;
    if (dtype == SPG_F64) return launch_score_t<double>(h, a, n, st);
    if (dtype == SPG_F32_AS_F64) return launch_score_t<float, double>(h, a, n, st);
    return launch_score_t<float>(h, a, n, st);
}

int launch_match(spg_handle *h, int base, int n, cudaStream_t st) {
    if (n == 0) return SPG_OK;
    MatchArgs a{};
    a.n_images = n;
    a.image_base = base;
    a.keys_valid = h->cand_dtype == SPG_F32;
    a.ws = h->ws;
    const int warps = n * h->ws.L;
    const int blocks = (warps * 32 + kMatchThreads - 1) / kMatchThreads;
    limb_match_kernel<<<blocks, kMatchThreads, 0, st>>>(a);
    h->stage_kernel[2] = "limb_match_kernel";
    h->launches++;
    SPG_CUDA(h, cudaGetLastError());
    return SPG_OK;
}

int launch_assemble(spg_handle *h, int base, int n, const spg_params *p, cudaStream_t st) {
    if (n == 0) return SPG_OK;
    AssembleArgs a{};
    a.n_images = n;
    a.image_base = base;
    a.len_rate = p->len_rate;
    a.connection_tole = p->connection_tole;
    a.min_mean_score = p->min_mean_score;
    a.remove_recon = p->remove_recon;
    a.min_parts = p->min_parts;
    a.refresh_len_check = p->refresh_len_check != 0;
    a.wire_flag = h->armed_flag; a.wire_flag_value = h->armed_value; a.done_counter = h->done_counter;
    h->armed_flag = nullptr;  // one shot
    a.ws = h->ws;
    a.ws.wire_first += base;  // records are indexed by the image's position in the call
    a.use_bulk = ((size_t)h->ws.L * h->ws.capP * sizeof(uint32_t)) % 16 == 0;  // bulk copies move multiples of 16 bytes
    const size_t smem = assemble_smem_bytes(h->ws.K, h->ws.capP, h->ws.capR) + assemble_conn_bytes(h->ws.L, h->ws.capP);
    if (smem > h->smem_optin) return fail(h, SPG_E_INVALID, "capacities need %zu B of shared memory in assemble (limit %zu)", smem, h->smem_optin);
    SPG_CUDA(h, cudaFuncSetAttribute(assemble_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    assemble_kernel<<<n, kAssembleThreads, smem, st>>>(a);
    h->stage_kernel[3] = "assemble_kernel";
    h->launches++;
    SPG_CUDA(h, cudaGetLastError());
    return SPG_OK;
}

int launch_match_assemble(spg_handle *h, int base, int n, const spg_params *p, cudaStream_t st) {
    if (n == 0) return SPG_OK;
    AssembleArgs a{};
    a.n_images = n;
    a.image_base = base;
    a.len_rate = p->len_rate;
    a.connection_tole = p->connection_tole;
    a.min_mean_score = p->min_mean_score;
    a.remove_recon = p->remove_recon;
    a.min_parts = p->min_parts;
    a.refresh_len_check = p->refresh_len_check != 0;
    a.wire_flag = h->armed_flag; a.wire_flag_value = h->armed_value; a.done_counter = h->done_counter;
    a.ws = h->ws;
    a.ws.wire_first += base;
    a.use_bulk = ((size_t)h->ws.K * h->ws.capP * sizeof(float)) % 16 == 0;  // bulk copies move multiples of 16 bytes
    const size_t smem = match_assemble_smem_bytes(h->ws.K, h->ws.L, h->ws.capP, h->ws.capR, h->ma_warps);
    if (smem > h->smem_optin) {  // very large capacities: the two stand-alone kernels need less shared memory
        int rc;
        if ((rc = launch_match(h, base, n, st))) return rc;
        return launch_assemble(h, base, n, p, st);  // consumes the armed signal itself
    }
    h->armed_flag = nullptr;  // one shot
    SPG_CUDA(h, cudaFuncSetAttribute(match_assemble_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    match_assemble_kernel<<<n, 32 * (1 + h->ma_warps), smem, st>>>(a, h->cand_dtype == SPG_F32);
    h->stage_kernel[2] = "match_assemble_kernel";
    h->stage_kernel[3] = "";
    h->launches++;
    SPG_CUDA(h, cudaGetLastError());
    return SPG_OK;
}

int run_all(spg_handle *h, const float *heat, int64_t his, int64_t hcs, const void *paf, int dtype, int64_t pis, int64_t pcs,
            int base, int n, int H, int W, double extent, const spg_params *p, cudaStream_t st) {
    int rc;
    SPG_CUDA(h, cudaMemsetAsync(h->ws.status + base, 0, sizeof(uint32_t) * (size_t)n, st));
    if ((rc = launch_nms(h, heat, his, hcs, base, n, H, W, p, st))) return rc;
    if ((rc = launch_score(h, paf, dtype, pis, pcs, base, n, H, W, extent, p, st))) return rc;
    if (h->fuse_ma) return launch_match_assemble(h, base, n, p, st);
    if ((rc = launch_match(h, base, n, st))) return rc;
    if ((rc = launch_assemble(h, base, n, p, st))) return rc;
    return SPG_OK;
}

__global__ void wire_signal_kernel(unsigned long long *word, unsigned long long value) {
    __threadfence_system();  // everything earlier on the stream has completed; order it before the flag for every observer
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(word), "l"(value) : "memory");
}

struct WireWords {
    unsigned long long *p[32];
    int n;
};
__global__ void wire_signal_many_kernel(WireWords w, unsigned long long value) {
    __threadfence_system();
    if ((int)threadIdx.x < w.n) asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(w.p[threadIdx.x]), "l"(value) : "memory");
}

__global__ void wire_wait_kernel(const unsigned long long *word, unsigned long long value) {
    unsigned long long v;
    do {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(word) : "memory");
        if (v < value) __nanosleep(500);
    } while (v < value);
}

}  // namespace

extern "C" {

#ifdef SPG_TRACE  // development builds only (make trace): the clock trace of the first CTAs of the last launches
int spg_trace_read(unsigned long long *out, size_t n_words, int clear) {
    const size_t n = std::min(n_words, (size_t)spg::kTraceCtas * spg::kTraceSlots);
    if (cudaMemcpyFromSymbol(out, spg::g_spg_trace, n * sizeof(unsigned long long)) != cudaSuccess) return -1;
    if (clear) {
        void *p = nullptr;
        if (cudaGetSymbolAddress(&p, spg::g_spg_trace) != cudaSuccess) return -1;
        if (cudaMemset(p, 0, sizeof(spg::g_spg_trace)) != cudaSuccess) return -1;
    }
    return 0;
}
#endif

int spg_abi_version(void) { return SPG_ABI_VERSION; }

const char *spg_last_error(const spg_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int spg_create(const spg_config *cfg, spg_handle **out) {
    if (!cfg || !out) return fail(nullptr, SPG_E_INVALID, "cfg/out is NULL");
    *out = nullptr;
    if (cfg->abi_version != SPG_ABI_VERSION) return fail(nullptr, SPG_E_INVALID, "ABI version %d != %d", cfg->abi_version, SPG_ABI_VERSION);
    if (cfg->n_parts < 1 || cfg->n_parts > kMaxParts || cfg->n_limbs < 1 || cfg->n_limbs > kMaxLimbs || !cfg->limbs)
        return fail(nullptr, SPG_E_INVALID, "n_parts in [1,%d], n_limbs in [1,%d], limbs non-NULL required", kMaxParts, kMaxLimbs);
    if (cfg->n_out_joints < 0 || cfg->n_out_joints > kMaxOutJoints || (cfg->n_out_joints && !cfg->out_from_part))
        return fail(nullptr, SPG_E_INVALID, "n_out_joints in [0,%d]", kMaxOutJoints);
    if (cfg->max_peaks_per_part < 1 || cfg->max_peaks_per_part > kMaxCapPeaks)
        return fail(nullptr, SPG_E_INVALID, "max_peaks_per_part in [1,%d]", kMaxCapPeaks);
    if (cfg->max_person_rows < 1 || cfg->max_person_rows > kMaxCapRows)
        return fail(nullptr, SPG_E_INVALID, "max_person_rows in [1,%d]", kMaxCapRows);
    if (cfg->max_cands_per_limb < 1 || cfg->max_batch < 1 || cfg->max_h < 2 || cfg->max_w < 2)
        return fail(nullptr, SPG_E_INVALID, "max_cands_per_limb, max_batch >= 1 and max_h, max_w >= 2 required");
    for (int k = 0; k < cfg->n_limbs * 2; k++)
        if (cfg->limbs[k] < 0 || cfg->limbs[k] >= cfg->n_parts) return fail(nullptr, SPG_E_INVALID, "limb table entry %d out of range", k);
    for (int g = 0; g < cfg->n_out_joints; g++)
        if (cfg->out_from_part[g] < 0 || cfg->out_from_part[g] >= cfg->n_parts) return fail(nullptr, SPG_E_INVALID, "out_from_part[%d] out of range", g);

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(nullptr, SPG_E_NO_DEVICE, "no CUDA device (this library has no CPU path)");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, SPG_E_INVALID, "device %d outside [0,%d)", cfg->device, ndev);
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) return fail(nullptr, SPG_E_CUDA, "cudaGetDeviceProperties failed");
    if (prop.major != 10) return fail(nullptr, SPG_E_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, prop.major, prop.minor);

    spg_handle *h = new (std::nothrow) spg_handle();
    if (!h) return fail(nullptr, SPG_E_INVALID, "out of host memory");
    h->cfg = *cfg;
    h->cfg.limbs = nullptr;
    h->cfg.out_from_part = nullptr;
    h->device = cfg->device;
    h->sm_count = prop.multiProcessorCount;
    h->smem_optin = prop.sharedMemPerBlockOptin;
    if (const char *e = getenv("SPG_NO_SCREEN")) h->screen = !(e[0] == '1');
    if (const char *e = getenv("SPG_PERSIST")) h->persist = !(e[0] == '0');  // 0: per-item kernels only (A/B tests)
    if (const char *e = getenv("SPG_MA_WARPS")) h->ma_warps = std::max(1, std::min(15, atoi(e)));
    if (const char *e = getenv("SPG_FUSE_MA")) h->fuse_ma = !(e[0] == '0');
    if (const char *e = getenv("SPG_POST_IDENT")) h->post_generic_ident = atoi(e) == 0;
    if (const char *e = getenv("SPG_EXACT_WARPS")) h->exact_warps = std::max(1, std::min(30, atoi(e)));  // the kernel keeps >= 1 screener
    DeviceGuard guard(h->device);

    const size_t N = cfg->max_batch, K = cfg->n_parts, L = cfg->n_limbs, J = cfg->n_out_joints;
    const size_t cP = cfg->max_peaks_per_part, cC = cfg->max_cands_per_limb, cR = cfg->max_person_rows;
    Workspace &ws = h->ws;
    ws.K = (int)K; ws.L = (int)L; ws.J = (int)J; ws.capP = (int)cP; ws.capC = (int)cC; ws.capR = (int)cR; ws.max_batch = (int)N;
    int rc = SPG_OK;
    auto A = [&](int r) { if (rc == SPG_OK) rc = r; };
    A(dalloc(h, &ws.peak_x, N * K * cP));
    A(dalloc(h, &ws.peak_y, N * K * cP));
    A(dalloc(h, &ws.peak_score, N * K * cP));
    A(dalloc(h, &ws.peak_anchor, N * K * cP));
    A(dalloc(h, &ws.peak_count, N * K));
    A(dalloc(h, &ws.cand_prio, N * L * cC));
    A(dalloc(h, &ws.cand_score, N * L * cC));
    A(dalloc(h, &ws.cand_ij, N * L * cC));
    A(dalloc(h, &ws.cand_key, N * L * cC));
    A(dalloc(h, &ws.cand_count, N * L));
    A(dalloc(h, &ws.surv_count, N * L));
    A(dalloc(h, &ws.conn_ij, N * L * cP));
    A(dalloc(h, &ws.conn_score, N * L * cP));
    A(dalloc(h, &ws.conn_norm, N * L * cP));
    A(dalloc(h, &ws.conn_count, N * L));
    A(dalloc(h, &ws.subset, N * cR * (K + 2) * 2));
    A(dalloc(h, &ws.n_persons, N));
    A(dalloc(h, &ws.people_xy, N * cR * std::max<size_t>(J, 1) * 2));
    A(dalloc(h, &ws.people_score, N * cR));
    A(dalloc(h, &ws.status, N));
    for (size_t i = 0; i < L * 2; i++) ws.limbs[i] = (int16_t)cfg->limbs[i];
    for (size_t g = 0; g < J; g++) ws.out_from_part[g] = (int16_t)cfg->out_from_part[g];
    if (rc == SPG_OK && cudaMemset(ws.status, 0, sizeof(uint32_t) * N) != cudaSuccess) rc = SPG_E_CUDA;
    if (rc == SPG_OK && cudaMemset(ws.peak_count, 0, sizeof(int32_t) * N * K) != cudaSuccess) rc = SPG_E_CUDA;
    for (int s = 0; s < 2 && rc == SPG_OK; s++)
        if (cudaStreamCreateWithFlags(&h->streams[s], cudaStreamNonBlocking) != cudaSuccess) rc = SPG_E_CUDA;
    if (rc != SPG_OK) {
        g_create_error = h->err.empty() ? "device allocation failed" : h->err;
        spg_destroy(h);
        return rc;
    }
    *out = h;
    return SPG_OK;
}

void spg_destroy(spg_handle *h) {
    if (!h) return;
    DeviceGuard guard(h->device);
    cudaDeviceSynchronize();
    for (void *p : h->allocs) cudaFree(p);
    if (h->in_heat) cudaFree(h->in_heat);
    if (h->in_paf) cudaFree(h->in_paf);
    if (h->heat_acc) cudaFree(h->heat_acc);
    if (h->pre_img) cudaFree(h->pre_img);
    if (h->done_counter) cudaFree(h->done_counter);
    for (auto &s : h->streams)
        if (s) cudaStreamDestroy(s);
    delete h;
}

int spg_get_device_view(const spg_handle *h, spg_device_view *v) {
    if (!h || !v) return SPG_E_INVALID;
    const Workspace &ws = h->ws;
    v->max_batch = ws.max_batch; v->n_parts = ws.K; v->n_limbs = ws.L; v->n_out_joints = ws.J;
    v->cap_peaks = ws.capP; v->cap_cands = ws.capC; v->cap_rows = ws.capR;
    v->peak_x = ws.peak_x; v->peak_y = ws.peak_y; v->peak_score = ws.peak_score; v->peak_anchor = ws.peak_anchor;
    v->peak_count = ws.peak_count;
    v->conn_ij = ws.conn_ij; v->conn_score = ws.conn_score; v->conn_norm = ws.conn_norm; v->conn_count = ws.conn_count;
    v->cand_count = ws.cand_count;
    v->surv_count = ws.surv_count;
    v->subset = ws.subset; v->n_persons = ws.n_persons; v->people_xy = ws.people_xy; v->people_score = ws.people_score;
    v->status = ws.status;
    return SPG_OK;
}

// ---- wire records + peer memory + stream-ordered signalling ------------------------------------------------------
int64_t spg_wire_record_bytes(const spg_handle *h) {
    if (!h) return 0;
    const int rows = h->ws.wire_rows > 0 ? h->ws.wire_rows : h->ws.capR;
    return 8 + (int64_t)rows * (2 * h->ws.J + 2) * (int64_t)sizeof(double);
}

int spg_set_wire_output(spg_handle *h, void *wire_dev, int64_t first_record, int32_t wire_rows) {
    if (!h) return SPG_E_INVALID;
    if (!wire_dev) {
        h->ws.wire = nullptr;
        h->ws.wire_first = 0;
        return SPG_OK;
    }
    if (wire_rows < 1 || wire_rows > h->ws.capR) return fail(h, SPG_E_INVALID, "wire_rows %d outside [1, max_person_rows=%d]", wire_rows, h->ws.capR);
    if (first_record < 0) return fail(h, SPG_E_INVALID, "first_record is negative");
    if ((reinterpret_cast<uintptr_t>(wire_dev) & 7) != 0) return fail(h, SPG_E_INVALID, "wire buffer must be 8-byte aligned");
    if ((size_t)wire_rows * (2 * h->ws.J + 2) * sizeof(double) > assemble_conn_bytes(h->ws.L, h->ws.capP))
        return fail(h, SPG_E_INVALID, "wire_rows %d do not fit the assemble kernel's staging area", wire_rows);
    h->ws.wire = static_cast<unsigned char *>(wire_dev);
    h->ws.wire_first = first_record;
    h->ws.wire_rows = wire_rows;
    return SPG_OK;
}

int spg_arm_wire_signal(spg_handle *h, uint64_t *word_dev, uint64_t value) {
    if (!h) return SPG_E_INVALID;
    if (!word_dev) {
        h->armed_flag = nullptr;
        return SPG_OK;
    }
    if (!h->ws.wire) return fail(h, SPG_E_STATE, "spg_arm_wire_signal needs a wire output (spg_set_wire_output) first");
    if (!h->done_counter) {
        DeviceGuard guard(h->device);
        SPG_CUDA(h, cudaMalloc(&h->done_counter, sizeof(unsigned int)));
        SPG_CUDA(h, cudaMemset(h->done_counter, 0, sizeof(unsigned int)));
    }
    h->armed_flag = reinterpret_cast<unsigned long long *>(word_dev);
    h->armed_value = value;
    return SPG_OK;
}

int spg_wire_create(int32_t device, uint64_t bytes, void **dev_ptr, unsigned char ipc_handle[64]) {
    if (!dev_ptr || !ipc_handle || bytes == 0) return SPG_E_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DeviceGuard guard(device);
    void *p = nullptr;
    // a dedicated cudaMalloc allocation: an IPC handle exports the whole allocation it points into
    if (cudaMalloc(&p, bytes) != cudaSuccess) return fail(nullptr, SPG_E_CUDA, "cudaMalloc of %llu wire bytes failed", (unsigned long long)bytes);
    cudaIpcMemHandle_t hd;
    if (cudaMemset(p, 0, bytes) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess || cudaIpcGetMemHandle(&hd, p) != cudaSuccess) {
        const char *why = cudaGetErrorString(cudaGetLastError());
        cudaFree(p);
        return fail(nullptr, SPG_E_CUDA, "exporting the wire buffer failed: %s", why);
    }
    memcpy(ipc_handle, &hd, 64);
    *dev_ptr = p;
    return SPG_OK;
}

int spg_wire_open(int32_t device, const unsigned char ipc_handle[64], void **peer_ptr) {
    if (!peer_ptr || !ipc_handle) return SPG_E_INVALID;
    DeviceGuard guard(device);
    cudaIpcMemHandle_t hd;
    memcpy(&hd, ipc_handle, 64);
    void *p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, SPG_E_CUDA, "cudaIpcOpenMemHandle failed: %s (no peer access between the two GPUs?)", cudaGetErrorString(e));
    }
    *peer_ptr = p;
    return SPG_OK;
}

int spg_wire_close(void *peer_ptr) { return (!peer_ptr || cudaIpcCloseMemHandle(peer_ptr) == cudaSuccess) ? SPG_OK : SPG_E_CUDA; }

int spg_wire_destroy(int32_t device, void *dev_ptr) {
    if (!dev_ptr) return SPG_OK;
    DeviceGuard guard(device);
    cudaDeviceSynchronize();
    return cudaFree(dev_ptr) == cudaSuccess ? SPG_OK : SPG_E_CUDA;
}

int spg_wire_signal(int32_t device, uint64_t *word_dev, uint64_t value, void *stream) {
    if (!word_dev) return SPG_E_INVALID;
    DeviceGuard guard(device);
    wire_signal_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<unsigned long long *>(word_dev), value);
    return cudaGetLastError() == cudaSuccess ? SPG_OK : fail(nullptr, SPG_E_CUDA, "wire_signal launch failed");
}

int spg_wire_signal_many(int32_t device, uint64_t *const *words_dev, int32_t n_words, uint64_t value, void *stream) {
    if (!words_dev || n_words < 1 || n_words > 32) return SPG_E_INVALID;
    DeviceGuard guard(device);
    WireWords w{};
    w.n = n_words;
    for (int i = 0; i < n_words; i++) {
        if (!words_dev[i]) return SPG_E_INVALID;
        w.p[i] = reinterpret_cast<unsigned long long *>(words_dev[i]);
    }
    wire_signal_many_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(w, value);
    return cudaGetLastError() == cudaSuccess ? SPG_OK : fail(nullptr, SPG_E_CUDA, "wire_signal_many launch failed");
}

int spg_wire_wait(int32_t device, const uint64_t *word_dev, uint64_t value, void *stream) {
    if (!word_dev) return SPG_E_INVALID;
    DeviceGuard guard(device);
    // cuStreamWaitValue64 through the runtime's driver entry-point lookup (no link-time dependency on libcuda)
    typedef int (*wait_fn_t)(cudaStream_t, unsigned long long, unsigned long long, unsigned int);
    static wait_fn_t wait_fn = nullptr;
    static bool looked = false;
    if (!looked) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuStreamWaitValue64", &fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            wait_fn = reinterpret_cast<wait_fn_t>(fn);
        cudaGetLastError();
        looked = true;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (wait_fn && wait_fn(st, (unsigned long long)reinterpret_cast<uintptr_t>(word_dev), value, 0u /* CU_STREAM_WAIT_VALUE_GEQ */) == 0) return SPG_OK;
    // no stream memory operations on this driver: a one-thread polling kernel (sleeps between polls)
    wire_wait_kernel<<<1, 1, 0, st>>>(reinterpret_cast<const unsigned long long *>(word_dev), value);
    return cudaGetLastError() == cudaSuccess ? SPG_OK : fail(nullptr, SPG_E_CUDA, "wire_wait launch failed");
}

int64_t spg_launch_count(const spg_handle *h) { return h ? h->launches : 0; }

const char *spg_stage_kernel(const spg_handle *h, int32_t stage) { return (h && stage >= 0 && stage < 5) ? h->stage_kernel[stage] : ""; }

// ---- post-network stage ------------------------------------------------------------------------
namespace {

// Checks shared by spg_postnet and spg_postnet_rotated; allocates the float64 keypoint sums when they outlive a launch
// and fills the arguments common to every launch of the call.  *done is set when there is nothing to launch (n == 0).
int postnet_setup(spg_handle *h, const spg_postnet_desc *d, int32_t n, int32_t H, int32_t W, float *heat_out, void *paf_out,
                  int32_t paf_dtype, bool rotated, PostArgs &a, bool *done) {
    *done = true;
    if (!d || !d->scales || d->n_scales < 1 || !d->flip_paf_ord || !d->flip_heat_ord) return fail(h, SPG_E_INVALID, "postnet descriptor incomplete");
    if ((!heat_out || !paf_out) && n > 0) return fail(h, SPG_E_INVALID, "heat_out/paf_out is NULL");
    if (paf_dtype != SPG_F32 && paf_dtype != SPG_F64) return fail(h, SPG_E_INVALID, "paf_dtype must be SPG_F32 or SPG_F64");
    if (paf_dtype == SPG_F32 && d->n_scales != 1)
        return fail(h, SPG_E_INVALID, "float32 body-part planes hold the reference's float64 values only for a single scale");
    if (d->stride < 1 || d->stride > 16) return fail(h, SPG_E_INVALID, "stride outside [1,16]");
    int rc;
    if ((rc = check_dims(h, n, H, W))) return rc;
    if (n == 0) return SPG_OK;
    const Workspace &ws = h->ws;
    if (ws.K + ws.L > kMaxNetChannels) return fail(h, SPG_E_INVALID, "too many channels for postnet");
    DeviceGuard guard(h->device);
    // float64 keypoint sums that outlive a launch: rotated items run one launch each
    if (d->n_scales > 1 && (rotated || d->stride != 4 || d->n_scales > kPostMaxScales)) {
        const size_t need = (size_t)h->cfg.max_batch * ws.K * H * W;
        if (h->heat_acc_elems < need) {
            if (h->heat_acc) cudaFree(h->heat_acc);
            h->heat_acc = nullptr; h->heat_acc_elems = 0;
            SPG_CUDA(h, cudaMalloc(&h->heat_acc, need * sizeof(double)));
            h->heat_acc_elems = need;
        }
    }
    // validate every scale and fill the common arguments
    a = PostArgs{};
    a.stride = d->stride; a.H = H; a.W = W; a.n_out = ws.K + ws.L; a.K = ws.K;
    for (int c = 0; c < ws.K; c++) {
        if (d->flip_heat_ord[c] < 0 || d->flip_heat_ord[c] >= ws.K) return fail(h, SPG_E_INVALID, "flip_heat_ord[%d] out of range", c);
        a.src_chan[c] = (short)(d->heat_chan0 + c);
        a.flip_chan[c] = (short)(d->heat_chan0 + d->flip_heat_ord[c]);
    }
    for (int k = 0; k < ws.L; k++) {
        if (d->flip_paf_ord[k] < 0 || d->flip_paf_ord[k] >= ws.L) return fail(h, SPG_E_INVALID, "flip_paf_ord[%d] out of range", k);
        a.src_chan[ws.K + k] = (short)(d->paf_chan0 + k);
        a.flip_chan[ws.K + k] = (short)(d->paf_chan0 + d->flip_paf_ord[k]);
    }
    a.heat = heat_out; a.paf = paf_out; a.heat_acc = h->heat_acc; a.paf_is_f64 = paf_dtype == SPG_F64;
    a.n_scales = d->n_scales; a.nan_scrub = d->nan_scrub != 0;
    a.sx1 = 1.0 / (double)d->stride; a.sy1 = a.sx1;  // cv2.resize(fx = stride): scale = 1/fx
    for (int t = 0; t < d->n_scales; t++) {
        const spg_postnet_scale &sc = d->scales[t];
        if (!sc.net_out) return fail(h, SPG_E_INVALID, "scale %d: net_out is NULL", t);
        if (sc.dtype != SPG_F32 && sc.dtype != SPG_F16) return fail(h, SPG_E_INVALID, "scale %d: network output must be SPG_F32 or SPG_F16", t);
        if (sc.h < 1 || sc.w < 1 || sc.crop_h < 1 || sc.crop_w < 1 || sc.crop_h > sc.h * d->stride || sc.crop_w > sc.w * d->stride)
            return fail(h, SPG_E_INVALID, "scale %d: crop %dx%d does not fit the up-sampled %dx%d output", t, sc.crop_h, sc.crop_w, sc.h * d->stride, sc.w * d->stride);
    }
    *done = false;
    return SPG_OK;
}

PostScale postnet_scale_of(const spg_postnet_scale &sc, int H, int W) {
    PostScale s{};
    s.net = sc.net_out; s.net_is_f16 = sc.dtype == SPG_F16;
    s.img_stride = sc.image_stride; s.pair_stride = sc.pair_stride; s.chan_stride = sc.chan_stride;
    s.h = sc.h; s.w = sc.w; s.crop_h = sc.crop_h; s.crop_w = sc.crop_w;
    // cv2.resize(dsize): inv_scale = dst/src, scale = 1/inv_scale (two roundings, as OpenCV)
    s.sx2 = 1.0 / ((double)W / (double)sc.crop_w);
    s.sy2 = 1.0 / ((double)H / (double)sc.crop_h);
    return s;
}

// The items [t_begin, t_end) of the loop (angle 0) with the stride-4 or the generic kernels; a.n_scales is the length of
// the whole loop, so sums that continue from earlier items, or into later ones, go through memory.
int postnet_launch_items(spg_handle *h, PostArgs &a, const spg_postnet_desc *d, int t_begin, int t_end, int32_t n, int32_t H,
                         int32_t W, cudaStream_t st) {
    // output tile: as large as the shared-memory tiles of the intermediate / source allow
    auto tile_dim = [&](double s2, double s1, int cap1, int cap0, int maxd, double margin) {
        const double c1 = std::min((double)cap1, ((double)cap0 - 7.0) / s1) - margin;  // intermediate span allowed
        return std::max(1, std::min(maxd, (int)(c1 / std::max(s2, 1e-6))));
    };
    const bool fast = d->stride == 4;  // the reference's model: four-phase kernel; other strides: table-driven generic kernel
    if (fast) {
        // the scale loop runs INSIDE the kernel (groups of kPostMaxScales): one tile geometry for all fused scales
        for (int t0 = t_begin; t0 < t_end; t0 += kPostMaxScales) {
            a.n_fused = std::min(kPostMaxScales, t_end - t0);
            a.scale_index = t0;
            a.tile_w = kPostTW; a.tile_h = kPostTH;
            for (int t = 0; t < a.n_fused; t++) {
                a.sc[t] = postnet_scale_of(d->scales[t0 + t], H, W);
                a.tile_w = std::min(a.tile_w, tile_dim(a.sc[t].sx2, a.sx1, kPostF_C1, kPostF_CS, kPostTW, 13.0));
                a.tile_h = std::min(a.tile_h, tile_dim(a.sc[t].sy2, a.sy1, kPostF_R1, kPostF_RS, kPostTH, 13.0));
            }
            a.tiles_x = (W + a.tile_w - 1) / a.tile_w;
            a.tiles_y = (H + a.tile_h - 1) / a.tile_h;
            if ((long long)a.tiles_x * a.tiles_y > 0x7fffffffLL || n > 65535) return fail(h, SPG_E_INVALID, "postnet grid too large");
            // a CTA builds its tile's tables once and walks over a chunk of channels -- as many as still leave
            // ~16 CTAs per SM in the grid (3 resident: several waves)
            const long long tiles = (long long)a.tiles_x * a.tiles_y * n;
            const int n_chunks = (int)std::min<long long>(a.n_out, std::max<long long>(1, ((long long)h->sm_count * 16 + tiles - 1) / tiles));
            a.chan_chunk = (a.n_out + n_chunks - 1) / n_chunks;
            dim3 grid((unsigned)(a.tiles_x * a.tiles_y), (unsigned)((a.n_out + a.chan_chunk - 1) / a.chan_chunk), (unsigned)n);
            bool ident = true, any16 = false, all16 = true;
            for (int t = 0; t < a.n_fused; t++) {
                ident = ident && a.sc[t].crop_h == H && a.sc[t].crop_w == W;
                any16 = any16 || a.sc[t].net_is_f16;
                all16 = all16 && a.sc[t].net_is_f16;
            }
            if (any16 != all16) return fail(h, SPG_E_INVALID, "the network outputs of all scales must have the same dtype");
            const bool single = d->n_scales == 1;
            const size_t smem = postF_smem_bytes(single ? 1 : kPostMaxScales);
#define SPG_POST_LAUNCH(S_, I_, F_)                                                                                           \
    do {                                                                                                                      \
        SPG_CUDA(h, (cudaFuncSetAttribute(postnet_kernel<S_, I_, F_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem))); \
        postnet_kernel<S_, I_, F_><<<grid, kPostThreads, smem, st>>>(a);                                                      \
    } while (0)
            if (single && ident && !h->post_generic_ident) {  // the reference's default: its own kernel (two passes, per-thread state hoisted)
                a.tile_w = kPostI_TW; a.tile_h = kPostI_TH;
                a.tiles_x = (W + a.tile_w - 1) / a.tile_w;
                a.tiles_y = (H + a.tile_h - 1) / a.tile_h;
                const long long tiles_i = (long long)a.tiles_x * a.tiles_y * n;
                const int chunks_i = (int)std::min<long long>(a.n_out, std::max<long long>(1, ((long long)h->sm_count * 32 + tiles_i - 1) / tiles_i));
                a.chan_chunk = (a.n_out + chunks_i - 1) / chunks_i;
                dim3 grid_i((unsigned)(a.tiles_x * a.tiles_y), (unsigned)((a.n_out + a.chan_chunk - 1) / a.chan_chunk), (unsigned)n);
                if (all16) postnet_x4_ident_kernel<true><<<grid_i, kPostThreads, 0, st>>>(a);
                else postnet_x4_ident_kernel<false><<<grid_i, kPostThreads, 0, st>>>(a);
                h->stage_kernel[4] = "postnet_x4_ident_kernel";
            } else if (single) {
                h->stage_kernel[4] = "postnet_kernel";
                if (ident) { if (all16) SPG_POST_LAUNCH(true, true, true); else SPG_POST_LAUNCH(true, true, false); }
                else { if (all16) SPG_POST_LAUNCH(true, false, true); else SPG_POST_LAUNCH(true, false, false); }
            } else {
                h->stage_kernel[4] = "postnet_kernel";
                if (ident) { if (all16) SPG_POST_LAUNCH(false, true, true); else SPG_POST_LAUNCH(false, true, false); }
                else { if (all16) SPG_POST_LAUNCH(false, false, true); else SPG_POST_LAUNCH(false, false, false); }
            }
#undef SPG_POST_LAUNCH
            h->launches++;
            SPG_CUDA(h, cudaGetLastError());
        }
        return SPG_OK;
    }
    for (int t = t_begin; t < t_end; t++) {  // generic kernel: one launch per scale, float64 accumulators in memory
        const PostScale s = postnet_scale_of(d->scales[t], H, W);
        a.net = s.net; a.net_is_f16 = s.net_is_f16; a.img_stride = s.img_stride; a.pair_stride = s.pair_stride; a.chan_stride = s.chan_stride;
        a.h = s.h; a.w = s.w; a.crop_h = s.crop_h; a.crop_w = s.crop_w; a.sx2 = s.sx2; a.sy2 = s.sy2;
        a.scale_index = t;
        a.tile_w = tile_dim(a.sx2, a.sx1, kPostC1, kPostCS, kPostTW, 7.0);
        a.tile_h = tile_dim(a.sy2, a.sy1, kPostR1, kPostRS, kPostTH, 7.0);
        a.tiles_x = (W + a.tile_w - 1) / a.tile_w;
        a.tiles_y = (H + a.tile_h - 1) / a.tile_h;
        if ((long long)a.tiles_x * a.tiles_y > 0x7fffffffLL || n > 65535) return fail(h, SPG_E_INVALID, "postnet grid too large");
        a.chan_chunk = 1;
        dim3 grid((unsigned)(a.tiles_x * a.tiles_y), (unsigned)a.n_out, (unsigned)n);
        postnet_generic_kernel<<<grid, kPostThreads, 0, st>>>(a);
        h->stage_kernel[4] = "postnet_generic_kernel";
        h->launches++;
        SPG_CUDA(h, cudaGetLastError());
    }
    return SPG_OK;
}

// cv2.getRotationMatrix2D((rows / 2, cols / 2), angle, 1) -- the centre is a Point2f, (rows, cols) passed as (x, y) as the
// reference does (evaluate.py:109-110) -- then the inversion cv2.warpAffine applies without WARP_INVERSE_MAP
// (imgproc/src/imgwarp.cpp), all in float64: the destination -> source map of the warp.
void rotation_inverse_map(double angle_deg, int rows, int cols, double m[6]) {
    const double cx = (double)(float)(rows / 2.0), cy = (double)(float)(cols / 2.0);
    const double ang = angle_deg * (3.14159265358979323846 / 180);
    const double alpha = std::cos(ang), beta = std::sin(ang);
    m[0] = alpha; m[1] = beta; m[2] = (1 - alpha) * cx - beta * cy;
    m[3] = -beta; m[4] = alpha; m[5] = beta * cx + (1 - alpha) * cy;
    double D = m[0] * m[4] - m[1] * m[3];
    D = D != 0 ? 1. / D : 0;
    const double a11 = m[4] * D, a22 = m[0] * D;
    m[0] = a11; m[1] *= -D;
    m[3] *= -D; m[4] = a22;
    const double b1 = -m[0] * m[2] - m[1] * m[5];
    const double b2 = -m[3] * m[2] - m[4] * m[5];
    m[2] = b1; m[5] = b2;
}

// Item t of the loop with a non-zero angle: one postnet_rot_kernel launch.
int postnet_launch_rotated(spg_handle *h, PostArgs &a, const spg_postnet_desc *d, int t, double angle_deg, int32_t n, int32_t H,
                           int32_t W, cudaStream_t st) {
    const PostScale s = postnet_scale_of(d->scales[t], H, W);
    a.net = s.net; a.net_is_f16 = s.net_is_f16; a.img_stride = s.img_stride; a.pair_stride = s.pair_stride; a.chan_stride = s.chan_stride;
    a.h = s.h; a.w = s.w; a.crop_h = s.crop_h; a.crop_w = s.crop_w; a.sx2 = s.sx2; a.sy2 = s.sy2;
    a.scale_index = t;
    PostRotArgs r{};
    r.Hp = s.h * a.stride; r.Wp = s.w * a.stride;
    rotation_inverse_map(-angle_deg, r.Hp, r.Wp, r.m);  // rotate_matrix_reverse (evaluate.py:110)
    // Tile: the largest of a ladder whose shared-memory tiles fit 64 KB (three CTAs per SM).  Capacities are upper bounds
    // of the spans the kernel finds: footprint = taps of the second resize (span (tile - 1) * ratio + 4, +1 for float
    // rounding); box = the footprint's rotated extent (|m0| fw + |m1| fh for x) + 2 for the floors of the fixed-point
    // taps and the second bilinear tap, +1 spare; source = taps of the x stride resize ((box - 1) / stride + 5, +1).
    const bool identity = s.crop_h == H && s.crop_w == W;
    static const int ladder[][2] = {{64, 32}, {32, 32}, {32, 16}, {16, 16}, {16, 8}, {8, 8}, {4, 4}, {2, 2}, {1, 1}};
    size_t smem = 0;
    bool fits = false;
    for (const auto &tl : ladder) {
        const int tw = std::min(tl[0], W), th = std::min(tl[1], H);
        const int fw = identity ? tw : std::min(s.crop_w, (int)std::ceil((tw - 1) * s.sx2) + 6);
        const int fh = identity ? th : std::min(s.crop_h, (int)std::ceil((th - 1) * s.sy2) + 6);
        const int bw = std::min(r.Wp, (int)std::ceil(std::fabs(r.m[0]) * (fw - 1) + std::fabs(r.m[1]) * (fh - 1)) + 4);
        const int bh = std::min(r.Hp, (int)std::ceil(std::fabs(r.m[3]) * (fw - 1) + std::fabs(r.m[4]) * (fh - 1)) + 4);
        const int cs = std::min(s.w, (int)std::ceil((bw - 1) / (double)a.stride) + 6);
        const int rs = std::min(s.h, (int)std::ceil((bh - 1) / (double)a.stride) + 6);
        a.tile_w = tw; a.tile_h = th;
        r.cap_fw = fw; r.cap_fh = fh; r.cap_bw = bw; r.cap_bh = bh; r.cap_cs = cs; r.cap_rs = rs;
        smem = postrot_smem_bytes(tw, th, fw, fh, bw, bh, cs, rs);
        if (smem <= 64 * 1024) { fits = true; break; }
    }
    if (!fits && smem > h->smem_optin)
        return fail(h, SPG_E_INVALID, "item %d: a %dx%d crop resized to %dx%d needs %zu bytes of shared memory even for a 1x1 tile", t,
                    s.crop_h, s.crop_w, H, W, smem);
    a.tiles_x = (W + a.tile_w - 1) / a.tile_w;
    a.tiles_y = (H + a.tile_h - 1) / a.tile_h;
    if ((long long)a.tiles_x * a.tiles_y > 0x7fffffffLL || n > 65535) return fail(h, SPG_E_INVALID, "postnet grid too large");
    // tables once per CTA, then a chunk of channels: as many chunks as leave ~16 CTAs per SM in the grid
    const long long tiles = (long long)a.tiles_x * a.tiles_y * n;
    const int n_chunks = (int)std::min<long long>(a.n_out, std::max<long long>(1, ((long long)h->sm_count * 16 + tiles - 1) / tiles));
    a.chan_chunk = (a.n_out + n_chunks - 1) / n_chunks;
    r.a = a;
    dim3 grid((unsigned)(a.tiles_x * a.tiles_y), (unsigned)((a.n_out + a.chan_chunk - 1) / a.chan_chunk), (unsigned)n);
    SPG_CUDA(h, cudaFuncSetAttribute(postnet_rot_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    postnet_rot_kernel<<<grid, kPostThreads, smem, st>>>(r);
    h->stage_kernel[4] = "postnet_rot_kernel";
    h->launches++;
    SPG_CUDA(h, cudaGetLastError());
    return SPG_OK;
}

}  // namespace

int spg_postnet(spg_handle *h, const spg_postnet_desc *d, int32_t n, int32_t H, int32_t W, float *heat_out, void *paf_out,
                int32_t paf_dtype, void *stream) {
    if (!h) return SPG_E_INVALID;
    PostArgs a;
    bool done;
    int rc = postnet_setup(h, d, n, H, W, heat_out, paf_out, paf_dtype, false, a, &done);
    if (rc || done) return rc;
    DeviceGuard guard(h->device);
    return postnet_launch_items(h, a, d, 0, d->n_scales, n, H, W, static_cast<cudaStream_t>(stream));
}

int spg_postnet_rotated(spg_handle *h, const spg_postnet_desc *d, const double *angle_deg, int32_t n, int32_t H, int32_t W,
                        float *heat_out, void *paf_out, int32_t paf_dtype, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (!d || d->n_scales < 1 || !angle_deg) return fail(h, SPG_E_INVALID, "postnet descriptor incomplete or angle_deg is NULL");
    bool any_rotated = false;
    for (int t = 0; t < d->n_scales; t++) {
        if (!std::isfinite(angle_deg[t])) return fail(h, SPG_E_INVALID, "angle_deg[%d] is not finite", t);
        any_rotated = any_rotated || angle_deg[t] != 0.0;
    }
    if (!any_rotated) return spg_postnet(h, d, n, H, W, heat_out, paf_out, paf_dtype, stream);
    PostArgs a;
    bool done;
    int rc = postnet_setup(h, d, n, H, W, heat_out, paf_out, paf_dtype, true, a, &done);
    if (rc || done) return rc;
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // items in the order of the loop (scale-major, angle-minor): consecutive angle-0 items go to the existing kernels as
    // one group, each rotated item is one launch; the float64 sums carry over through memory
    for (int t = 0; t < d->n_scales;) {
        if (angle_deg[t] == 0.0) {
            int t1 = t;
            while (t1 < d->n_scales && angle_deg[t1] == 0.0) t1++;
            if ((rc = postnet_launch_items(h, a, d, t, t1, n, H, W, st))) return rc;
            t = t1;
        } else {
            if ((rc = postnet_launch_rotated(h, a, d, t, angle_deg[t], n, H, W, st))) return rc;
            t++;
        }
    }
    return SPG_OK;
}

// ---- pre-network stage -------------------------------------------------------------------------
namespace {

// cv2.resize(fx = fy = scale)'s dsize (saturate_cast<int>: rint, half to even, in float64) and padRightDownCorner's size
int prenet_size(spg_handle *h, int32_t height, int32_t width, double scale, int32_t max_downsample, int32_t *crop_h,
                int32_t *crop_w, int32_t *pad_h, int32_t *pad_w) {
    if (height < 1 || width < 1 || height > 32767 || width > 32767)
        return fail(h, SPG_E_INVALID, "image %dx%d outside [1, 32767]", height, width);
    if (!std::isfinite(scale) || scale <= 0) return fail(h, SPG_E_INVALID, "scale must be finite and > 0");
    if (max_downsample <= 0) return fail(h, SPG_E_INVALID, "max_downsample must be > 0");
    const double ch = std::nearbyint((double)height * scale), cw = std::nearbyint((double)width * scale);
    if (ch < 1 || cw < 1) return fail(h, SPG_E_INVALID, "scale %g resizes a %dx%d image to nothing", scale, height, width);
    const double ph = std::ceil(ch / max_downsample) * max_downsample, pw = std::ceil(cw / max_downsample) * max_downsample;
    if (ph > 32767 || pw > 32767)
        return fail(h, SPG_E_INVALID, "scale %g pads a %dx%d image to %.0fx%.0f, above 32767", scale, height, width, ph, pw);
    if (crop_h) *crop_h = (int32_t)ch;
    if (crop_w) *crop_w = (int32_t)cw;
    if (pad_h) *pad_h = (int32_t)ph;
    if (pad_w) *pad_w = (int32_t)pw;
    return SPG_OK;
}

}  // namespace

int spg_prenet_size(int32_t height, int32_t width, double scale, int32_t max_downsample, int32_t *crop_h, int32_t *crop_w,
                    int32_t *pad_h, int32_t *pad_w) {
    return prenet_size(nullptr, height, width, scale, max_downsample, crop_h, crop_w, pad_h, pad_w);
}

int spg_prenet(spg_handle *h, const unsigned char *image_dev, int64_t row_stride, int32_t height, int32_t width,
               int32_t channels, double scale, const double *angle_deg, int32_t n_angles, int32_t max_downsample,
               int32_t pad_value, float *out, int64_t item_stride, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (channels != 3) return fail(h, SPG_E_INVALID, "channels = %d: only 3-channel images are supported", channels);
    if (pad_value < 0 || pad_value > 255) return fail(h, SPG_E_INVALID, "pad_value %d outside [0, 255]", pad_value);
    int32_t H, W, Hp, Wp;
    int rc = prenet_size(h, height, width, scale, max_downsample, &H, &W, &Hp, &Wp);
    if (rc) return rc;
    if (!image_dev || !out) return fail(h, SPG_E_INVALID, "image_dev/out is NULL");
    if (row_stride < (int64_t)width * 3) return fail(h, SPG_E_INVALID, "row_stride %lld below width * 3", (long long)row_stride);
    if (n_angles < 1 || !angle_deg) return fail(h, SPG_E_INVALID, "at least one angle is needed");
    for (int k = 0; k < n_angles; k++)
        if (!std::isfinite(angle_deg[k])) return fail(h, SPG_E_INVALID, "angle_deg[%d] is not finite", k);
    const int64_t item = (int64_t)2 * Hp * Wp * 3;
    if (n_angles > 1 && item_stride < item) return fail(h, SPG_E_INVALID, "item_stride %lld below 2 * Hp * Wp * 3", (long long)item_stride);
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // the padded image: grown on demand, no other allocation is touched
    const size_t need = (size_t)Hp * Wp * 3;
    if (h->pre_img_bytes < need) {
        if (h->pre_img) cudaFree(h->pre_img);
        h->pre_img = nullptr; h->pre_img_bytes = 0;
        SPG_CUDA(h, cudaMalloc(&h->pre_img, need));
        h->pre_img_bytes = need;
    }
    PrenetResizeArgs r{};
    r.src = image_dev; r.src_row = row_stride; r.h = height; r.w = width; r.H = H; r.W = W; r.Hp = Hp; r.Wp = Wp;
    r.sx = 1.0 / scale; r.sy = r.sx; r.pad_value = pad_value; r.copy = H == height && W == width; r.dst = h->pre_img;
    // tile height: the tile's source rows, at most ceil((th - 1) / scale) + 5, fit the shared-memory rows
    r.tile_h = kPreMaxTH;
    while (r.tile_h > 1 && std::ceil((r.tile_h - 1) * r.sy) + 5 > kPreRows) r.tile_h /= 2;
    prenet_resize_kernel<<<dim3((unsigned)((Wp + kPreTW - 1) / kPreTW), (unsigned)((Hp + r.tile_h - 1) / r.tile_h)), kPreThreads, 0, st>>>(r);
    h->launches++;
    SPG_CUDA(h, cudaGetLastError());
    const dim3 grid((unsigned)((Wp + kPreThreads - 1) / kPreThreads), (unsigned)Hp);
    for (int k = 0; k < n_angles; k++) {
        PrenetEmitArgs e{};
        e.img = h->pre_img; e.Hp = Hp; e.Wp = Wp; e.out = out + (int64_t)k * item_stride;
        if (angle_deg[k] != 0.0) {
            rotation_inverse_map(angle_deg[k], Hp, Wp, e.m);  // rotate_matrix (evaluate.py:109), inverted as warpAffine does
            prenet_emit_kernel<true><<<grid, kPreThreads, 0, st>>>(e);
        } else {
            prenet_emit_kernel<false><<<grid, kPreThreads, 0, st>>>(e);
        }
        h->launches++;
        SPG_CUDA(h, cudaGetLastError());
    }
    return SPG_OK;
}

// ---- stages ------------------------------------------------------------------------------------
int spg_nms_peaks(spg_handle *h, const float *heat, int64_t image_stride, int64_t chan_stride, int32_t n, int32_t H, int32_t W,
                  const spg_params *p, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (!heat && n > 0) return fail(h, SPG_E_INVALID, "heat_dev is NULL");
    int rc;
    if ((rc = check_dims(h, n, H, W)) || (rc = check_params(h, p))) return rc;
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    SPG_CUDA(h, cudaMemsetAsync(h->ws.status, 0, sizeof(uint32_t) * (size_t)n, st));
    if ((rc = launch_nms(h, heat, image_stride, chan_stride, 0, n, H, W, p, st))) return rc;
    h->stage = 1;
    return SPG_OK;
}

int spg_limb_score(spg_handle *h, const void *paf, int32_t dtype, int64_t image_stride, int64_t chan_stride, int32_t n, int32_t H,
                   int32_t W, double extent, const spg_params *p, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (!paf && n > 0) return fail(h, SPG_E_INVALID, "paf_dev is NULL");
    if (dtype != SPG_F32 && dtype != SPG_F64 && dtype != SPG_F32_AS_F64) return fail(h, SPG_E_INVALID, "paf_dtype must be SPG_F32, SPG_F64 or SPG_F32_AS_F64");
    if (h->stage < 1) return fail(h, SPG_E_STATE, "spg_limb_score needs peaks (spg_nms_peaks or spg_upload_peaks) first");
    int rc;
    if ((rc = check_dims(h, n, H, W)) || (rc = check_params(h, p))) return rc;
    DeviceGuard guard(h->device);
    if ((rc = launch_score(h, paf, dtype, image_stride, chan_stride, 0, n, H, W, extent, p, static_cast<cudaStream_t>(stream)))) return rc;
    h->stage = std::max(h->stage, 2);
    return SPG_OK;
}

int spg_limb_match(spg_handle *h, int32_t n, const spg_params *p, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (h->stage < 2) return fail(h, SPG_E_STATE, "spg_limb_match needs spg_limb_score first");
    int rc;
    if (n < 0 || n > h->cfg.max_batch) return fail(h, SPG_E_INVALID, "n_images out of range");
    if ((rc = check_params(h, p))) return rc;
    DeviceGuard guard(h->device);
    if ((rc = launch_match(h, 0, n, static_cast<cudaStream_t>(stream)))) return rc;
    h->stage = std::max(h->stage, 3);
    return SPG_OK;
}

int spg_assemble(spg_handle *h, int32_t n, const spg_params *p, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (h->stage < 3) return fail(h, SPG_E_STATE, "spg_assemble needs connections (spg_limb_match or spg_upload_connections) first");
    int rc;
    if (n < 0 || n > h->cfg.max_batch) return fail(h, SPG_E_INVALID, "n_images out of range");
    if ((rc = check_params(h, p))) return rc;
    DeviceGuard guard(h->device);
    if ((rc = launch_assemble(h, 0, n, p, static_cast<cudaStream_t>(stream)))) return rc;
    h->stage = 4;
    return SPG_OK;
}

int spg_match_assemble(spg_handle *h, int32_t n, const spg_params *p, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (h->stage < 2) return fail(h, SPG_E_STATE, "spg_match_assemble needs spg_limb_score first");
    int rc;
    if (n < 0 || n > h->cfg.max_batch) return fail(h, SPG_E_INVALID, "n_images out of range");
    if ((rc = check_params(h, p))) return rc;
    DeviceGuard guard(h->device);
    if ((rc = launch_match_assemble(h, 0, n, p, static_cast<cudaStream_t>(stream)))) return rc;
    h->stage = 4;
    return SPG_OK;
}

int spg_group_batch(spg_handle *h, const float *heat, int64_t his, int64_t hcs, const void *paf, int32_t dtype, int64_t pis, int64_t pcs,
                    int32_t n, int32_t H, int32_t W, double extent, const spg_params *p, void *stream) {
    if (!h) return SPG_E_INVALID;
    if ((!heat || !paf) && n > 0) return fail(h, SPG_E_INVALID, "heat_dev/paf_dev is NULL");
    if (dtype != SPG_F32 && dtype != SPG_F64 && dtype != SPG_F32_AS_F64) return fail(h, SPG_E_INVALID, "paf_dtype must be SPG_F32, SPG_F64 or SPG_F32_AS_F64");
    int rc;
    if ((rc = check_dims(h, n, H, W)) || (rc = check_params(h, p))) return rc;
    DeviceGuard guard(h->device);
    if ((rc = run_all(h, heat, his, hcs, paf, dtype, pis, pcs, 0, n, H, W, extent, p, static_cast<cudaStream_t>(stream)))) return rc;
    h->stage = 4;
    return SPG_OK;
}

int spg_host_alloc(void **ptr, uint64_t bytes) {
    if (!ptr) return SPG_E_INVALID;
    return cudaMallocHost(ptr, bytes) == cudaSuccess ? SPG_OK : SPG_E_CUDA;
}
int spg_host_free(void *ptr) { return cudaFreeHost(ptr) == cudaSuccess ? SPG_OK : SPG_E_CUDA; }

int spg_group_host(spg_handle *h, const float *heat_host, const void *paf_host, int32_t dtype, int32_t n, int32_t H, int32_t W,
                   double extent, const spg_params *p, int32_t *out_n, double *out_xy, double *out_score, uint32_t *out_status) {
    if (!h) return SPG_E_INVALID;
    if ((!heat_host || !paf_host) && n > 0) return fail(h, SPG_E_INVALID, "heat_host/paf_host is NULL");
    if (dtype != SPG_F32 && dtype != SPG_F64 && dtype != SPG_F32_AS_F64) return fail(h, SPG_E_INVALID, "paf_dtype must be SPG_F32, SPG_F64 or SPG_F32_AS_F64");
    int rc;
    if ((rc = check_dims(h, n, H, W)) || (rc = check_params(h, p))) return rc;
    DeviceGuard guard(h->device);
    const Workspace &ws = h->ws;
    const size_t plane = (size_t)H * W;
    const size_t esz = dtype == SPG_F64 ? 8 : 4;
    const size_t heat_img = (size_t)ws.K * plane * sizeof(float), paf_img = (size_t)ws.L * plane * esz;
    // chunk so that copy(c+1) overlaps kernels(c); keep at least ~8 chunks for large batches
    const int chunk = std::max(1, std::min(n, std::max(8, n / 8)));
    const size_t need_heat = 2 * (size_t)chunk * heat_img, need_paf = 2 * (size_t)chunk * paf_img;
    if (h->in_heat_bytes < need_heat) {
        if (h->in_heat) cudaFree(h->in_heat);
        h->in_heat = nullptr; h->in_heat_bytes = 0;
        SPG_CUDA(h, cudaMalloc(&h->in_heat, need_heat));
        h->in_heat_bytes = need_heat;
    }
    if (h->in_paf_bytes < need_paf) {
        if (h->in_paf) cudaFree(h->in_paf);
        h->in_paf = nullptr; h->in_paf_bytes = 0;
        SPG_CUDA(h, cudaMalloc(&h->in_paf, need_paf));
        h->in_paf_bytes = need_paf;
    }
    const size_t RSJ = (size_t)ws.capR * ws.J * 2;
    int ci = 0;
    for (int base = 0; base < n; base += chunk, ci++) {
        const int m = std::min(chunk, n - base);
        cudaStream_t st = h->streams[ci & 1];
        unsigned char *dh = static_cast<unsigned char *>(h->in_heat) + (size_t)(ci & 1) * chunk * heat_img;
        unsigned char *dp = static_cast<unsigned char *>(h->in_paf) + (size_t)(ci & 1) * chunk * paf_img;
        // stream order protects the staging buffers: chunk ci reuses the buffers of chunk ci-2 on the same stream
        SPG_CUDA(h, cudaMemcpyAsync(dh, reinterpret_cast<const unsigned char *>(heat_host) + (size_t)base * heat_img, (size_t)m * heat_img, cudaMemcpyHostToDevice, st));
        SPG_CUDA(h, cudaMemcpyAsync(dp, static_cast<const unsigned char *>(paf_host) + (size_t)base * paf_img, (size_t)m * paf_img, cudaMemcpyHostToDevice, st));
        if ((rc = run_all(h, reinterpret_cast<const float *>(dh), (int64_t)ws.K * plane, (int64_t)plane, dp, dtype, (int64_t)ws.L * plane,
                          (int64_t)plane, base, m, H, W, extent, p, st)))
            return rc;
        if (out_n) SPG_CUDA(h, cudaMemcpyAsync(out_n + base, ws.n_persons + base, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, st));
        if (out_xy && ws.J) SPG_CUDA(h, cudaMemcpyAsync(out_xy + (size_t)base * RSJ, ws.people_xy + (size_t)base * RSJ, sizeof(double) * RSJ * m, cudaMemcpyDeviceToHost, st));
        if (out_score) SPG_CUDA(h, cudaMemcpyAsync(out_score + (size_t)base * ws.capR, ws.people_score + (size_t)base * ws.capR, sizeof(double) * ws.capR * m, cudaMemcpyDeviceToHost, st));
        if (out_status) SPG_CUDA(h, cudaMemcpyAsync(out_status + base, ws.status + base, sizeof(uint32_t) * m, cudaMemcpyDeviceToHost, st));
    }
    SPG_CUDA(h, cudaStreamSynchronize(h->streams[0]));
    SPG_CUDA(h, cudaStreamSynchronize(h->streams[1]));
    h->stage = 4;
    return SPG_OK;
}

// ---- state transfer ------------------------------------------------------------------------------
int spg_upload_peaks(spg_handle *h, int32_t img, const int32_t *part_count, const double *x, const double *y, const float *score, void *stream) {
    if (!h || !part_count) return SPG_E_INVALID;
    if (img < 0 || img >= h->cfg.max_batch) return fail(h, SPG_E_INVALID, "image_index out of range");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Workspace &ws = h->ws;
    // the image's dense [K][capP] tables are laid out on the host and go up in three copies + the counters
    const size_t KP = (size_t)ws.K * ws.capP;
    std::vector<double> dx(KP, 0.0), dy(KP, 0.0);
    std::vector<float> ds(KP, 0.0f);
    size_t off = 0;
    for (int c = 0; c < ws.K; c++) {
        const int m = part_count[c];
        if (m < 0 || m > ws.capP) return fail(h, SPG_E_INVALID, "part %d has %d peaks; capacity is %d", c, m, ws.capP);
        if (m && (!x || !y || !score)) return fail(h, SPG_E_INVALID, "peak arrays are NULL");
        for (int q = 0; q < m; q++) {
            dx[(size_t)c * ws.capP + q] = x[off + q];
            dy[(size_t)c * ws.capP + q] = y[off + q];
            ds[(size_t)c * ws.capP + q] = score[off + q];
        }
        off += m;
    }
    const size_t dst = (size_t)img * KP;
    SPG_CUDA(h, cudaMemcpyAsync(ws.peak_x + dst, dx.data(), sizeof(double) * KP, cudaMemcpyHostToDevice, st));
    SPG_CUDA(h, cudaMemcpyAsync(ws.peak_y + dst, dy.data(), sizeof(double) * KP, cudaMemcpyHostToDevice, st));
    SPG_CUDA(h, cudaMemcpyAsync(ws.peak_score + dst, ds.data(), sizeof(float) * KP, cudaMemcpyHostToDevice, st));
    SPG_CUDA(h, cudaMemcpyAsync(ws.peak_count + (size_t)img * ws.K, part_count, sizeof(int32_t) * ws.K, cudaMemcpyHostToDevice, st));
    SPG_CUDA(h, cudaMemsetAsync(ws.status + img, 0, sizeof(uint32_t), st));
    SPG_CUDA(h, cudaStreamSynchronize(st));  // the host arrays are temporaries: one synchronisation per image
    h->stage = std::max(h->stage, 1);
    return SPG_OK;
}

int spg_upload_connections(spg_handle *h, int32_t img, const int32_t *conn_count, const int32_t *ij, const double *score, const double *norm, void *stream) {
    if (!h || !conn_count) return SPG_E_INVALID;
    if (img < 0 || img >= h->cfg.max_batch) return fail(h, SPG_E_INVALID, "image_index out of range");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Workspace &ws = h->ws;
    // dense [L][capP] tables built on the host: three copies + the counters and ONE synchronisation per image
    // (round 1 synchronised once per limb -- up to 30 host round trips per image)
    const size_t LP = (size_t)ws.L * ws.capP;
    std::vector<uint32_t> dij(LP, 0u);
    std::vector<double> dsc(LP, 0.0), dnm(LP, 0.0);
    size_t off = 0;
    for (int k = 0; k < ws.L; k++) {
        const int m = conn_count[k];
        if (m > ws.capP) return fail(h, SPG_E_INVALID, "limb %d has %d connections; capacity is %d", k, m, ws.capP);
        if (m <= 0) continue;
        if (!ij || !score || !norm) return fail(h, SPG_E_INVALID, "connection arrays are NULL");
        for (int r = 0; r < m; r++) {
            const int32_t i = ij[(off + r) * 2], j = ij[(off + r) * 2 + 1];
            if (i < 0 || j < 0 || i >= ws.capP || j >= ws.capP) return fail(h, SPG_E_INVALID, "connection index out of range");
            dij[(size_t)k * ws.capP + r] = ((uint32_t)i << 16) | (uint32_t)j;
            dsc[(size_t)k * ws.capP + r] = score[off + r];
            dnm[(size_t)k * ws.capP + r] = norm[off + r];
        }
        off += m;
    }
    const size_t dst = (size_t)img * LP;
    SPG_CUDA(h, cudaMemcpyAsync(ws.conn_ij + dst, dij.data(), sizeof(uint32_t) * LP, cudaMemcpyHostToDevice, st));
    SPG_CUDA(h, cudaMemcpyAsync(ws.conn_score + dst, dsc.data(), sizeof(double) * LP, cudaMemcpyHostToDevice, st));
    SPG_CUDA(h, cudaMemcpyAsync(ws.conn_norm + dst, dnm.data(), sizeof(double) * LP, cudaMemcpyHostToDevice, st));
    SPG_CUDA(h, cudaMemcpyAsync(ws.conn_count + (size_t)img * ws.L, conn_count, sizeof(int32_t) * ws.L, cudaMemcpyHostToDevice, st));
    SPG_CUDA(h, cudaStreamSynchronize(st));
    h->stage = std::max(h->stage, 3);
    return SPG_OK;
}

#define SPG_D2H(dst, src, count)                                                                                          \
    do {                                                                                                                  \
        if (dst) SPG_CUDA(h, cudaMemcpyAsync((dst), (src), sizeof(*(dst)) * (size_t)(count), cudaMemcpyDeviceToHost, st)); \
    } while (0)

int spg_download_peaks(spg_handle *h, int32_t n, int32_t *peak_count, double *x, double *y, float *score, uint32_t *anchor, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (n < 0 || n > h->cfg.max_batch) return fail(h, SPG_E_INVALID, "n_images out of range");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Workspace &ws = h->ws;
    const size_t m = (size_t)n * ws.K * ws.capP;
    SPG_D2H(peak_count, ws.peak_count, (size_t)n * ws.K);
    SPG_D2H(x, ws.peak_x, m);
    SPG_D2H(y, ws.peak_y, m);
    SPG_D2H(score, ws.peak_score, m);
    SPG_D2H(anchor, ws.peak_anchor, m);
    SPG_CUDA(h, cudaStreamSynchronize(st));
    return SPG_OK;
}

int spg_download_connections(spg_handle *h, int32_t n, int32_t *conn_count, int32_t *cand_count, uint32_t *ij, double *score, double *norm, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (n < 0 || n > h->cfg.max_batch) return fail(h, SPG_E_INVALID, "n_images out of range");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Workspace &ws = h->ws;
    const size_t m = (size_t)n * ws.L * ws.capP;
    SPG_D2H(conn_count, ws.conn_count, (size_t)n * ws.L);
    SPG_D2H(cand_count, ws.cand_count, (size_t)n * ws.L);
    SPG_D2H(ij, ws.conn_ij, m);
    SPG_D2H(score, ws.conn_score, m);
    SPG_D2H(norm, ws.conn_norm, m);
    SPG_CUDA(h, cudaStreamSynchronize(st));
    return SPG_OK;
}

int spg_download_people(spg_handle *h, int32_t n, int32_t *n_persons, double *subset, double *people_xy, double *people_score, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (n < 0 || n > h->cfg.max_batch) return fail(h, SPG_E_INVALID, "n_images out of range");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Workspace &ws = h->ws;
    SPG_D2H(n_persons, ws.n_persons, (size_t)n);
    SPG_D2H(subset, ws.subset, (size_t)n * ws.capR * (ws.K + 2) * 2);
    SPG_D2H(people_xy, ws.people_xy, (size_t)n * ws.capR * ws.J * 2);
    SPG_D2H(people_score, ws.people_score, (size_t)n * ws.capR);
    SPG_CUDA(h, cudaStreamSynchronize(st));
    return SPG_OK;
}

int spg_download_status(spg_handle *h, int32_t n, uint32_t *status, void *stream) {
    if (!h) return SPG_E_INVALID;
    if (n < 0 || n > h->cfg.max_batch) return fail(h, SPG_E_INVALID, "n_images out of range");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    SPG_D2H(status, h->ws.status, (size_t)n);
    SPG_CUDA(h, cudaStreamSynchronize(st));
    return SPG_OK;
}

}  // extern "C"
