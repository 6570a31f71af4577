// ccm_capi.cu -- implementation of include/blf_ccm.h: argument checking, kernel dispatch,
// persistent-grid sizing, the pipelined host-buffer entry point and the optional NCCL exchange.
// No CPU evaluation path exists in this library.
#include "../../include/blf_ccm.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvtx3/nvToolsExt.h>   // header-only: ranges cost a pointer test unless a profiler is attached

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <type_traits>

#include "ccm_kernels.cuh"
#include "dyn_kernels.h"
#include "host_expand.h"
#include "rls_kernels.cuh"
#include "sys_kernels.cuh"

using namespace blfccm;

// ------------------------------------------------------------------------------------------------
// error handling
// ------------------------------------------------------------------------------------------------

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                    \
    do {                                                                                  \
        cudaError_t e_ = (expr);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(BLF_CCM_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                              \
    } while (0)

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------

static constexpr int kHostSlots = 4;
static constexpr int kHostCopyStreams = 5;   // host evaluation: up to 3 upload + 2 download streams
static constexpr int kHostThreadsAuto = 4;   // expansion workers when not set (measured best: profiles/r02_host_sweep.log)
static constexpr int kHostUpStreamsAuto = 1;
static constexpr int kStageSlots = 8;    // pinned staging chunks of the compact control-matrix download
static constexpr int kMaxPartials = 8192;

struct KernelInfo {
    int blocks_per_sm = 0;
};

struct TensorMapEntry {
    const double* ptr = nullptr;
    int horizon = 0;
    long long chains = 0;
    CUtensorMap map;
};

// one blf_ccm_device_alloc_compressible allocation: a reserved virtual range with one physical
// compressible allocation mapped onto it
struct VmmRange {
    size_t size = 0;
    CUmemGenericAllocationHandle mem = 0;
};

struct blf_ccm_handle {
    unsigned magic = 0xB1FCC3A1u;
    int device = -1;
    int sm_count = 0;
    size_t mem_pitch = 0;      // cudaDeviceProp::memPitch: upper bound of a 2-D copy's pitches
    bool have_params = false;
    double length = 0, width = 0, spring = 0, damper = 0;
    Prm uni{};
    int last_path = BLF_CCM_PATH_NONE;
    long long launches = 0;
    std::map<const void*, KernelInfo> kinfo;
    // rollout scratch (block_best, counter, partials): ONE set per handle.  Calls that use it on
    // different streams are ordered by the library (scratch_acquire), they never overlap.
    CostIdx* block_best = nullptr;   // kMaxPartials pairs
    unsigned int* counter = nullptr;
    double* partials = nullptr;      // [n_rollouts][slots] per-(rollout, tile) cost partial sums
    size_t partials_bytes = 0;
    std::vector<TensorMapEntry> tmaps;   // cached TMA descriptors of rollout twist planes
    unsigned tmap_next = 0;
    double* gen_work = nullptr;      // scratch of the general-size RLS kernel
    size_t gen_bytes = 0;
    cudaEvent_t scratch_ev = nullptr;
    cudaStream_t scratch_stream = nullptr;   // stream of the last launch that used the scratch
    bool scratch_busy = false;
    // host pipeline
    cudaStream_t hstream[kHostSlots] = {};
    cudaEvent_t hev_up[kHostSlots] = {}, hev_done[kHostSlots] = {};   // time-chunked host rollouts
    cudaEvent_t hev_down[kHostSlots] = {};                            // host evaluation: slot downloaded
    double* single_out = nullptr;   // 64 doubles of mapped pinned host memory (n = 1 fast path): results + flag
    unsigned long long single_seq = 0;
    // compact control-matrix download of the host evaluation: pinned staging ring + expansion pool
    cudaStream_t hxstream[kHostCopyStreams] = {};   // [0..2] uploads, [3..4] downloads of the host evaluation
    cudaEvent_t hev_stage[kStageSlots] = {};
    double* hstage = nullptr;       // kStageSlots * hstage_chunk * 8 doubles, pinned
    long long hstage_chunk = 0;
    int host_threads = -1;          // -1 automatic, 0 = dense download (no host expansion)
    HostPool* pool = nullptr;
    double* hbuf[kHostSlots] = {};
    long long hchunk = 0;      // contacts per chunk the slots are sized for
    size_t hbytes = 0;
    long long host_chunk_pref = 131072;   // measured: profiles/r02_host_sweep.log
    // tuning overrides (environment, read once at create; 0 = automatic)
    int tune_cpt = 0;            // BLF_CCM_TUNE_CPT=2: use the 128-bit two-contacts-per-lane SoA kernel
    int tune_blocks_per_sm = 0;  // BLF_CCM_TUNE_BLOCKS_PER_SM>0: persistent grid with that many CTAs/SM
                                 // (looping kernels only); default = one tile per warp
    int tune_rollout_split = 0;  // BLF_CCM_TUNE_ROLLOUT_SPLIT>0: warps per tile of the fused rollout
    int tune_rollout_ws = 0;     // BLF_CCM_TUNE_ROLLOUT_WS: 1 force / 2 forbid the warp-specialised rollout
    int tune_no_pack = 0;        // BLF_CCM_TUNE_NO_PACK=1: J^T wrench for narrow Jacobians with the column-per-lane kernel
    int tune_no_rows = 0;        // BLF_CCM_TUNE_NO_ROWS=1: J^T wrench without base/out row staging
    int tune_gf_stages = 0;      // BLF_CCM_TUNE_GF_STAGES=4: lane-packed J^T wrench with the four-stage ring (default two: twice the warps per SM)
    int tune_no_pdl = 0;         // BLF_CCM_TUNE_NO_PDL=1: plain launches (no programmatic dependent launch)
    int tune_rollout_chunk_mb = 0;  // BLF_CCM_TUNE_ROLLOUT_CHUNK_MB: twist bytes per time chunk of the host rollout (default 8)
    int tune_host_up = 0, tune_host_down = 0;   // BLF_CCM_TUNE_HOST_UP / _DOWN: copy streams per direction of the host evaluation
    int tune_host_ramp = 1;      // BLF_CCM_TUNE_HOST_RAMP=0: equal chunks instead of the ramped schedule
    int tune_host_noexpand = 0;  // BLF_CCM_TUNE_HOST_NOEXPAND=1: measurement aid, the workers skip the expansion (results WRONG)
    int tune_llt_general = 0;    // BLF_CCM_TUNE_LLT_GENERAL=1: mass-matrix solve with the block-level kernel whatever the size
    int tune_fbd_tile_kb = 0;    // BLF_CCM_TUNE_FBD_TILE_KB: shared-memory target per CTA of the floating-base Euler step (default 24)
    int tune_fbd_no_bulk = 0;    // BLF_CCM_TUNE_FBD_NO_BULK=1: floating-base Euler step with per-thread copies even when 16-byte aligned
    int tune_rls_pipe = 0;       // BLF_CCM_TUNE_RLS_PIPE=1: the plain one-estimator-per-thread RLS kernel instead of the pipelined one
    // peer-memory arg-min exchange
    int p2p_nranks = 0, p2p_rank = -1;
    bool p2p_connected = false;
    P2pSlot* p2p_local = nullptr;             // this rank's mailbox [2][nranks]
    P2pSlot* p2p_peer[kP2pMaxRanks] = {};     // every rank's mailbox as mapped here
    unsigned long long p2p_epoch = 0;
    CostIdx* p2p_fused_out = nullptr;         // non-NULL: rollout reductions also run the exchange
    // compressible allocations by base address; every other device pointer is cudaMalloc memory.
    // Locked: owners may free from another thread (e.g. a garbage collector).
    std::map<uintptr_t, VmmRange> vmm;
    std::mutex vmm_mutex;
};

static int env_int(const char* name)
{
    const char* v = getenv(name);
    return v ? atoi(v) : 0;
}

static bool valid(const blf_ccm_handle* h) { return h && h->magic == 0xB1FCC3A1u; }

// Makes the handle's device current for the duration of one API call and restores the caller's
// device afterwards: a multi-GPU host process (torch with another current device) must not find its
// thread switched to another GPU behind its back.
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int dev)
    {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) {
            err = cudaSetDevice(dev);
            switched = (err == cudaSuccess);
        }
    }
    ~DeviceGuard()
    {
        if (switched) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// One NVTX range per C-ABI call, named after the entry point (nsys / ncu --nvtx show the host side
// of every call: argument checks, launches, and for the _host entry points the whole pipeline).
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

#define CHECK_HANDLE(h)                                                        \
    if (!valid(h)) return fail(BLF_CCM_ERR_INVALID_HANDLE, "invalid handle"); \
    NvtxRange nvtx_range_(__func__);                                           \
    DeviceGuard dev_guard_((h)->device);                                       \
    if (dev_guard_.err != cudaSuccess)                                         \
    return fail(BLF_CCM_ERR_CUDA, "cudaSetDevice(%d): %s", (h)->device, cudaGetErrorString(dev_guard_.err))

// The rollout scratch is one set per handle.  A call that uses it on another stream than the last
// user first orders itself after everything that user has submitted (an event recorded on the old
// stream now covers its earlier launches), so two rollout calls on different streams are serialised
// instead of corrupting each other's partial sums or the last-block counter.  The single-stream
// path pays nothing.
static int scratch_acquire(blf_ccm_handle* h, cudaStream_t st);
static int scratch_quiesce(blf_ccm_handle* h);
static void vmm_release_all(blf_ccm_handle* h);

extern "C" const char* blf_ccm_version(void) { return "blf_ccm 0.1.0 (sm_100a)"; }
extern "C" const char* blf_ccm_last_error(void) { return g_err; }

extern "C" int blf_ccm_destroy(blf_ccm_handle* h);

extern "C" int blf_ccm_create(int device, blf_ccm_handle** out)
{
    if (!out) return fail(BLF_CCM_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0) {
        cudaGetLastError();
        return fail(BLF_CCM_ERR_NO_DEVICE,
                    "no CUDA device available (%s); this backend has no CPU path",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= count)
        return fail(BLF_CCM_ERR_INVALID_ARG, "device %d out of range [0,%d)", device, count);
    DeviceGuard dev_guard_(device);
    if (dev_guard_.err != cudaSuccess)
        return fail(BLF_CCM_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(dev_guard_.err));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(BLF_CCM_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a",
                    device, prop.major, prop.minor);
    blf_ccm_handle* h = new (std::nothrow) blf_ccm_handle();
    if (!h) return fail(BLF_CCM_ERR_INVALID_ARG, "out of host memory");
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    h->mem_pitch = prop.memPitch;
    h->tune_cpt = env_int("BLF_CCM_TUNE_CPT");
    h->tune_fbd_tile_kb = env_int("BLF_CCM_TUNE_FBD_TILE_KB");
    h->tune_fbd_no_bulk = env_int("BLF_CCM_TUNE_FBD_NO_BULK");
    h->tune_blocks_per_sm = env_int("BLF_CCM_TUNE_BLOCKS_PER_SM");
    h->tune_rollout_split = env_int("BLF_CCM_TUNE_ROLLOUT_SPLIT");
    h->tune_no_pdl = env_int("BLF_CCM_TUNE_NO_PDL");
    h->tune_host_noexpand = env_int("BLF_CCM_TUNE_HOST_NOEXPAND");
    h->tune_host_up = env_int("BLF_CCM_TUNE_HOST_UP");
    h->tune_host_down = env_int("BLF_CCM_TUNE_HOST_DOWN");
    if (const char* v = getenv("BLF_CCM_TUNE_HOST_RAMP")) h->tune_host_ramp = atoi(v);
    h->tune_rls_pipe = env_int("BLF_CCM_TUNE_RLS_PIPE");
    h->tune_llt_general = env_int("BLF_CCM_TUNE_LLT_GENERAL");
    h->tune_rollout_chunk_mb = env_int("BLF_CCM_TUNE_ROLLOUT_CHUNK_MB");
    h->tune_no_rows = env_int("BLF_CCM_TUNE_NO_ROWS");
    h->tune_gf_stages = env_int("BLF_CCM_TUNE_GF_STAGES");
    h->tune_no_pack = env_int("BLF_CCM_TUNE_NO_PACK");
    h->tune_rollout_ws = env_int("BLF_CCM_TUNE_ROLLOUT_WS");
    if (const char* v = getenv("BLF_CCM_HOST_THREADS")) h->host_threads = atoi(v);
    cudaError_t ce = cudaMalloc(&h->block_best, sizeof(CostIdx) * kMaxPartials);
    if (ce == cudaSuccess) ce = cudaMalloc(&h->counter, sizeof(unsigned int));
    if (ce == cudaSuccess) ce = cudaMemset(h->counter, 0, sizeof(unsigned int));
    if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&h->scratch_ev, cudaEventDisableTiming);
    if (ce != cudaSuccess) {   // nothing leaks on a failed create
        cudaGetLastError();
        blf_ccm_destroy(h);
        return fail(BLF_CCM_ERR_CUDA, "blf_ccm_create: %s", cudaGetErrorString(ce));
    }
    *out = h;
    return BLF_CCM_OK;
}

static int scratch_acquire(blf_ccm_handle* h, cudaStream_t st)
{
    if (h->scratch_busy && h->scratch_stream != st) {
        cudaError_t e = cudaEventRecord(h->scratch_ev, h->scratch_stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(st, h->scratch_ev, 0);
        if (e != cudaSuccess) {   // e.g. the old stream was destroyed by its owner
            cudaGetLastError();
            CUDA_TRY(cudaDeviceSynchronize());
        }
    }
    h->scratch_stream = st;
    h->scratch_busy = true;
    return BLF_CCM_OK;
}

// before the scratch is freed / reallocated: nothing submitted earlier may still touch it
static int scratch_quiesce(blf_ccm_handle* h)
{
    if (!h->scratch_busy) return BLF_CCM_OK;
    if (cudaStreamSynchronize(h->scratch_stream) != cudaSuccess) {
        cudaGetLastError();
        CUDA_TRY(cudaDeviceSynchronize());
    }
    h->scratch_busy = false;
    return BLF_CCM_OK;
}

static void p2p_release(blf_ccm_handle* h)
{
    for (int r = 0; r < h->p2p_nranks; ++r)
        if (h->p2p_peer[r] && r != h->p2p_rank) cudaIpcCloseMemHandle(h->p2p_peer[r]);
    if (h->p2p_local) cudaFree(h->p2p_local);
    h->p2p_local = nullptr;
    for (auto& p : h->p2p_peer) p = nullptr;
    h->p2p_nranks = 0;
    h->p2p_rank = -1;
    h->p2p_connected = false;
    h->p2p_epoch = 0;
    h->p2p_fused_out = nullptr;
}

extern "C" int blf_ccm_destroy(blf_ccm_handle* h)
{
    if (!valid(h)) return fail(BLF_CCM_ERR_INVALID_HANDLE, "invalid handle");
    DeviceGuard dev_guard_(h->device);
    delete h->pool;
    h->pool = nullptr;
    for (int s = 0; s < kStageSlots; ++s)
        if (h->hev_stage[s]) cudaEventDestroy(h->hev_stage[s]);
    for (int s = 0; s < kHostCopyStreams; ++s)
        if (h->hxstream[s]) cudaStreamDestroy(h->hxstream[s]);
    if (h->hstage) cudaFreeHost(h->hstage);
    if (h->scratch_ev) cudaEventDestroy(h->scratch_ev);
    for (int s = 0; s < kHostSlots; ++s) {
        if (h->hstream[s]) cudaStreamDestroy(h->hstream[s]);
        if (h->hbuf[s]) cudaFree(h->hbuf[s]);
        if (h->hev_up[s]) cudaEventDestroy(h->hev_up[s]);
        if (h->hev_done[s]) cudaEventDestroy(h->hev_done[s]);
        if (h->hev_down[s]) cudaEventDestroy(h->hev_down[s]);
    }
    p2p_release(h);
    vmm_release_all(h);
    if (h->single_out) cudaFreeHost(h->single_out);
    if (h->block_best) cudaFree(h->block_best);
    if (h->counter) cudaFree(h->counter);
    if (h->partials) cudaFree(h->partials);
    if (h->gen_work) cudaFree(h->gen_work);
    h->magic = 0;
    delete h;
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_set_uniform_params(blf_ccm_handle* h, double length, double width,
                                          double spring_coeff, double damper_coeff)
{
    if (!valid(h)) return fail(BLF_CCM_ERR_INVALID_HANDLE, "invalid handle");
    h->length = length;
    h->width = width;
    h->spring = spring_coeff;
    h->damper = damper_coeff;
    h->uni = make_prm(length, width, spring_coeff, damper_coeff);
    h->have_params = true;
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_last_path(const blf_ccm_handle* h) { return valid(h) ? h->last_path : BLF_CCM_PATH_NONE; }
extern "C" int64_t blf_ccm_launch_count(const blf_ccm_handle* h) { return valid(h) ? h->launches : -1; }
extern "C" int blf_ccm_device(const blf_ccm_handle* h) { return valid(h) ? h->device : -1; }
extern "C" int blf_ccm_sm_count(const blf_ccm_handle* h) { return valid(h) ? h->sm_count : -1; }

// ------------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------------

template <typename K>
static int persistent_blocks(blf_ccm_handle* h, K kernel, int threads, size_t smem, int* out)
{
    const void* key = reinterpret_cast<const void*>(kernel);
    auto it = h->kinfo.find(key);
    if (it == h->kinfo.end()) {
        if (smem > 48 * 1024)
            CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          static_cast<int>(smem)));
        KernelInfo ki;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ki.blocks_per_sm, kernel, threads,
                                                               smem));
        if (ki.blocks_per_sm < 1)
            return fail(BLF_CCM_ERR_CUDA, "kernel does not fit on an SM (threads %d, smem %zu)",
                        threads, smem);
        it = h->kinfo.emplace(key, ki).first;
    }
    int per_sm = it->second.blocks_per_sm;
    if (h->tune_blocks_per_sm > 0) per_sm = std::min(per_sm, h->tune_blocks_per_sm);
    *out = h->tune_blocks_per_sm > 0 ? per_sm * h->sm_count : 0x7fffffff;
    return BLF_CCM_OK;
}

// Launch with programmatic stream serialization (PDL): see ccm_soa_kernel.  BLF_CCM_TUNE_NO_PDL=1
// falls back to a plain launch (for A/B measurements).
template <typename K, typename A>
static cudaError_t launch_pdl(const blf_ccm_handle* h, K kernel, long long grid, int threads,
                              size_t smem, cudaStream_t st, const A& args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(static_cast<unsigned>(threads));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = h->tune_no_pdl ? 0 : 1;
    return cudaLaunchKernelEx(&cfg, kernel, args);
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static bool aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

// compile-time dispatch over the 15 non-empty output masks
template <template <unsigned, bool> class F, bool HET, typename... Args>
static int dispatch_mask(unsigned mask, Args&&... args)
{
    switch (mask) {
#define BLFCCM_CASE(M) \
    case M:            \
        return F<M, HET>::run(std::forward<Args>(args)...);
        BLFCCM_CASE(1) BLFCCM_CASE(2) BLFCCM_CASE(3) BLFCCM_CASE(4) BLFCCM_CASE(5) BLFCCM_CASE(6)
        BLFCCM_CASE(7) BLFCCM_CASE(8) BLFCCM_CASE(9) BLFCCM_CASE(10) BLFCCM_CASE(11)
        BLFCCM_CASE(12) BLFCCM_CASE(13) BLFCCM_CASE(14) BLFCCM_CASE(15)
#undef BLFCCM_CASE
    default:
        return fail(BLF_CCM_ERR_INVALID_ARG, "out_mask %u has no valid output bit", mask);
    }
}

// ---- SoA -----------------------------------------------------------------------------------------

template <unsigned MASK, bool HET>
struct SoaLaunch {
    static int run(blf_ccm_handle* h, const SoaArgs& a, bool vec2, cudaStream_t st)
    {
        constexpr int threads = 128;
        if (vec2) {
            constexpr int TILE = 64;
            const size_t smem = (MASK & M_CTRL) ? size_t(threads / 32) * TILE * 288 : 0;
            auto k = ccm_soa_vec2_kernel<MASK, HET>;
            int cap = 0;
            if (int rc = persistent_blocks(h, k, threads, smem, &cap)) return rc;
            const long long tiles = (a.n + TILE - 1) / TILE;
            const long long want = (tiles + threads / 32 - 1) / (threads / 32);
            const int grid = static_cast<int>(std::min<long long>(want, cap));
            k<<<grid, threads, smem, st>>>(a);
        } else {
            const size_t smem = (MASK & M_CTRL) ? size_t(threads / 32) * 32 * 288 : 0;
            auto k = ccm_soa_kernel<MASK, HET, false>;
            int cap = 0;
            if (int rc = persistent_blocks(h, k, threads, smem, &cap)) return rc;  // smem attribute
            const long long grid = (a.n + threads - 1) / threads;
            if (grid > 0x7fffffffLL) return fail(BLF_CCM_ERR_INVALID_ARG, "n too large for one launch");
            CUDA_TRY(launch_pdl(h, k, grid, threads, smem, st, a));
        }
        CUDA_TRY(cudaGetLastError());
        h->launches++;
        return BLF_CCM_OK;
    }
};

static int fill_soa_args(blf_ccm_handle* h, long long n, const double* const* in_planes,
                         const double* const* param_planes, unsigned out_mask, unsigned compute_mask,
                         double* const* wrench_planes, double* const* autodyn_planes, double* ctrl,
                         double* const* regressor_planes, SoaArgs& a, bool& vec)
{
    if (n < 0) return fail(BLF_CCM_ERR_INVALID_ARG, "n < 0");
    if (!in_planes) return fail(BLF_CCM_ERR_INVALID_ARG, "in_planes is NULL");
    if (!param_planes && !h->have_params)
        return fail(BLF_CCM_ERR_NOT_INITIALIZED,
                    "no parameters: call blf_ccm_set_uniform_params or pass param_planes");
    memset(&a, 0, sizeof(a));
    a.n = n;
    a.uni = h->uni;
    vec = true;
    const unsigned live = live_planes(compute_mask);
    for (int i = 0; i < 30; ++i) {
        if (!(live & (1u << i))) continue;
        if (!in_planes[i]) return fail(BLF_CCM_ERR_INVALID_ARG, "in_planes[%d] is NULL but live for out_mask %u", i, out_mask);
        if (!aligned8(in_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "in_planes[%d] not 8-byte aligned", i);
        a.in[i] = in_planes[i];
        vec = vec && aligned16(in_planes[i]);
    }
    if (param_planes)
        for (int i = 0; i < 4; ++i) {
            if (!param_planes[i] || !aligned8(param_planes[i]))
                return fail(BLF_CCM_ERR_INVALID_ARG, "param_planes[%d] NULL or misaligned", i);
            a.prm[i] = param_planes[i];
            vec = vec && aligned16(param_planes[i]);
        }
    auto take = [&](double* const* src, double** dst, int cnt, const char* what) -> int {
        if (!src) return fail(BLF_CCM_ERR_INVALID_ARG, "%s is NULL but requested by out_mask", what);
        for (int i = 0; i < cnt; ++i) {
            if (!src[i] || !aligned8(src[i]))
                return fail(BLF_CCM_ERR_INVALID_ARG, "%s[%d] NULL or misaligned", what, i);
            dst[i] = src[i];
            vec = vec && aligned16(src[i]);
        }
        return BLF_CCM_OK;
    };
    if (out_mask & BLF_CCM_WRENCH)
        if (int rc = take(wrench_planes, a.wrench, 6, "wrench_planes")) return rc;
    if (out_mask & BLF_CCM_AUTODYN)
        if (int rc = take(autodyn_planes, a.autodyn, 6, "autodyn_planes")) return rc;
    if (out_mask & BLF_CCM_REGRESSOR)
        if (int rc = take(regressor_planes, a.reg, 12, "regressor_planes")) return rc;
    if (out_mask & BLF_CCM_CTRL) {
        if (!ctrl || !aligned8(ctrl)) return fail(BLF_CCM_ERR_INVALID_ARG, "ctrl NULL or misaligned");
        a.ctrl = ctrl;
        a.ctrl_bulk = aligned16(ctrl) ? 1 : 0;
        vec = vec && a.ctrl_bulk;
    }
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_eval_batch_soa(blf_ccm_handle* h, int64_t n, const double* const* in_planes,
                                      const double* const* param_planes, unsigned out_mask,
                                      double* const* wrench_planes, double* const* autodyn_planes,
                                      double* ctrl, double* const* regressor_planes, void* stream)
{
    CHECK_HANDLE(h);
    if (out_mask == 0 || out_mask > 15u) return fail(BLF_CCM_ERR_INVALID_ARG, "out_mask %u invalid", out_mask);
    if (n == 0) return BLF_CCM_OK;  // empty batch: nothing to read, nothing to write
    SoaArgs a;
    bool vec = false;
    if (int rc = fill_soa_args(h, n, in_planes, param_planes, out_mask, out_mask, wrench_planes,
                               autodyn_planes, ctrl, regressor_planes, a, vec))
        return rc;
    // planes only need 8-byte alignment; the dense 6x6 leaves by bulk copy when 16-byte aligned
    h->last_path = ((out_mask & BLF_CCM_CTRL) && !a.ctrl_bulk) ? BLF_CCM_PATH_DIRECT64 : BLF_CCM_PATH_BULK;
    const bool vec2 = vec && h->tune_cpt == 2;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (param_planes) return dispatch_mask<SoaLaunch, true>(out_mask, h, a, vec2, st);
    return dispatch_mask<SoaLaunch, false>(out_mask, h, a, vec2, st);
}

// ---- AoS -----------------------------------------------------------------------------------------

template <unsigned MASK, bool HET>
struct AosLaunch {
    static int run(blf_ccm_handle* h, const AosArgs& a, bool bulk, cudaStream_t st)
    {
        if (bulk) {
            constexpr int threads = 64;
            const size_t smem = size_t(threads / 32) * AosSmem<MASK, HET>::bytes;
            auto k = ccm_aos_kernel<MASK, HET>;
            int cap = 0;
            if (int rc = persistent_blocks(h, k, threads, smem, &cap)) return rc;
            const long long tiles = (a.n + 31) / 32;
            const long long want = (tiles + threads / 32 - 1) / (threads / 32);
            const int grid = static_cast<int>(std::min<long long>(want, cap));
            CUDA_TRY(launch_pdl(h, k, grid, threads, smem, st, a));
        } else {
            constexpr int threads = 128;
            auto k = ccm_aos_scalar_kernel<MASK, HET>;
            int cap = 0;
            if (int rc = persistent_blocks(h, k, threads, 0, &cap)) return rc;
            const long long want = (a.n + threads - 1) / threads;
            const int grid = static_cast<int>(std::min<long long>(want, cap));
            k<<<grid, threads, 0, st>>>(a);
        }
        CUDA_TRY(cudaGetLastError());
        h->launches++;
        return BLF_CCM_OK;
    }
};

static int launch_aos(blf_ccm_handle* h, long long n, const double* twists, const double* poses,
                      const double* null_poses, const blf_ccm_params* params, unsigned out_mask,
                      double* wrench, double* autodyn, double* ctrl, double* regressor,
                      cudaStream_t st, bool ctrl_compact = false)
{
    if (n < 0) return fail(BLF_CCM_ERR_INVALID_ARG, "n < 0");
    if (out_mask == 0 || out_mask > 15u) return fail(BLF_CCM_ERR_INVALID_ARG, "out_mask %u invalid", out_mask);
    if (n == 0) return BLF_CCM_OK;  // empty batch
    if (!params && !h->have_params)
        return fail(BLF_CCM_ERR_NOT_INITIALIZED,
                    "no parameters: call blf_ccm_set_uniform_params or pass params");
    const bool need_state = (out_mask & (BLF_CCM_WRENCH | BLF_CCM_AUTODYN | BLF_CCM_REGRESSOR)) != 0;
    bool bulk = true;
    auto chk = [&](const void* p, bool needed, const char* what) -> int {
        if (!needed) return BLF_CCM_OK;
        if (!p) return fail(BLF_CCM_ERR_INVALID_ARG, "%s is NULL but required by out_mask %u", what, out_mask);
        if (!aligned8(p)) return fail(BLF_CCM_ERR_INVALID_ARG, "%s not 8-byte aligned", what);
        bulk = bulk && aligned16(p);
        return BLF_CCM_OK;
    };
    if (int rc = chk(poses, true, "poses")) return rc;
    if (int rc = chk(twists, need_state, "twists")) return rc;
    if (int rc = chk(null_poses, need_state, "null_poses")) return rc;
    if (int rc = chk(params, params != nullptr, "params")) return rc;
    if (int rc = chk(wrench, out_mask & BLF_CCM_WRENCH, "wrench")) return rc;
    if (int rc = chk(autodyn, out_mask & BLF_CCM_AUTODYN, "autodyn")) return rc;
    if (int rc = chk(ctrl, out_mask & BLF_CCM_CTRL, "ctrl")) return rc;
    if (int rc = chk(regressor, out_mask & BLF_CCM_REGRESSOR, "regressor")) return rc;
    h->last_path = bulk ? BLF_CCM_PATH_BULK : BLF_CCM_PATH_DIRECT64;
    AosArgs a;
    memset(&a, 0, sizeof(a));
    a.twists = twists;
    a.poses = poses;
    a.nulls = null_poses;
    a.prm = reinterpret_cast<const double*>(params);
    a.wrench = wrench;
    a.autodyn = autodyn;
    a.ctrl = ctrl;
    a.reg = regressor;
    a.uni = h->uni;
    a.n = n;
    a.ctrl_compact = ctrl_compact ? 1 : 0;
    if (params) return dispatch_mask<AosLaunch, true>(out_mask, h, a, bulk, st);
    return dispatch_mask<AosLaunch, false>(out_mask, h, a, bulk, st);
}

extern "C" int blf_ccm_eval_batch_aos(blf_ccm_handle* h, int64_t n, const double* twists,
                                      const double* poses, const double* null_poses,
                                      const blf_ccm_params* params, unsigned out_mask,
                                      double* wrench, double* autodyn, double* ctrl,
                                      double* regressor, void* stream)
{
    CHECK_HANDLE(h);
    return launch_aos(h, n, twists, poses, null_poses, params, out_mask, wrench, autodyn, ctrl,
                      regressor, static_cast<cudaStream_t>(stream));
}

// ---- one contact state from host memory: the per-instance facade's getters -----------------------

template <unsigned MASK, bool HET>
struct SingleLaunch {
    static int run(blf_ccm_handle* h, const SingleArgs& a, cudaStream_t st)
    {
        ccm_single_kernel<MASK><<<1, 32, 0, st>>>(a);
        CUDA_TRY(cudaGetLastError());
        h->launches++;
        return BLF_CCM_OK;
    }
};

static int eval_single_host(blf_ccm_handle* h, const double* twist, const double* pose,
                            const double* null_pose, const blf_ccm_params* params, unsigned out_mask,
                            double* wrench, double* autodyn, double* ctrl, double* regressor)
{
    if (!h->single_out) {
        CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&h->single_out), 64 * sizeof(double), cudaHostAllocMapped));
        memset(h->single_out, 0, 64 * sizeof(double));
    }
    if (!h->hstream[0]) CUDA_TRY(cudaStreamCreateWithFlags(&h->hstream[0], cudaStreamNonBlocking));
    SingleArgs a;
    memset(&a, 0, sizeof(a));
    if (twist) memcpy(a.tw, twist, sizeof(a.tw));
    memcpy(a.pose, pose, sizeof(a.pose));
    if (null_pose) memcpy(a.null, null_pose, sizeof(a.null));
    a.prm = params ? make_prm(params->length, params->width, params->spring_coeff, params->damper_coeff)
                   : h->uni;
    a.out = h->single_out;   // unified addressing: the mapped host pointer is valid on the device
    a.seq = ++h->single_seq;
    cudaStream_t st = h->hstream[0];
    if (int rc = dispatch_mask<SingleLaunch, false>(out_mask, h, a, st)) return rc;
    // The kernel writes its results and then the sequence number into the mapped block; polling
    // that word costs less than a stream synchronisation (measured per getter: DESIGN.md section 1).
    // A launch that died never writes it: after a bounded spin the stream is asked instead.
    {
        const volatile unsigned long long* flag =
            reinterpret_cast<const volatile unsigned long long*>(h->single_out + 60);
        bool seen = false;
        for (int spin = 0; spin < 200000 && !seen; ++spin) {
            seen = (*flag == a.seq);
            if (!seen) _mm_pause();
        }
        if (seen) std::atomic_thread_fence(std::memory_order_acquire);
        else CUDA_TRY(cudaStreamSynchronize(st));
    }
    const double* o = h->single_out;
    if (out_mask & BLF_CCM_WRENCH) memcpy(wrench, o, 6 * sizeof(double));
    if (out_mask & BLF_CCM_AUTODYN) memcpy(autodyn, o + 6, 6 * sizeof(double));
    if (out_mask & BLF_CCM_REGRESSOR) memcpy(regressor, o + 12, 12 * sizeof(double));
    if (out_mask & BLF_CCM_CTRL) memcpy(ctrl, o + 24, 36 * sizeof(double));
    h->last_path = BLF_CCM_PATH_BULK;
    return BLF_CCM_OK;
}

// ---- host buffers: chunked, four slots; upload, kernel and download streams overlapped ---------------------------

extern "C" int blf_ccm_eval_batch_host(blf_ccm_handle* h, int64_t n, const double* twists,
                                       const double* poses, const double* null_poses,
                                       const blf_ccm_params* params, unsigned out_mask,
                                       double* wrench, double* autodyn, double* ctrl,
                                       double* regressor)
{
    CHECK_HANDLE(h);
    if (n < 0) return fail(BLF_CCM_ERR_INVALID_ARG, "n < 0");
    if (out_mask == 0 || out_mask > 15u) return fail(BLF_CCM_ERR_INVALID_ARG, "out_mask %u invalid", out_mask);
    if (n == 0) return BLF_CCM_OK;
    const bool need_state = (out_mask & (BLF_CCM_WRENCH | BLF_CCM_AUTODYN | BLF_CCM_REGRESSOR)) != 0;
    if (!poses || (need_state && (!twists || !null_poses)))
        return fail(BLF_CCM_ERR_INVALID_ARG, "an input array required by out_mask %u is NULL", out_mask);
    if (((out_mask & BLF_CCM_WRENCH) && !wrench) || ((out_mask & BLF_CCM_AUTODYN) && !autodyn) ||
        ((out_mask & BLF_CCM_CTRL) && !ctrl) || ((out_mask & BLF_CCM_REGRESSOR) && !regressor))
        return fail(BLF_CCM_ERR_INVALID_ARG, "an output array requested by out_mask %u is NULL", out_mask);
    if (!params && !h->have_params)
        return fail(BLF_CCM_ERR_NOT_INITIALIZED,
                    "no parameters: call blf_ccm_set_uniform_params or pass params");
    if (n == 1)   // the per-instance facade: one launch, results through mapped pinned memory
        return eval_single_host(h, twists, poses, null_poses, params, out_mask, wrench, autodyn, ctrl,
                                regressor);

    // ---- chunk schedule ---------------------------------------------------------------------------
    // Every chunk costs a fixed ~40 us of dead time on the PCIe engines (six copies, each started
    // and retired on its own: 173 M evals/s with 65 536-contact chunks, 188 M with 262 144,
    // profiles/r02_host_sweep.log), so chunks should be large; but the first chunk's upload and the
    // last chunk's download + expansion are not overlapped with anything, so the schedule ramps:
    // chunk/4, chunk/2, chunk ... chunk, chunk/2, chunk/4 (BLF_CCM_TUNE_HOST_RAMP=0: equal chunks).
    const long long chunk = std::max<long long>(2, (std::min<long long>(n, h->host_chunk_pref) + 1) & ~1LL);   // even
    std::vector<long long> offs, cnts;
    {
        const bool ramp = h->tune_host_ramp != 0 && n >= 4 * chunk;
        long long off = 0;
        auto push = [&](long long c) {
            c = std::min(c, n - off);
            if (c <= 0) return;
            offs.push_back(off);
            cnts.push_back(c);
            off += c;
        };
        if (ramp) {
            push(chunk / 4 & ~1LL);
            push(chunk / 2 & ~1LL);
            const long long tail = (chunk / 2 & ~1LL) + (chunk / 4 & ~1LL);
            while (n - off > tail + chunk) push(chunk);
            // what is left (between tail and tail + chunk contacts): one middle chunk, then the ramp down
            push(std::max<long long>(0, n - off - tail) & ~1LL);
            push(chunk / 2 & ~1LL);
            push(n - off);
        } else {
            while (off < n) push(chunk);
        }
    }
    const long long nchunks = static_cast<long long>(offs.size());

    // slot layout in doubles per contact (every section starts 16-byte aligned: all even counts)
    const size_t per_contact = 6 + 12 + 12 + 4 + 6 + 6 + 36 + 12;
    const size_t need = size_t(chunk) * per_contact * sizeof(double);
    if (h->hbytes < need) {
        for (int s = 0; s < kHostSlots; ++s) {
            if (h->hbuf[s]) CUDA_TRY(cudaFree(h->hbuf[s]));
            h->hbuf[s] = nullptr;
        }
        h->hbytes = 0;
        for (int s = 0; s < kHostSlots; ++s) CUDA_TRY(cudaMalloc(&h->hbuf[s], need));
        h->hbytes = need;
    }
    h->hchunk = chunk;
    for (int s = 0; s < kHostSlots; ++s) {
        if (!h->hstream[s]) CUDA_TRY(cudaStreamCreateWithFlags(&h->hstream[s], cudaStreamNonBlocking));
        if (!h->hev_up[s]) CUDA_TRY(cudaEventCreateWithFlags(&h->hev_up[s], cudaEventDisableTiming));
        if (!h->hev_done[s]) CUDA_TRY(cudaEventCreateWithFlags(&h->hev_done[s], cudaEventDisableTiming));
    }
    for (int s = 0; s < kHostCopyStreams; ++s)
        if (!h->hxstream[s]) CUDA_TRY(cudaStreamCreateWithFlags(&h->hxstream[s], cudaStreamNonBlocking));
    for (int s = 0; s < kStageSlots; ++s)
        if (!h->hev_stage[s]) CUDA_TRY(cudaEventCreateWithFlags(&h->hev_stage[s], cudaEventDisableTiming));

    // Control matrix: 24 of the 36 doubles are structural zeros and 5 more are duplicates.  With
    // host threads available the kernel writes the 7 distinct values (padded to 8 doubles) and only
    // those 64 bytes per contact cross PCIe -- 160 instead of 384 bytes per evaluation come back --
    // into a pinned staging ring; worker threads expand them into the caller's dense Matrix6x6
    // array (structural zeros +0.0, bit-identical to the dense kernel output) while later chunks
    // are in flight.  host_threads == 0 keeps the dense download (A/B: profiles/r02_host_sweep.log).
    int nthreads = h->host_threads;
    if (nthreads < 0) {
        int hw = static_cast<int>(std::thread::hardware_concurrency());
        if (const char* lws = getenv("LOCAL_WORLD_SIZE")) hw /= std::max(1, atoi(lws));  // one process per GPU
        nthreads = std::max(1, std::min(kHostThreadsAuto, hw / 2));
    }
    const bool compact = (out_mask & BLF_CCM_CTRL) && nthreads > 0;
    if (compact) {
        if (h->hstage_chunk < chunk) {
            if (h->hstage) CUDA_TRY(cudaFreeHost(h->hstage));
            h->hstage = nullptr;
            h->hstage_chunk = 0;
            CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&h->hstage),
                                   size_t(kStageSlots) * chunk * 8 * sizeof(double), cudaHostAllocDefault));
            h->hstage_chunk = chunk;
        }
        if (nchunks < 2) nthreads = 1;   // a single chunk: one worker is enough
        if (!h->pool) h->pool = new (std::nothrow) HostPool();
        if (!h->pool) return fail(BLF_CCM_ERR_INVALID_ARG, "out of host memory");
        h->pool->resize(nthreads);
    }

    // shared with the expansion workers
    std::atomic<long long> ready{0};                 // chunks whose download has completed
    std::atomic<long long> done[kStageSlots];        // cumulative worker completions per staging slot
    std::atomic<bool> abort{false};
    for (auto& d : done) d.store(0);
    if (compact) {
        double* stage = h->hstage;
        const long long schunk = h->hstage_chunk;
        const bool skip = h->tune_host_noexpand != 0;
        const long long* poffs = offs.data();
        const long long* pcnts = cnts.data();
        h->pool->start([=, &ready, &done, &abort](int j) {
            for (long long c = 0; c < nchunks; ++c) {
                int spins = 0;
                while (ready.load(std::memory_order_acquire) <= c) {
                    if (abort.load(std::memory_order_relaxed)) return;
                    if (++spins < 2000) _mm_pause();
                    else std::this_thread::yield();
                }
                const long long off = poffs[c], cnt = pcnts[c];
                // even slice boundaries (chunk offsets are even too): a contact PAIR is nine whole
                // 64-byte lines of the dense array, which the AVX-512 expansion stores line by line
                const long long lo = (cnt * j / nthreads) & ~1LL;
                const long long hi = j == nthreads - 1 ? cnt : ((cnt * (j + 1) / nthreads) & ~1LL);
                if (!skip)
                    expand_ctrl(stage + size_t(c % kStageSlots) * schunk * 8 + lo * 8, ctrl + (off + lo) * 36, hi - lo);
                done[c % kStageSlots].fetch_add(1, std::memory_order_release);
            }
        });
    }
    // on any error below the workers must be released before the atomics leave scope
    struct PoolJoin {
        HostPool* p;
        std::atomic<bool>& abort;
        bool failed = true;
        ~PoolJoin()
        {
            if (!p) return;
            if (failed) abort.store(true);
            p->wait();
        }
    } join{compact ? h->pool : nullptr, abort};

    // Streams: `nup` upload and `ndown` download streams (chunk k uses stream k mod the count) and
    // one for the kernels, chained by events; kHostSlots chunk buffers in flight on the device.  With
    // two upload streams the start-up and retirement of one copy overlap the transfer of the other.
    const int nup = std::max(1, std::min(3, h->tune_host_up > 0 ? h->tune_host_up : kHostUpStreamsAuto));
    const int ndown = std::max(1, std::min(2, h->tune_host_down > 0 ? h->tune_host_down : 1));
    cudaStream_t comp = h->hstream[1];
    const size_t D = sizeof(double);
    auto enqueue = [&](long long index) -> int {
        const long long off = offs[index], c = cnts[index];
        const int slot = static_cast<int>(index % kHostSlots), sslot = static_cast<int>(index % kStageSlots);
        cudaStream_t up = h->hxstream[index % nup], down = h->hxstream[3 + index % ndown];
        double* b = h->hbuf[slot];
        double* d_tw = b;
        double* d_po = d_tw + chunk * 6;
        double* d_nu = d_po + chunk * 12;
        double* d_pr = d_nu + chunk * 12;
        double* d_w = d_pr + chunk * 4;
        double* d_a = d_w + chunk * 6;
        double* d_c = d_a + chunk * 6;
        double* d_r = d_c + chunk * 36;
        // the device slot is free once the chunk that used it last (index - kHostSlots) is downloaded
        if (index >= kHostSlots)
            CUDA_TRY(cudaStreamWaitEvent(up, h->hev_stage[(index - kHostSlots) % kStageSlots], 0));
        if (need_state) {
            CUDA_TRY(cudaMemcpyAsync(d_tw, twists + off * 6, c * 6 * D, cudaMemcpyHostToDevice, up));
            CUDA_TRY(cudaMemcpyAsync(d_nu, null_poses + off * 12, c * 12 * D, cudaMemcpyHostToDevice, up));
        }
        CUDA_TRY(cudaMemcpyAsync(d_po, poses + off * 12, c * 12 * D, cudaMemcpyHostToDevice, up));
        if (params)
            CUDA_TRY(cudaMemcpyAsync(d_pr, params + off, c * 4 * D, cudaMemcpyHostToDevice, up));
        CUDA_TRY(cudaEventRecord(h->hev_up[slot], up));
        CUDA_TRY(cudaStreamWaitEvent(comp, h->hev_up[slot], 0));
        if (int rc = launch_aos(h, c, d_tw, d_po, d_nu,
                                params ? reinterpret_cast<const blf_ccm_params*>(d_pr) : nullptr,
                                out_mask, d_w, d_a, d_c, d_r, comp, compact))
            return rc;
        CUDA_TRY(cudaEventRecord(h->hev_done[slot], comp));
        CUDA_TRY(cudaStreamWaitEvent(down, h->hev_done[slot], 0));
        if (out_mask & BLF_CCM_WRENCH)
            CUDA_TRY(cudaMemcpyAsync(wrench + off * 6, d_w, c * 6 * D, cudaMemcpyDeviceToHost, down));
        if (out_mask & BLF_CCM_AUTODYN)
            CUDA_TRY(cudaMemcpyAsync(autodyn + off * 6, d_a, c * 6 * D, cudaMemcpyDeviceToHost, down));
        if (out_mask & BLF_CCM_CTRL) {
            if (compact)
                CUDA_TRY(cudaMemcpyAsync(h->hstage + size_t(sslot) * h->hstage_chunk * 8, d_c, c * 8 * D,
                                         cudaMemcpyDeviceToHost, down));
            else
                CUDA_TRY(cudaMemcpyAsync(ctrl + off * 36, d_c, c * 36 * D, cudaMemcpyDeviceToHost, down));
        }
        if (out_mask & BLF_CCM_REGRESSOR)
            CUDA_TRY(cudaMemcpyAsync(regressor + off * 12, d_r, c * 12 * D, cudaMemcpyDeviceToHost, down));
        CUDA_TRY(cudaEventRecord(h->hev_stage[sslot], down));
        return BLF_CCM_OK;
    };
    // staging slot of chunk k is free once every worker has expanded chunk k - kStageSlots
    auto stage_free = [&](long long k) {
        return !compact || k < kStageSlots ||
               done[k % kStageSlots].load(std::memory_order_acquire) >= (k / kStageSlots) * nthreads;
    };
    long long next_enq = 0, next_ready = 0;
    while (next_ready < nchunks) {
        while (next_enq < nchunks && next_enq < next_ready + kStageSlots && stage_free(next_enq))
            if (int rc = enqueue(next_enq++)) return rc;
        if (next_enq == next_ready) {   // everything enqueued is published; the next slot is still being expanded
            _mm_pause();
            continue;
        }
        CUDA_TRY(cudaEventSynchronize(h->hev_stage[next_ready % kStageSlots]));
        ready.store(++next_ready, std::memory_order_release);
    }
    CUDA_TRY(cudaStreamSynchronize(comp));
    for (int s = 0; s < kHostCopyStreams; ++s) CUDA_TRY(cudaStreamSynchronize(h->hxstream[s]));
    join.failed = false;   // the destructor waits for the last expansions
    return BLF_CCM_OK;
}

// tuning knob for the host pipeline (not part of the reference-facing surface)
extern "C" int blf_ccm_set_host_chunk(blf_ccm_handle* h, int64_t contacts)
{
    if (!valid(h)) return fail(BLF_CCM_ERR_INVALID_HANDLE, "invalid handle");
    if (contacts < 32) return fail(BLF_CCM_ERR_INVALID_ARG, "chunk must be >= 32 contacts");
    h->host_chunk_pref = contacts & ~1LL;   // even: see the expansion workers
    return BLF_CCM_OK;
}

// worker threads that expand the compact control-matrix download; 0 = dense download, -1 = automatic
extern "C" int blf_ccm_set_host_threads(blf_ccm_handle* h, int threads)
{
    if (!valid(h)) return fail(BLF_CCM_ERR_INVALID_HANDLE, "invalid handle");
    if (threads < -1 || threads > 64) return fail(BLF_CCM_ERR_INVALID_ARG, "threads must be -1 (automatic) or 0..64");
    h->host_threads = threads;
    return BLF_CCM_OK;
}

// ---- surface points ------------------------------------------------------------------------------

extern "C" int blf_ccm_eval_surface_points(blf_ccm_handle* h, const double* host_twist,
                                           const double* host_pose, const double* host_null_pose,
                                           int64_t m, const double* xy, double* force_out,
                                           double* torque_out, void* stream)
{
    CHECK_HANDLE(h);
    if (!h->have_params) return fail(BLF_CCM_ERR_NOT_INITIALIZED, "call blf_ccm_set_uniform_params first");
    if (m < 0 || !host_twist || !host_pose || !host_null_pose || (m > 0 && !xy))
        return fail(BLF_CCM_ERR_INVALID_ARG, "NULL input or m < 0");
    if (m == 0) return BLF_CCM_OK;
    PointArgs a;
    memcpy(a.tw, host_twist, sizeof(a.tw));
    memcpy(a.pose, host_pose, sizeof(a.pose));
    memcpy(a.null, host_null_pose, sizeof(a.null));
    a.length = h->length;
    a.width = h->width;
    a.k = h->spring;
    a.b = h->damper;
    a.xy = xy;
    a.force = force_out;
    a.torque = torque_out;
    a.m = m;
    const int threads = 128;
    const int grid = static_cast<int>(std::min<long long>((m + threads - 1) / threads, 8LL * h->sm_count));
    ccm_surface_points_kernel<<<grid, threads, 0, static_cast<cudaStream_t>(stream)>>>(a);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return BLF_CCM_OK;
}

// ---- rollout cost + arg-min ----------------------------------------------------------------------

extern "C" int blf_ccm_argmin_exchange_p2p(blf_ccm_handle* h, const void* best, void* global_best,
                                           void* stream);

// an empty shard has no reduction launch to carry the fused exchange: run it on its own
static int exchange_if_fused(blf_ccm_handle* h, const void* best, void* stream)
{
    if (!h->p2p_connected || !h->p2p_fused_out) return BLF_CCM_OK;
    return blf_ccm_argmin_exchange_p2p(h, best, h->p2p_fused_out, stream);
}

// nranks = 0 unless the fused exchange is enabled (blf_ccm_rollout_set_exchange)
static void fill_reduce_p2p(blf_ccm_handle* h, const CostIdx* mine, P2pArgs& p)
{
    memset(&p, 0, sizeof(p));
    if (!h->p2p_connected || !h->p2p_fused_out) return;
    for (int r = 0; r < h->p2p_nranks; ++r) p.peer[r] = h->p2p_peer[r];
    p.mine = mine;
    p.out = h->p2p_fused_out;
    p.epoch = ++h->p2p_epoch;
    p.nranks = h->p2p_nranks;
    p.rank = h->p2p_rank;
}

template <unsigned OUT, bool HET>
struct CostLaunch {
    static int run(blf_ccm_handle* h, const SoaArgs& a, cudaStream_t st)
    {
        constexpr int threads = 128;
        const size_t smem = (OUT & M_CTRL) ? size_t(threads / 32) * 32 * 288 : 0;
        auto k = ccm_soa_kernel<OUT, HET, true>;
        int cap = 0;
        if (int rc = persistent_blocks(h, k, threads, smem, &cap)) return rc;
        const long long grid = (a.n + threads - 1) / threads;
        if (grid > 0x7fffffffLL) return fail(BLF_CCM_ERR_INVALID_ARG, "n too large for one launch");
        CUDA_TRY(launch_pdl(h, k, grid, threads, smem, st, a));
        CUDA_TRY(cudaGetLastError());
        h->launches++;
        return BLF_CCM_OK;
    }
};

template <bool HET>
static int dispatch_cost(unsigned out, blf_ccm_handle* h, const SoaArgs& a, cudaStream_t st)
{
    switch (out) {  // outputs written besides the cost: any subset of wrench|autodyn|ctrl
    case 0: return CostLaunch<0, HET>::run(h, a, st);
    case 1: return CostLaunch<1, HET>::run(h, a, st);
    case 2: return CostLaunch<2, HET>::run(h, a, st);
    case 3: return CostLaunch<3, HET>::run(h, a, st);
    case 4: return CostLaunch<4, HET>::run(h, a, st);
    case 5: return CostLaunch<5, HET>::run(h, a, st);
    case 6: return CostLaunch<6, HET>::run(h, a, st);
    case 7: return CostLaunch<7, HET>::run(h, a, st);
    default: return fail(BLF_CCM_ERR_INVALID_ARG, "rollout out_mask %u: only wrench|autodyn|ctrl", out);
    }
}

extern "C" int blf_ccm_rollout_cost_argmin_soa(blf_ccm_handle* h, int64_t n_rollouts,
                                               int64_t rollout_len, const double* const* in_planes,
                                               const double* const* param_planes, unsigned out_mask,
                                               double* const* wrench_planes,
                                               double* const* autodyn_planes, double* ctrl,
                                               const double* host_wrench_ref,
                                               const double* host_weights, int64_t index_base,
                                               double* cost, void* best, void* stream)
{
    CHECK_HANDLE(h);
    if (n_rollouts < 0 || rollout_len <= 0) return fail(BLF_CCM_ERR_INVALID_ARG, "n_rollouts < 0 or rollout_len <= 0");
    if (out_mask > 7u) return fail(BLF_CCM_ERR_INVALID_ARG, "rollout out_mask %u: only wrench|autodyn|ctrl", out_mask);
    if (!host_wrench_ref || !host_weights || !best)
        return fail(BLF_CCM_ERR_INVALID_ARG, "wrench_ref, weights and best are required");
    if (!aligned16(best)) return fail(BLF_CCM_ERR_INVALID_ARG, "best must be 16-byte aligned");
    if (n_rollouts == 0) {  // nothing to compare: best = (+inf, -1); still take part in the exchange
        if (int rc = blf_ccm_argmin_pairs(h, 0, best, best, stream)) return rc;
        return exchange_if_fused(h, best, stream);
    }
    SoaArgs a;
    bool vec = false;
    if (int rc = fill_soa_args(h, n_rollouts * rollout_len, in_planes, param_planes, out_mask,
                               out_mask | BLF_CCM_WRENCH, wrench_planes, autodyn_planes, ctrl,
                               nullptr, a, vec))
        return rc;
    // per-(rollout, tile) partial sums: a rollout of length L intersects at most (L+62)/32 tiles
    const int slots = static_cast<int>((rollout_len + 62) / 32);
    const size_t need = size_t(n_rollouts) * slots * sizeof(double);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (h->partials_bytes < need) {
        if (h->partials) {
            if (int rc = scratch_quiesce(h)) return rc;  // a previous launch may still read the old buffer
            CUDA_TRY(cudaFree(h->partials));
            h->partials = nullptr;
            h->partials_bytes = 0;
        }
        CUDA_TRY(cudaMalloc(&h->partials, need));
        h->partials_bytes = need;
    }
    if (int rc = scratch_acquire(h, st)) return rc;
    a.rollout_len = rollout_len;
    memcpy(a.ref, host_wrench_ref, sizeof(a.ref));
    a.wf = host_weights[0];
    a.wt = host_weights[1];
    a.partials = h->partials;
    a.slots = slots;
    h->last_path = ((out_mask & BLF_CCM_CTRL) && !a.ctrl_bulk) ? BLF_CCM_PATH_DIRECT64 : BLF_CCM_PATH_BULK;
    if (int rc = param_planes ? dispatch_cost<true>(out_mask, h, a, st)
                              : dispatch_cost<false>(out_mask, h, a, st))
        return rc;

    ReduceArgs ra;
    ra.partials = h->partials;
    ra.slots = slots;
    ra.fixed_count = 0;
    ra.n_rollouts = n_rollouts;
    ra.rollout_len = rollout_len;
    ra.index_base = index_base;
    ra.cost = cost;
    ra.block_best = h->block_best;
    ra.counter = h->counter;
    ra.best = static_cast<CostIdx*>(best);
    fill_reduce_p2p(h, ra.best, ra.p2p);
    const int threads = 128;
    const int grid = static_cast<int>(std::min<long long>((n_rollouts + threads - 1) / threads, kMaxPartials));
    CUDA_TRY(launch_pdl(h, ccm_cost_reduce_kernel, grid, threads, 0, st, ra));
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_argmin_pairs(blf_ccm_handle* h, int n_pairs, const void* pairs, void* best,
                                    void* stream)
{
    CHECK_HANDLE(h);
    if (n_pairs < 0 || !pairs || !best) return fail(BLF_CCM_ERR_INVALID_ARG, "NULL pairs/best or n_pairs < 0");
    ccm_argmin_pairs_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const CostIdx*>(pairs), n_pairs, static_cast<CostIdx*>(best));
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return BLF_CCM_OK;
}

// ---- batched recursive least squares -------------------------------------------------------------

// software-pipelined SoA kernel: grid = what is resident (BPS blocks per SM), blocks walk over tiles
template <int P, int M, int BPS>
static int rls_launch_pipe(blf_ccm_handle* h, const RlsArgs& a, cudaStream_t st)
{
    using Cfg = RlsPipe<P, M>;
    auto kern = rls_advance_pipe_kernel<P, M, BPS>;
    // opt in to > 48 KB of dynamic shared memory (a per-device function attribute; the call is a
    // few hundred nanoseconds, so it is simply repeated rather than cached across threads)
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    const long long ntiles = (a.n + Cfg::THREADS - 1) / Cfg::THREADS;
    const long long resident = static_cast<long long>(h->sm_count) * BPS;
    const int grid = static_cast<int>(std::min<long long>(ntiles, resident));
    if (grid > 0) kern<<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(a, ntiles);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return BLF_CCM_OK;
}

template <int P, int M, bool AOS>
static int rls_launch(blf_ccm_handle* h, const RlsArgs& a, cudaStream_t st)
{
    if constexpr (!AOS) {
        constexpr int kDefaultBps = (P <= 2 ? 3 : 2);
        // measured (profiles/r01_rls_throughput_v3.log): 96.7 % vs 88.1 % of the HBM peak at 8.4 M
        // estimators, 82 % vs 78 % at 819 200; a 4-blocks/SM build (128 registers, 168 B spilled)
        // dropped to 77 % and was removed
        if (h->tune_rls_pipe != 1) return rls_launch_pipe<P, M, kDefaultBps>(h, a, st);
    }
    const int threads = 128;
    const long long grid = (a.n + threads - 1) / threads;
    if (grid > 0x7fffffffLL) return fail(BLF_CCM_ERR_INVALID_ARG, "n too large for one launch");
    rls_advance_kernel<P, M, AOS><<<static_cast<int>(grid), threads, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return BLF_CCM_OK;
}

template <int P, bool AOS>
static int rls_dispatch_m(int m, blf_ccm_handle* h, const RlsArgs& a, cudaStream_t st)
{
    switch (m) {
    case 1: return rls_launch<P, 1, AOS>(h, a, st);
    case 2: return rls_launch<P, 2, AOS>(h, a, st);
    case 3: return rls_launch<P, 3, AOS>(h, a, st);
    case 4: return rls_launch<P, 4, AOS>(h, a, st);
    case 5: return rls_launch<P, 5, AOS>(h, a, st);
    case 6: return rls_launch<P, 6, AOS>(h, a, st);
    default: return fail(BLF_CCM_ERR_INVALID_ARG, "m = %d unsupported (1..6)", m);
    }
}

template <bool AOS>
static int rls_dispatch(int p, int m, blf_ccm_handle* h, const RlsArgs& a, cudaStream_t st)
{
    switch (p) {
    case 1: return rls_dispatch_m<1, AOS>(m, h, a, st);
    case 2: return rls_dispatch_m<2, AOS>(m, h, a, st);
    case 3: return rls_dispatch_m<3, AOS>(m, h, a, st);
    case 4: return rls_dispatch_m<4, AOS>(m, h, a, st);
    default: return fail(BLF_CCM_ERR_INVALID_ARG, "p = %d unsupported (1..4)", p);
    }
}

// sizes / covariances the register kernels cover: 1..4 parameters, 1..6 measurements and
// lambda * r[i] > 0 for every measurement (S symmetric positive definite, LDL^T without pivoting);
// everything else the reference accepts goes to rls_advance_generic_kernel (partial-pivot LU)
static bool rls_fast_path(int p, int m, double lambda, const double* cov)
{
    if (p > kRlsMaxP || m > kRlsMaxM) return false;
    for (int i = 0; i < m; ++i)
        if (!(lambda * cov[i] > 0.0)) return false;
    return true;
}

static int rls_check_sizes(int p, int m, double lambda, const double* cov)
{
    if (p < 1 || p > 512) return fail(BLF_CCM_ERR_INVALID_ARG, "p = %d unsupported (1..512)", p);
    if (m < 1 || m > 512) return fail(BLF_CCM_ERR_INVALID_ARG, "m = %d unsupported (1..512)", m);
    if (!cov) return fail(BLF_CCM_ERR_INVALID_ARG, "measurement covariance is NULL");
    if (!(lambda != 0.0)) return fail(BLF_CCM_ERR_INVALID_ARG, "lambda must be non-zero");
    return BLF_CCM_OK;
}

// the general kernel: scratch = [lambda r (m) | pointer table (SoA) | work], grown on demand
static int rls_generic(blf_ccm_handle* h, long long n, int p, int m, const double* const* host_tabs,
                       const double* dY, const double* dz, double* dtheta, double* dP,
                       const double* host_cov, double lambda, cudaStream_t st)
{
    const size_t ntab = host_tabs ? size_t(m) * p + m + p + size_t(p) * p : 0;
    const size_t head = (size_t(m) + ntab + 1) & ~size_t(1);           // doubles; pointers are 8 bytes too
    const size_t need = (head + size_t(rls_gen_work_doubles(p, m)) * size_t(n)) * sizeof(double);
    if (h->gen_bytes < need) {
        if (h->gen_work) {
            CUDA_TRY(cudaDeviceSynchronize());
            CUDA_TRY(cudaFree(h->gen_work));
            h->gen_work = nullptr;
            h->gen_bytes = 0;
        }
        CUDA_TRY(cudaMalloc(&h->gen_work, need));
        h->gen_bytes = need;
    }
    std::vector<double> headbuf(head, 0.0);
    for (int i = 0; i < m; ++i) headbuf[i] = lambda * host_cov[i];
    if (host_tabs) memcpy(headbuf.data() + m, host_tabs, ntab * sizeof(double*));
    // pageable source: the copy has left the host buffer when the call returns
    CUDA_TRY(cudaMemcpyAsync(h->gen_work, headbuf.data(), head * sizeof(double), cudaMemcpyHostToDevice, st));
    RlsGenArgs a;
    memset(&a, 0, sizeof(a));
    a.tabs = host_tabs ? reinterpret_cast<const double* const*>(h->gen_work + m) : nullptr;
    a.Y = dY;
    a.z = dz;
    a.theta = dtheta;
    a.cov = dP;
    a.lr = h->gen_work;
    a.work = h->gen_work + head;
    a.lambda = lambda;
    a.n = n;
    a.p = p;
    a.m = m;
    const int threads = 64;
    const long long grid = (n + threads - 1) / threads;
    if (grid > 0x7fffffffLL) return fail(BLF_CCM_ERR_INVALID_ARG, "n too large for one launch");
    rls_advance_generic_kernel<<<static_cast<int>(grid), threads, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return BLF_CCM_OK;
}

extern "C" int blf_rls_advance_batch(blf_ccm_handle* h, int64_t n, int p, int m,
                                     const double* const* regressor_planes,
                                     const double* const* measurement_planes,
                                     const double* host_measurement_cov, double lambda,
                                     double* const* state_planes, double* const* cov_planes,
                                     void* stream)
{
    CHECK_HANDLE(h);
    if (n < 0) return fail(BLF_CCM_ERR_INVALID_ARG, "n < 0");
    if (int rc = rls_check_sizes(p, m, lambda, host_measurement_cov)) return rc;
    if (n == 0) return BLF_CCM_OK;
    if (!regressor_planes || !measurement_planes || !state_planes || !cov_planes)
        return fail(BLF_CCM_ERR_INVALID_ARG, "a plane-pointer array is NULL");
    auto bad = [](const void* q) { return !q || !aligned8(q); };
    if (!rls_fast_path(p, m, lambda, host_measurement_cov)) {
        // any size / indefinite lambda R: the reference's own algorithm (pivoted LU)
        std::vector<const double*> tabs;
        for (int i = 0; i < m * p; ++i) tabs.push_back(regressor_planes[i]);
        for (int i = 0; i < m; ++i) tabs.push_back(measurement_planes[i]);
        for (int i = 0; i < p; ++i) tabs.push_back(state_planes[i]);
        for (int i = 0; i < p * p; ++i) tabs.push_back(cov_planes[i]);
        for (size_t i = 0; i < tabs.size(); ++i)
            if (bad(tabs[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "plane %zu NULL or misaligned", i);
        return rls_generic(h, n, p, m, tabs.data(), nullptr, nullptr, nullptr, nullptr, host_measurement_cov,
                           lambda, static_cast<cudaStream_t>(stream));
    }
    RlsArgs a;
    memset(&a, 0, sizeof(a));
    a.n = n;
    a.lambda = lambda;
    for (int i = 0; i < m; ++i) a.w[i] = lambda * host_measurement_cov[i];
    for (int i = 0; i < m * p; ++i) {
        if (bad(regressor_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "regressor_planes[%d] NULL or misaligned", i);
        a.Y[i] = regressor_planes[i];
    }
    for (int i = 0; i < m; ++i) {
        if (bad(measurement_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "measurement_planes[%d] NULL or misaligned", i);
        a.z[i] = measurement_planes[i];
    }
    for (int i = 0; i < p; ++i) {
        if (bad(state_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "state_planes[%d] NULL or misaligned", i);
        a.theta[i] = state_planes[i];
    }
    for (int i = 0; i < p * p; ++i) {
        if (bad(cov_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "cov_planes[%d] NULL or misaligned", i);
        a.cov[i] = cov_planes[i];
    }
    return rls_dispatch<false>(p, m, h, a, static_cast<cudaStream_t>(stream));
}

extern "C" int blf_rls_advance_host(blf_ccm_handle* h, int64_t n, int p, int m, const double* Y,
                                    const double* z, const double* host_measurement_cov,
                                    double lambda, double* theta, double* P)
{
    CHECK_HANDLE(h);
    if (n < 0) return fail(BLF_CCM_ERR_INVALID_ARG, "n < 0");
    if (int rc = rls_check_sizes(p, m, lambda, host_measurement_cov)) return rc;
    if (n == 0) return BLF_CCM_OK;
    if (!Y || !z || !theta || !P) return fail(BLF_CCM_ERR_INVALID_ARG, "NULL array");
    const size_t per = size_t(m * p + m + p + p * p);
    const size_t need = size_t(n) * per * sizeof(double);
    if (h->hbytes < need) {
        for (int s = 0; s < kHostSlots; ++s) {
            if (h->hbuf[s]) CUDA_TRY(cudaFree(h->hbuf[s]));
            h->hbuf[s] = nullptr;
        }
        for (int s = 0; s < kHostSlots; ++s) CUDA_TRY(cudaMalloc(&h->hbuf[s], need));
        h->hbytes = need;
    }
    if (!h->hstream[0]) CUDA_TRY(cudaStreamCreateWithFlags(&h->hstream[0], cudaStreamNonBlocking));
    cudaStream_t st = h->hstream[0];
    double* dY = h->hbuf[0];
    double* dz = dY + size_t(n) * m * p;
    double* dth = dz + size_t(n) * m;
    double* dP = dth + size_t(n) * p;
    const size_t D = sizeof(double);
    CUDA_TRY(cudaMemcpyAsync(dY, Y, size_t(n) * m * p * D, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dz, z, size_t(n) * m * D, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dth, theta, size_t(n) * p * D, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dP, P, size_t(n) * p * p * D, cudaMemcpyHostToDevice, st));
    if (!rls_fast_path(p, m, lambda, host_measurement_cov)) {
        if (int rc = rls_generic(h, n, p, m, nullptr, dY, dz, dth, dP, host_measurement_cov, lambda, st)) return rc;
    } else {
        RlsArgs a;
        memset(&a, 0, sizeof(a));
        a.n = n;
        a.lambda = lambda;
        for (int i = 0; i < m; ++i) a.w[i] = lambda * host_measurement_cov[i];
        a.Y[0] = dY;
        a.z[0] = dz;
        a.theta[0] = dth;
        a.cov[0] = dP;
        if (int rc = rls_dispatch<true>(p, m, h, a, st)) return rc;
    }
    CUDA_TRY(cudaMemcpyAsync(theta, dth, size_t(n) * p * D, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(P, dP, size_t(n) * p * p * D, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_rls_advance_contacts(blf_ccm_handle* h, int64_t n,
                                            const double* const* in_planes,
                                            const double* const* geometry_planes,
                                            const double* const* measured_wrench_planes,
                                            const double* host_measurement_cov, double lambda,
                                            double* const* state_planes, double* const* cov_planes,
                                            void* stream)
{
    CHECK_HANDLE(h);
    if (n < 0) return fail(BLF_CCM_ERR_INVALID_ARG, "n < 0");
    if (int rc = rls_check_sizes(2, 6, lambda, host_measurement_cov)) return rc;
    if (!rls_fast_path(2, 6, lambda, host_measurement_cov))
        return fail(BLF_CCM_ERR_INVALID_ARG, "the fused identification step needs lambda * measurement covariance > 0 "
                                             "for all six wrench components (use blf_rls_advance_batch otherwise)");
    if (n == 0) return BLF_CCM_OK;
    if (!geometry_planes && !h->have_params)
        return fail(BLF_CCM_ERR_NOT_INITIALIZED,
                    "no geometry: call blf_ccm_set_uniform_params or pass geometry_planes");
    if (!in_planes || !measured_wrench_planes || !state_planes || !cov_planes)
        return fail(BLF_CCM_ERR_INVALID_ARG, "a plane-pointer array is NULL");
    CcmRlsArgs a;
    memset(&a, 0, sizeof(a));
    a.n = n;
    a.lambda = lambda;
    a.length = h->length;
    a.width = h->width;
    auto bad = [](const void* q) { return !q || !aligned8(q); };
    const unsigned live = live_planes(M_REGRESSOR);
    for (int i = 0; i < 30; ++i) {
        if (!(live & (1u << i))) continue;
        if (bad(in_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "in_planes[%d] NULL or misaligned", i);
        a.in[i] = in_planes[i];
    }
    for (int i = 0; i < 6; ++i) {
        if (bad(measured_wrench_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "measured_wrench_planes[%d] NULL or misaligned", i);
        a.z[i] = measured_wrench_planes[i];
        a.w[i] = lambda * host_measurement_cov[i];
    }
    for (int i = 0; i < 2; ++i) {
        if (bad(state_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "state_planes[%d] NULL or misaligned", i);
        a.theta[i] = state_planes[i];
        if (geometry_planes) {
            if (bad(geometry_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "geometry_planes[%d] NULL or misaligned", i);
            a.geom[i] = geometry_planes[i];
        }
    }
    for (int i = 0; i < 4; ++i) {
        if (bad(cov_planes[i])) return fail(BLF_CCM_ERR_INVALID_ARG, "cov_planes[%d] NULL or misaligned", i);
        a.cov[i] = cov_planes[i];
    }
    const int threads = 128;
    const long long grid = (n + threads - 1) / threads;
    if (grid > 0x7fffffffLL) return fail(BLF_CCM_ERR_INVALID_ARG, "n too large for one launch");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (geometry_planes) ccm_rls_kernel<true><<<static_cast<int>(grid), threads, 0, st>>>(a);
    else ccm_rls_kernel<false><<<static_cast<int>(grid), threads, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return BLF_CCM_OK;
}

// ---- memory / stream helpers ---------------------------------------------------------------------

extern "C" int blf_ccm_device_alloc(blf_ccm_handle* h, uint64_t bytes, void** out)
{
    CHECK_HANDLE(h);
    if (!out) return fail(BLF_CCM_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (bytes == 0) return BLF_CCM_OK;
    CUDA_TRY(cudaMalloc(out, bytes));
    return BLF_CCM_OK;
}

// Compute Data Compression is requested per allocation through the driver's virtual-memory calls
// (cuMemCreate with CU_MEM_ALLOCATION_COMP_GENERIC).  The entry points are looked up once through
// the runtime (no -lcuda), as cuTensorMapEncodeTiled is; ok is false when one of them is missing.
struct VmmApi {
    bool ok = false;
    CUresult (*get_attribute)(int*, CUdevice_attribute, CUdevice) = nullptr;
    CUresult (*granularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags) = nullptr;
    CUresult (*create)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long) = nullptr;
    CUresult (*properties)(CUmemAllocationProp*, CUmemGenericAllocationHandle) = nullptr;
    CUresult (*reserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
    CUresult (*map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
    CUresult (*set_access)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
    CUresult (*unmap)(CUdeviceptr, size_t) = nullptr;
    CUresult (*address_free)(CUdeviceptr, size_t) = nullptr;
    CUresult (*release)(CUmemGenericAllocationHandle) = nullptr;
};

static const VmmApi& vmm_api()
{
    static const VmmApi api = [] {
        VmmApi a;
        bool all = true;
        auto get = [&all](const char* name, auto& fn) {
            void* p = nullptr;
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess ||
                q != cudaDriverEntryPointSuccess) {
                cudaGetLastError();
                p = nullptr;
            }
            fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(p);
            all = all && p != nullptr;
        };
        get("cuDeviceGetAttribute", a.get_attribute);
        get("cuMemGetAllocationGranularity", a.granularity);
        get("cuMemCreate", a.create);
        get("cuMemGetAllocationPropertiesFromHandle", a.properties);
        get("cuMemAddressReserve", a.reserve);
        get("cuMemMap", a.map);
        get("cuMemSetAccess", a.set_access);
        get("cuMemUnmap", a.unmap);
        get("cuMemAddressFree", a.address_free);
        get("cuMemRelease", a.release);
        a.ok = all;
        return a;
    }();
    return api;
}

// A compressible mapping of `bytes` on the handle's device, or false (nothing held) when the device
// has no compression, the driver does not grant it for this allocation, or any step fails.
static bool vmm_map_compressible(blf_ccm_handle* h, uint64_t bytes, void** out)
{
    const VmmApi& api = vmm_api();
    int supported = 0;
    if (!api.ok ||
        api.get_attribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, h->device) != CUDA_SUCCESS ||
        !supported)
        return false;
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = h->device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    if (api.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0)
        return false;
    const size_t size = (bytes + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle mem = 0;
    if (api.create(&mem, size, &prop, 0) != CUDA_SUCCESS) return false;
    // the driver may drop the request silently: only what it reports as granted counts
    CUmemAllocationProp got = {};
    bool ok = api.properties(&got, mem) == CUDA_SUCCESS &&
              got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC;
    CUdeviceptr base = 0;
    ok = ok && api.reserve(&base, size, gran, 0, 0) == CUDA_SUCCESS;
    bool mapped = ok && api.map(base, size, 0, mem, 0) == CUDA_SUCCESS;
    CUmemAccessDesc access = {};
    access.location = prop.location;
    access.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    ok = mapped && api.set_access(base, size, &access, 1) == CUDA_SUCCESS;
    if (!ok) {
        if (mapped) api.unmap(base, size);
        if (base) api.address_free(base, size);
        api.release(mem);
        return false;
    }
    {
        std::lock_guard<std::mutex> lock(h->vmm_mutex);
        h->vmm[static_cast<uintptr_t>(base)] = VmmRange{size, mem};
    }
    *out = reinterpret_cast<void*>(base);
    return true;
}

// Unlike cudaFree, cuMemUnmap does not wait for work still using the range: the device is
// synchronised first.
static int vmm_unmap(blf_ccm_handle* h, uintptr_t base, const VmmRange& r)
{
    CUDA_TRY(cudaDeviceSynchronize());
    const VmmApi& api = vmm_api();
    CUresult e = api.unmap(base, r.size);
    if (e == CUDA_SUCCESS) e = api.address_free(base, r.size);
    if (e == CUDA_SUCCESS) e = api.release(r.mem);
    if (e != CUDA_SUCCESS) return fail(BLF_CCM_ERR_CUDA, "releasing a compressible allocation: CUresult %d", int(e));
    return BLF_CCM_OK;
}

static void vmm_release_all(blf_ccm_handle* h)
{
    std::lock_guard<std::mutex> lock(h->vmm_mutex);
    for (const auto& kv : h->vmm) vmm_unmap(h, kv.first, kv.second);
    h->vmm.clear();
}

extern "C" int blf_ccm_device_alloc_compressible(blf_ccm_handle* h, uint64_t bytes, void** out, int* granted)
{
    CHECK_HANDLE(h);
    if (!out) return fail(BLF_CCM_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (granted) *granted = 0;
    if (bytes == 0) return BLF_CCM_OK;
    CUDA_TRY(cudaFree(nullptr));   // the driver calls below need the device's primary context current
    if (vmm_map_compressible(h, bytes, out)) {
        if (granted) *granted = 1;
        return BLF_CCM_OK;
    }
    CUDA_TRY(cudaMalloc(out, bytes));
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_pointer_is_compressible(blf_ccm_handle* h, const void* ptr, int* out)
{
    CHECK_HANDLE(h);
    if (!out) return fail(BLF_CCM_ERR_INVALID_ARG, "out is NULL");
    const uintptr_t p = reinterpret_cast<uintptr_t>(ptr);
    std::lock_guard<std::mutex> lock(h->vmm_mutex);
    auto it = h->vmm.upper_bound(p);
    *out = it != h->vmm.begin() && p < std::prev(it)->first + std::prev(it)->second.size;
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_device_free(blf_ccm_handle* h, void* ptr)
{
    CHECK_HANDLE(h);
    if (!ptr) return BLF_CCM_OK;
    {
        std::lock_guard<std::mutex> lock(h->vmm_mutex);
        auto it = h->vmm.find(reinterpret_cast<uintptr_t>(ptr));
        if (it != h->vmm.end()) {
            const VmmRange r = it->second;
            h->vmm.erase(it);
            return vmm_unmap(h, reinterpret_cast<uintptr_t>(ptr), r);
        }
    }
    CUDA_TRY(cudaFree(ptr));
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_host_alloc(blf_ccm_handle* h, uint64_t bytes, void** out)
{
    CHECK_HANDLE(h);
    if (!out) return fail(BLF_CCM_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (bytes == 0) return BLF_CCM_OK;
    CUDA_TRY(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_host_free(blf_ccm_handle* h, void* ptr)
{
    CHECK_HANDLE(h);
    if (ptr) CUDA_TRY(cudaFreeHost(ptr));
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_copy_h2d(blf_ccm_handle* h, void* dst_device, const void* src_host,
                                uint64_t bytes, void* stream)
{
    CHECK_HANDLE(h);
    if (bytes && (!dst_device || !src_host)) return fail(BLF_CCM_ERR_INVALID_ARG, "NULL pointer");
    if (bytes)
        CUDA_TRY(cudaMemcpyAsync(dst_device, src_host, bytes, cudaMemcpyHostToDevice,
                                 static_cast<cudaStream_t>(stream)));
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_copy_d2h(blf_ccm_handle* h, void* dst_host, const void* src_device,
                                uint64_t bytes, void* stream)
{
    CHECK_HANDLE(h);
    if (bytes && (!dst_host || !src_device)) return fail(BLF_CCM_ERR_INVALID_ARG, "NULL pointer");
    if (bytes)
        CUDA_TRY(cudaMemcpyAsync(dst_host, src_device, bytes, cudaMemcpyDeviceToHost,
                                 static_cast<cudaStream_t>(stream)));
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_stream_synchronize(blf_ccm_handle* h, void* stream)
{
    CHECK_HANDLE(h);
    CUDA_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    return BLF_CCM_OK;
}

// ---- optional NCCL exchange (dlopen: no link-time dependency) ------------------------------------

typedef int (*nccl_allgather_fn)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef const char* (*nccl_errstr_fn)(int);

extern "C" int blf_ccm_argmin_allgather_nccl(blf_ccm_handle* h, void* comm, int nranks,
                                             const void* best, void* gathered, void* global_best,
                                             void* stream)
{
    CHECK_HANDLE(h);
    if (!comm || nranks <= 0 || !best || !gathered || !global_best)
        return fail(BLF_CCM_ERR_INVALID_ARG, "NULL comm/buffers or nranks <= 0");
    static nccl_allgather_fn allgather = nullptr;
    static nccl_errstr_fn errstr = nullptr;
    if (!allgather) {
        void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return fail(BLF_CCM_ERR_NCCL, "libnccl not found: %s", dlerror());
        allgather = reinterpret_cast<nccl_allgather_fn>(dlsym(lib, "ncclAllGather"));
        errstr = reinterpret_cast<nccl_errstr_fn>(dlsym(lib, "ncclGetErrorString"));
        if (!allgather) return fail(BLF_CCM_ERR_NCCL, "ncclAllGather not found in libnccl");
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // 16 bytes per rank as ncclInt8 (datatype 0)
    const int rc = allgather(best, gathered, 16, /*ncclInt8*/ 0, comm, st);
    if (rc != 0) return fail(BLF_CCM_ERR_NCCL, "ncclAllGather: %s", errstr ? errstr(rc) : "error");
    return blf_ccm_argmin_pairs(h, nranks, gathered, global_best, stream);
}

// ---- peer-memory arg-min exchange (NVLink / NVSwitch P2P through CUDA IPC) ------------------------

extern "C" int blf_ccm_p2p_mailbox_create(blf_ccm_handle* h, int nranks, int rank, void* ipc_handle_out)
{
    CHECK_HANDLE(h);
    if (nranks < 1 || nranks > kP2pMaxRanks || rank < 0 || rank >= nranks || !ipc_handle_out)
        return fail(BLF_CCM_ERR_INVALID_ARG, "nranks 1..%d, 0 <= rank < nranks, ipc_handle_out non-NULL",
                    kP2pMaxRanks);
    static_assert(sizeof(cudaIpcMemHandle_t) == BLF_CCM_IPC_HANDLE_BYTES, "IPC handle size");
    p2p_release(h);
    const size_t bytes = sizeof(P2pSlot) * 2 * nranks;
    CUDA_TRY(cudaMalloc(&h->p2p_local, bytes));
    CUDA_TRY(cudaMemset(h->p2p_local, 0, bytes));
    CUDA_TRY(cudaDeviceSynchronize());   // zeroed before any peer can write
    cudaIpcMemHandle_t ipc;
    CUDA_TRY(cudaIpcGetMemHandle(&ipc, h->p2p_local));
    memcpy(ipc_handle_out, &ipc, sizeof(ipc));
    h->p2p_nranks = nranks;
    h->p2p_rank = rank;
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_p2p_mailbox_connect(blf_ccm_handle* h, const void* all_ipc_handles)
{
    CHECK_HANDLE(h);
    if (!h->p2p_local) return fail(BLF_CCM_ERR_NOT_INITIALIZED, "call blf_ccm_p2p_mailbox_create first");
    if (!all_ipc_handles) return fail(BLF_CCM_ERR_INVALID_ARG, "all_ipc_handles is NULL");
    if (h->p2p_connected) return fail(BLF_CCM_ERR_INVALID_ARG, "mailbox already connected");
    const char* src = static_cast<const char*>(all_ipc_handles);
    for (int r = 0; r < h->p2p_nranks; ++r) {
        if (r == h->p2p_rank) {
            h->p2p_peer[r] = h->p2p_local;
            continue;
        }
        cudaIpcMemHandle_t ipc;
        memcpy(&ipc, src + size_t(r) * sizeof(ipc), sizeof(ipc));
        void* mapped = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&mapped, ipc, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(BLF_CCM_ERR_CUDA, "cudaIpcOpenMemHandle(rank %d): %s (peer access over NVLink/PCIe "
                        "between the two devices is required)", r, cudaGetErrorString(e));
        }
        h->p2p_peer[r] = static_cast<P2pSlot*>(mapped);
    }
    h->p2p_connected = true;
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_argmin_exchange_p2p(blf_ccm_handle* h, const void* best, void* global_best,
                                           void* stream)
{
    CHECK_HANDLE(h);
    if (!h->p2p_connected) return fail(BLF_CCM_ERR_NOT_INITIALIZED, "mailbox not connected");
    if (!best || !global_best) return fail(BLF_CCM_ERR_INVALID_ARG, "NULL best / global_best");
    P2pArgs a;
    memset(&a, 0, sizeof(a));
    for (int r = 0; r < h->p2p_nranks; ++r) a.peer[r] = h->p2p_peer[r];
    a.mine = static_cast<const CostIdx*>(best);
    a.out = static_cast<CostIdx*>(global_best);
    a.epoch = ++h->p2p_epoch;
    a.nranks = h->p2p_nranks;
    a.rank = h->p2p_rank;
    ccm_p2p_exchange_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(a);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_rollout_set_exchange(blf_ccm_handle* h, void* global_best)
{
    CHECK_HANDLE(h);
    if (global_best && !h->p2p_connected)
        return fail(BLF_CCM_ERR_NOT_INITIALIZED, "mailbox not connected");
    if (global_best && !aligned16(global_best))
        return fail(BLF_CCM_ERR_INVALID_ARG, "global_best must be 16-byte aligned");
    h->p2p_fused_out = static_cast<CostIdx*>(global_best);
    return BLF_CCM_OK;
}

extern "C" int blf_ccm_p2p_mailbox_destroy(blf_ccm_handle* h)
{
    CHECK_HANDLE(h);
    CUDA_TRY(cudaDeviceSynchronize());
    p2p_release(h);
    return BLF_CCM_OK;
}

// ---- System component (rows 2 and 3 of SURVEY.md section 8(f)) -----------------------------------
#include "sys_capi.inc"
