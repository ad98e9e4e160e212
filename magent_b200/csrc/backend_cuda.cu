// backend_cuda.cu -- the sm_100a backend: CUDA runtime plumbing + every kernel of the engine.
//
// Kernels (DESIGN.md §5):
//   step_kernel_cta   one CTA per arena runs the whole step pipeline (run_step) with __syncthreads
//                     between phases; arenas are looped grid-stride.          [many small arenas]
//   step_kernel_grid  cooperative launch; the whole grid is one team per arena with grid.sync()
//                     between phases.                                          [one huge arena]
//   cull_kernel_*     clear_dead: stable compaction into the ping-pong SoA buffers.
//   offsets_kernel    prefix of per-arena counts -> ABI concatenation offsets.
//   minimap_*         per (arena, group) histogram of coarse cells + normalisation.
//   obs_render_kernel the observation gather: the HBM-write-bound kernel the roofline is quoted on.
//   info_kernel       id/pos/alive/reward gathers and the action scatter.
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdio.h>
#include <stdlib.h>
#include <string>
#include <string.h>
#include <atomic>
#include <mutex>
#include <vector>

#include "backend.h"
#if defined(MG_PHASE_TIMING)
namespace mg { __device__ long long mg_phase_clock[8 * 32]; }
#endif
#include "obs_phases.h"

namespace cg = cooperative_groups;

namespace mg {
[[noreturn]] void fatal(const char *fmt, ...);
namespace be {

#define CUDA_CHECK(expr)                                                                          \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) mg::fatal("CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e),   \
                                         __FILE__, __LINE__, #expr);                              \
    } while (0)

static std::atomic<long long> g_launches{0};       // instrumentation only (magent_b200_launch_count)

// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to (function, device), not to an engine: it is only ever raised,
// under a lock, so that a second engine with a smaller need cannot pull it from under the first
enum { ATTR_STEP = 0, ATTR_OBS0 = 1, ATTR_N = 1 + 8, ATTR_MAX_DEVICES = 64 };
static std::mutex g_attr_mu;
static size_t g_attr_smem[ATTR_MAX_DEVICES][ATTR_N];
template <class K>
static void ensure_dynamic_smem(int device, int slot, K kernel, size_t smem) {
    std::lock_guard<std::mutex> lk(g_attr_mu);
    size_t &have = g_attr_smem[device % ATTR_MAX_DEVICES][slot];
    if (smem <= have) return;
    CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    have = smem;
}

// Per-engine device context.  Everything the backend needs to remember between calls lives here, nothing in
// process-global state: two engines on two devices (or on one) never see each other's scratch.
struct Ctx {
    int device = 0, sms = 0;
    cudaStream_t stream = nullptr;       // every kernel of this engine; created blocking, so work queued on the legacy
                                         // default stream (torch's default stream) stays ordered with it both ways
    cudaStream_t copy = nullptr;         // wire / dense DMA traffic (non-blocking; ordered by events)
    cudaEvent_t ev_wire = nullptr, ev_done = nullptr;
    bool profile = false;
    std::vector<cudaEvent_t> events;     // pairs recorded around obs-render launches
    size_t events_used = 0;
    // products of the last launch_obs_prepare
    float *mm_pad = nullptr; size_t mm_pad_n = 0; int mm_stride = 0;
    // per-observer headers of the render kernel
    int4 *obs_hdr = nullptr; size_t obs_hdr_n = 0;
    // cudaFuncSetAttribute caches (per device: a context never changes device)
    struct ObsCfg { size_t smem = (size_t)-1; int ctas_per_sm = 1; } obs_cfg[8];
    int *pin_done = nullptr; size_t pin_done_n = 0;         // pinned read-back of EngineDev::done
    int *pin_counts = nullptr; size_t pin_counts_n = 0;     // pinned read-back of EngineDev::off (clear_dead)
    cudaEvent_t ev_counts = nullptr;
    // wire path (host-buffer observations)
    WireMark *wire_slots = nullptr; size_t wire_slots_n = 0;         // [n_total][n_in] worst-case slots
    WireMark *wire_stream = nullptr; size_t wire_stream_n = 0;       // compacted marks
    WireHdr *wire_hdr = nullptr; size_t wire_hdr_n = 0;
    long long *wire_base = nullptr; size_t wire_base_n = 0;          // [n_chunks + 1] (device)
    int *wire_chunk_total = nullptr;
    // page-locked staging of the above
    WireHdr *h_wire_hdr = nullptr; size_t h_wire_hdr_n = 0;
    WireMark *h_wire_marks = nullptr; size_t h_wire_marks_n = 0;
    long long *h_wire_base = nullptr; size_t h_wire_base_n = 0;
    float *h_mm = nullptr; size_t h_mm_n = 0;
    std::vector<cudaEvent_t> wave_events;
    int waves_queued = 0;
    std::vector<cudaEvent_t> dma_events; size_t dma_head = 0, dma_tail = 0;
    // CUDA graphs (capture_begin / capture_end / graph_launch)
    bool capturing = false;
    std::vector<cudaGraphExec_t> graphs;
};

static void no_capture(const Ctx *c, const char *what) {
    if (c->capturing) mg::fatal("%s is not possible while a CUDA graph is being captured (run one un-captured step first so that "
                                "every buffer has its size)", what);
}

struct DeviceGuard {                     // every entry point runs on its context's device, whatever the caller selected
    explicit DeviceGuard(const Ctx *c) { int cur = -1; cudaGetDevice(&cur); if (cur != c->device) CUDA_CHECK(cudaSetDevice(c->device)); }
};

const char *name() { return "cuda-sm_100a"; }

#if defined(MG_PHASE_TIMING)
extern "C" __attribute__((visibility("default"))) void magent_b200_debug_phase_clocks(long long *out) {
    CUDA_CHECK(cudaMemcpyFromSymbol(out, mg::mg_phase_clock, sizeof(long long) * 8 * 32));
}
#endif

int device_count() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

Ctx *create(int device, std::string *err) {
    int n = device_count();
    if (n <= 0) { if (err) *err = "cudaGetDeviceCount found no device"; return nullptr; }
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess) device = 0;
    }
    if (device >= n) { if (err) *err = "device_id out of range"; return nullptr; }
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) { if (err) *err = cudaGetErrorString(e); return nullptr; }
    cudaDeviceProp prop;
    CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    Ctx *c = new Ctx();
    c->device = device;
    c->sms = prop.multiProcessorCount;
    CUDA_CHECK(cudaStreamCreate(&c->stream));
    CUDA_CHECK(cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking));
    CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_wire, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_counts, cudaEventDisableTiming));
    return c;
}
void destroy(Ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (cudaGraphExec_t e : c->graphs) if (e) cudaGraphExecDestroy(e);
    cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->copy);
    for (cudaEvent_t e : c->events) cudaEventDestroy(e);
    for (cudaEvent_t e : c->wave_events) cudaEventDestroy(e);
    for (cudaEvent_t e : c->dma_events) cudaEventDestroy(e);
    cudaEventDestroy(c->ev_wire); cudaEventDestroy(c->ev_done);
    cudaFree(c->mm_pad); cudaFree(c->obs_hdr);
    cudaFree(c->wire_slots); cudaFree(c->wire_stream); cudaFree(c->wire_hdr); cudaFree(c->wire_base); cudaFree(c->wire_chunk_total);
    cudaEventDestroy(c->ev_counts); cudaFreeHost(c->pin_counts);
    cudaFreeHost(c->pin_done); cudaFreeHost(c->h_wire_hdr); cudaFreeHost(c->h_wire_marks); cudaFreeHost(c->h_wire_base); cudaFreeHost(c->h_mm);
    cudaStreamDestroy(c->stream); cudaStreamDestroy(c->copy);
    delete c;
}
int device_of(const Ctx *c) { return c->device; }
int sm_count(const Ctx *c) { return c->sms; }
void *stream_handle(const Ctx *c) { return (void *)c->stream; }

void *dmalloc(Ctx *c, size_t bytes) { no_capture(c, "a device allocation"); DeviceGuard g(c); void *p = nullptr; CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 16)); return p; }
void dfree(Ctx *c, void *p) { if (p) { DeviceGuard g(c); cudaFree(p); } }
void dmemset(Ctx *c, void *p, int byte, size_t bytes) { DeviceGuard g(c); CUDA_CHECK(cudaMemsetAsync(p, byte, bytes, c->stream)); }
void h2d(Ctx *c, void *dst, const void *src, size_t bytes) {
    if (!bytes) return;
    no_capture(c, "a blocking host-to-device copy");
    DeviceGuard g(c);
    CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
}
void d2h(Ctx *c, void *dst, const void *src, size_t bytes) {
    if (!bytes) return;
    no_capture(c, "a blocking device-to-host copy");
    DeviceGuard g(c);
    CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
}
void d2d(Ctx *c, void *dst, const void *src, size_t bytes) {
    if (!bytes) return;
    DeviceGuard g(c);
    CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, c->stream));
}
void *host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 16, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void host_free(void *p) { if (p) cudaFreeHost(p); }
bool host_register(void *p, size_t bytes) {
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) { cudaGetLastError(); return false; }
    return true;
}
void host_unregister(void *p) { if (cudaHostUnregister(p) != cudaSuccess) cudaGetLastError(); }
bool is_device_ptr(const void *p) {
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}
bool is_pinned_host_ptr(const void *p) {
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}
void sync(Ctx *c) { no_capture(c, "a synchronisation"); DeviceGuard g(c); CUDA_CHECK(cudaStreamSynchronize(c->stream)); CUDA_CHECK(cudaStreamSynchronize(c->copy)); }
long long launch_count() { return g_launches.load(); }
void profile_enable(Ctx *c, bool on) { c->profile = on; c->events_used = 0; }
static void profile_pair(Ctx *c, cudaEvent_t *e0, cudaEvent_t *e1) {
    if (c->events_used + 2 > c->events.size()) {
        for (int i = 0; i < 64; ++i) { cudaEvent_t e; CUDA_CHECK(cudaEventCreate(&e)); c->events.push_back(e); }
    }
    *e0 = c->events[c->events_used]; *e1 = c->events[c->events_used + 1];
    c->events_used += 2;
}
// total device time of the obs-render launches recorded since profile_enable(true); no sync was added
// to the timed region: the events are read here, after the fact
void profile_read(Ctx *c, double *ms, long long *n) {
    DeviceGuard g(c);
    double total = 0.0;
    for (size_t i = 0; i + 1 < c->events_used; i += 2) {
        CUDA_CHECK(cudaEventSynchronize(c->events[i + 1]));
        float t = 0;
        CUDA_CHECK(cudaEventElapsedTime(&t, c->events[i], c->events[i + 1]));
        total += t;
    }
    *ms = total; *n = (long long)(c->events_used / 2);
}

bool capture_begin(Ctx *c) {
    DeviceGuard guard(c);
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    CUDA_CHECK(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed));
    c->capturing = true;
    return true;
}
int capture_end(Ctx *c) {
    DeviceGuard guard(c);
    cudaGraph_t g = nullptr;
    c->capturing = false;
    CUDA_CHECK(cudaStreamEndCapture(c->stream, &g));
    cudaGraphExec_t exec = nullptr;
    CUDA_CHECK(cudaGraphInstantiate(&exec, g, 0));
    CUDA_CHECK(cudaGraphDestroy(g));
    c->graphs.push_back(exec);
    return (int)c->graphs.size() - 1;
}
bool capturing(const Ctx *c) { return c->capturing; }
void graph_launch(Ctx *c, int id) {
    DeviceGuard guard(c);
    if (id < 0 || id >= (int)c->graphs.size() || !c->graphs[id]) mg::fatal("invalid graph id %d", id);
    CUDA_CHECK(cudaGraphLaunch(c->graphs[id], c->stream));
}
void graph_destroy_all(Ctx *c) {
    DeviceGuard guard(c);
    for (cudaGraphExec_t e : c->graphs) if (e) cudaGraphExecDestroy(e);
    c->graphs.clear();
}

static void post_launch(const char *what) {
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) mg::fatal("kernel launch failed (%s): %s", what, cudaGetErrorString(e));
}

// ------------------------------------------------------------------------------------------------
// team contexts
__device__ __forceinline__ int block_excl_scan(int v, int &total) {
    __shared__ int warp_sums[32];
    __shared__ int block_total;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    int incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) warp_sums[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int w = lane < nw ? warp_sums[lane] : 0;
        int wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += t;
        }
        if (lane < nw) warp_sums[lane] = wi - w;          // exclusive prefix of warp totals
        if (lane == 31) block_total = wi;
    }
    __syncthreads();
    int excl = incl - v + warp_sums[wid];
    total = block_total;
    __syncthreads();
    return excl;
}

struct CtaCtx {
    GroupEnum *enum_smem;
    MG_HD GroupEnum *enums() { return enum_smem; }
    MG_HD bool is_cta_leader() const {
#if defined(__CUDA_ARCH__)
        return threadIdx.x == 0;
#else
        return true;
#endif
    }
    MG_HD void sync_cta() {
#if defined(__CUDA_ARCH__)
        __syncthreads();
#endif
    }
    int *flag_smem;
    MG_HD int *flags(ArenaHdr *) { return flag_smem; }
    int cnt[MG_N_COUNTERS];
    MG_HD void add_count(const EngineDev &, int kind, long long v) { cnt[kind] += (int)v; }
    // warp-reduced, then one shared-memory add per warp and ONE global atomic per counter per arena-step (the 8 counters
    // are 8 addresses for the whole GPU: a global atomic per warp made them a hot spot)
    int *cnt_smem;                      // [MG_N_COUNTERS], zero between arena-steps
    MG_HD void flush_counts(const EngineDev &E) {
#if defined(__CUDA_ARCH__)
#pragma unroll
        for (int k = 0; k < MG_N_COUNTERS; ++k) {
            int v = cnt[k];
            cnt[k] = 0;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
            if (v && (threadIdx.x & 31) == 0) atomicAdd(&cnt_smem[k], v);
        }
        __syncthreads();
        if (threadIdx.x < MG_N_COUNTERS) {
            const int v = cnt_smem[threadIdx.x];
            cnt_smem[threadIdx.x] = 0;
            if (v) atomicAdd((unsigned long long *)&E.counters[threadIdx.x], (unsigned long long)v);
        }
#endif
    }
    MG_HD int tid() const {
#if defined(__CUDA_ARCH__)
        return threadIdx.x;
#else
        return 0;
#endif
    }
    MG_HD int nth() const {
#if defined(__CUDA_ARCH__)
        return blockDim.x;
#else
        return 1;
#endif
    }
    MG_HD void sync() {
#if defined(__CUDA_ARCH__)
        __syncthreads();
#endif
    }
    template <class P, class Em>
    MG_HD int scan(int n, P pred, Em emit) {
#if defined(__CUDA_ARCH__)
        int running = 0;
        for (int tile = 0; tile < n; tile += blockDim.x) {
            int i = tile + threadIdx.x;
            int p = i < n ? pred(i) : 0;
            int tot;
            int ex = block_excl_scan(p, tot);
            if (p) emit(i, running + ex);
            running += tot;
        }
        return running;
#else
        return 0;
#endif
    }
};

struct GridCtx {
    GroupEnum *enum_smem;
    MG_HD GroupEnum *enums() { return enum_smem; }
    MG_HD bool is_cta_leader() const {
#if defined(__CUDA_ARCH__)
        return threadIdx.x == 0;
#else
        return true;
#endif
    }
    MG_HD void sync_cta() {
#if defined(__CUDA_ARCH__)
        __syncthreads();
#endif
    }
    int *scratch;       // [2][4096]
    int parity;
    MG_HD int *flags(ArenaHdr *hdr) { return hdr->changed; }
    int cnt[MG_N_COUNTERS];
    MG_HD void add_count(const EngineDev &, int kind, long long v) { cnt[kind] += (int)v; }
    // one warp-reduced atomic per counter per warp, once per arena-step
    MG_HD void flush_counts(const EngineDev &E) {
#if defined(__CUDA_ARCH__)
#pragma unroll
        for (int k = 0; k < MG_N_COUNTERS; ++k) {
            int v = cnt[k];
            cnt[k] = 0;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
            if (v && (threadIdx.x & 31) == 0) atomicAdd((unsigned long long *)&E.counters[k], (unsigned long long)v);
        }
#endif
    }
    MG_HD int tid() const {
#if defined(__CUDA_ARCH__)
        return blockIdx.x * blockDim.x + threadIdx.x;
#else
        return 0;
#endif
    }
    MG_HD int nth() const {
#if defined(__CUDA_ARCH__)
        return gridDim.x * blockDim.x;
#else
        return 1;
#endif
    }
    MG_HD void sync() {
#if defined(__CUDA_ARCH__)
        cg::this_grid().sync();
#endif
    }
    template <class P, class Em>
    MG_HD int scan(int n, P pred, Em emit) {
#if defined(__CUDA_ARCH__)
        // contiguous chunk per CTA keeps the emitted order == index order
        const int nb = gridDim.x, bid = blockIdx.x;
        const int L = (n + nb - 1) / nb;
        const int lo = min(n, bid * L), hi = min(n, lo + L);
        int cnt = 0;
        for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) cnt += pred(i);
        int cta_total;
        block_excl_scan(cnt, cta_total);
        int *sc = scratch + (parity & 1) * 4096;
        parity ^= 1;
        if (threadIdx.x == 0) sc[bid] = cta_total;
        cg::this_grid().sync();
        int below = 0, all = 0;
        for (int b = threadIdx.x; b < nb; b += blockDim.x) { int v = sc[b]; all += v; if (b < bid) below += v; }
        int base, total;
        block_excl_scan(below, base);
        block_excl_scan(all, total);
        int running = base;
        for (int tile = lo; tile < hi; tile += blockDim.x) {
            int i = tile + threadIdx.x;
            int p = i < hi ? pred(i) : 0;
            int tot;
            int ex = block_excl_scan(p, tot);
            if (p) emit(i, running + ex);
            running += tot;
        }
        return total;
#else
        return 0;
#endif
    }
};

__device__ __forceinline__ void load_engine(EngineDev *sE, const EngineDev *gE) {
    const int *src = (const int *)gE;
    int *dst = (int *)sE;
    for (int i = threadIdx.x; i < (int)(sizeof(EngineDev) / sizeof(int)); i += blockDim.x) dst[i] = src[i];
    __syncthreads();
}

constexpr int STEP_THREADS = 1024;      // launch bound; the launch picks 256..1024 (step_block_size)
constexpr int GRID_THREADS = 512;       // block size of the cooperative whole-grid team

// bytes of per-arena step scratch (the arrays step_scratch_to_smem() re-homes)
static size_t step_scratch_bytes(int cap_total, int max_body) {
    return (size_t)cap_total * (9 * 4 + 4 * (size_t)max_body) + (((size_t)cap_total + 15) & ~(size_t)15);
}

// Point the scratch arrays of the CTA's private EngineDev copy at dynamic shared memory.  One CTA works on one
// arena at a time, so the scratch needs no per-arena stride (scratch_stride = 0): every dependent load of the
// relaxation / list walks becomes an LDS instead of an L2/HBM round trip.  The shuffle scratch (dead after
// phase_rank_target) shares storage with the mover scratch (first written in phase_attack_apply_starve):
// 41 B/agent => two 2x1000-agent arenas per SM.
__device__ __forceinline__ void step_scratch_to_smem(EngineDev *sE, unsigned char *base) {
    const size_t n = (size_t)sE->cap_total;
    int *p = (int *)base;
    sE->att_rank = p; p += n;  sE->tgt = p; p += n;       sE->in_head = p; p += n;  sE->in_next = p; p += n;
    sE->death = p; p += n;
    sE->mv_nx = p; sE->jv = p; p += n;
    sE->mv_ny = p; sE->sh_head = p; p += n;
    sE->mv_key = (unsigned *)p; sE->sh_next = p; p += n;
    sE->hp_fin = (float *)p; sE->att_agent = p; p += n;
    sE->cl_next = p; sE->sh_first = p; p += n * sE->max_body;
    sE->mv_state = (unsigned char *)p;
    sE->scratch_stride = 0;
}

__global__ void __launch_bounds__(STEP_THREADS) step_kernel_cta(const EngineDev *gE, StepArgs S, int scratch_in_smem) {
    extern __shared__ __align__(16) unsigned char step_smem[];
    __shared__ EngineDev sE;
    load_engine(&sE, gE);
    if (scratch_in_smem) {
        if (threadIdx.x == 0) step_scratch_to_smem(&sE, step_smem);
        __syncthreads();
    }
    __shared__ int relax_flags[3];
    __shared__ int counter_sums[MG_N_COUNTERS];
    __shared__ GroupEnum enum_store[2];
    if (threadIdx.x < MG_N_COUNTERS) counter_sums[threadIdx.x] = 0;
    CtaCtx c;
    c.flag_smem = relax_flags;
    c.cnt_smem = counter_sums;
    c.enum_smem = enum_store;
    for (int k = 0; k < MG_N_COUNTERS; ++k) c.cnt[k] = 0;
    for (int a = blockIdx.x; a < sE.A; a += gridDim.x) run_step(c, sE, S, a);
}

__global__ void __launch_bounds__(STEP_THREADS) step_kernel_grid(const EngineDev *gE, StepArgs S) {
    __shared__ EngineDev sE;
    load_engine(&sE, gE);
    __shared__ GroupEnum enum_store[2];
    GridCtx c;
    c.scratch = sE.team_scratch;
    c.parity = 0;
    c.enum_smem = enum_store;
    for (int k = 0; k < MG_N_COUNTERS; ++k) c.cnt[k] = 0;
    for (int a = 0; a < sE.A; ++a) run_step(c, sE, S, a);
}

__global__ void __launch_bounds__(STEP_THREADS) cull_kernel_cta(const EngineDev *gE, unsigned curmask) {
    __shared__ EngineDev sE;
    load_engine(&sE, gE);
    CtaCtx c;
    c.flag_smem = nullptr;
    c.cnt_smem = nullptr;
    c.enum_smem = nullptr;
    for (int a = blockIdx.x; a < sE.A; a += gridDim.x) run_cull(c, sE, curmask, a);
}

__global__ void __launch_bounds__(STEP_THREADS) cull_kernel_grid(const EngineDev *gE, unsigned curmask) {
    __shared__ EngineDev sE;
    load_engine(&sE, gE);
    GridCtx c;
    c.scratch = sE.team_scratch;
    c.parity = 0;
    c.enum_smem = nullptr;
    for (int a = 0; a < sE.A; ++a) run_cull(c, sE, curmask, a);
}

static const int GRID_MODE_THRESHOLD = 32768;    // agents per arena above which the whole grid teams up

// CTA-per-arena block size: the phases are latency-bound loops over the arena's agents, so with many
// arenas we want many (small) CTAs resident per SM; with few arenas the single CTA should be wide.
static int step_block_size(int sms, int arenas, int max_agents) {
    if (arenas >= 2 * sms) return 256;
    if (max_agents >= 768) return 1024;
    return max_agents >= 384 ? 512 : 256;
}

static int coop_grid(const Ctx *c, const void *kernel) {
    int per_sm = 0;
    CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, GRID_THREADS, 0));
    if (per_sm < 1) mg::fatal("cooperative kernel does not fit on an SM");
    int g = per_sm * c->sms;
    return g > 4096 ? 4096 : g;
}

void launch_step(Ctx *c, const EngineDev *dE, const EngineDev &hE, const StepArgs &S, int max_agents) {
    DeviceGuard guard(c);
    const int g_sms = c->sms;
    if (max_agents > GRID_MODE_THRESHOLD) {
        int grid = coop_grid(c, (const void *)step_kernel_grid);
        StepArgs s = S;
        void *args[] = {(void *)&dE, (void *)&s};
        CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)step_kernel_grid, dim3(grid), dim3(GRID_THREADS), args, 0, c->stream));
        post_launch("step_kernel_grid");
    } else {
        // scratch in shared memory whenever one arena's scratch fits: fewer, wider CTAs (latency per phase drops
        // from HBM/L2 round trips to LDS), and the concurrently active arenas stay L2-resident
        const size_t sbytes = step_scratch_bytes(hE.cap_total, hE.max_body);
        static const int smem_pref = getenv("MAGENT_B200_STEP_SMEM") ? atoi(getenv("MAGENT_B200_STEP_SMEM")) : -1;
        const bool in_smem = sbytes <= 200 * 1024 && smem_pref != 0;
        int threads = step_block_size(g_sms, hE.A, max_agents);
        size_t smem = 0;
        if (in_smem) {
            smem = sbytes;
            // few arenas: one wide CTA each; many arenas: narrower CTAs so that two fit on an SM and overlap
            threads = max_agents >= 768 ? (hE.A > g_sms ? 512 : 1024) : (max_agents >= 384 ? 512 : 256);
            ensure_dynamic_smem(c->device, ATTR_STEP, step_kernel_cta, smem);
        }
        // measurement knob (profiles/scripts): MAGENT_B200_STEP_THREADS=256..1024 overrides the block size choice above
        static const int threads_pref = getenv("MAGENT_B200_STEP_THREADS") ? atoi(getenv("MAGENT_B200_STEP_THREADS")) : 0;
        if (threads_pref >= 32 && threads_pref <= STEP_THREADS) threads = threads_pref & ~31;
        int per_sm = 1;
        CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, step_kernel_cta, threads, smem));
        if (per_sm < 1) per_sm = 1;
        int grid = hE.A < per_sm * g_sms ? hE.A : per_sm * g_sms;
        step_kernel_cta<<<grid, threads, smem, c->stream>>>(dE, S, in_smem ? 1 : 0);
        post_launch("step_kernel_cta");
    }
}

void launch_cull(Ctx *c, const EngineDev *dE, const EngineDev &hE, unsigned curmask, int max_agents) {
    DeviceGuard guard(c);
    const int g_sms = c->sms;
    if (max_agents > GRID_MODE_THRESHOLD) {
        int grid = coop_grid(c, (const void *)cull_kernel_grid);
        void *args[] = {(void *)&dE, (void *)&curmask};
        CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)cull_kernel_grid, dim3(grid), dim3(GRID_THREADS), args, 0, c->stream));
        post_launch("cull_kernel_grid");
    } else {
        int grid = hE.A < 8 * g_sms ? hE.A : 8 * g_sms;
        // measurement knob (profiles/README.md): MAGENT_B200_CULL_THREADS overrides the block size
        static const int cull_pref = getenv("MAGENT_B200_CULL_THREADS") ? atoi(getenv("MAGENT_B200_CULL_THREADS")) : 0;
        // the compaction is a chain of block scans (three barriers per tile of blockDim agents): arenas of ~1000 agents
        // per group run fastest with 512 threads (measured 256 / 512 / 1024: 1.243 / 1.230 / 1.237 ms per whole step)
        int threads = max_agents >= 768 ? 512 : step_block_size(g_sms, hE.A, max_agents);
        if (cull_pref >= 32 && cull_pref <= STEP_THREADS) threads = cull_pref & ~31;
        cull_kernel_cta<<<grid, threads, 0, c->stream>>>(dE, curmask);
        post_launch("cull_kernel_cta");
    }
}

// off[g][0..A] = exclusive prefix of n[g][0..A-1]; one CTA per group
__global__ void __launch_bounds__(1024) offsets_kernel(const EngineDev *gE) {
    const int g = blockIdx.x;
    const int A = gE->A;
    const int *n = gE->n + (size_t)g * A;
    int *off = gE->off + (size_t)g * (A + 1);
    int running = 0;
    for (int tile = 0; tile < A; tile += blockDim.x) {
        int a = tile + threadIdx.x;
        int v = a < A ? n[a] : 0;
        int tot;
        int ex = block_excl_scan(v, tot);
        if (a < A) off[a] = running + ex;
        running += tot;
    }
    if (threadIdx.x == 0) off[A] = running;
}

void launch_offsets(Ctx *c, const EngineDev *dE, const EngineDev &hE) {
    DeviceGuard guard(c);
    offsets_kernel<<<hE.G, 1024, 0, c->stream>>>(dE);
    post_launch("offsets_kernel");
}

// arena of the idx-th agent in the concatenation of group g
__device__ __forceinline__ int locate_arena(const int *off, int A, int idx) {
    int lo = 0, hi = A;                 // invariant: off[lo] <= idx < off[hi]
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (off[mid] <= idx) lo = mid; else hi = mid;
    }
    return lo;
}

// One thread per agent, CTAs dealt per arena (blockIdx says which arena: no search).  `n_total` is the host's count, which
// may still be the one from before the last cull (an upper bound): the device-side offsets decide.
__global__ void __launch_bounds__(256) info_kernel(const EngineDev *gE, unsigned curmask, int kind, int g,
                                                   void *buf, int n_total, int chunks_per_arena) {
    const EngineDev &E = *gE;
    const int *off = E.off + (size_t)g * (E.A + 1);
    const AgentSoA &s = E.grp[g].soa[(curmask >> g) & 1u];
    const int a = blockIdx.x / chunks_per_arena;
    const int i = (blockIdx.x - a * chunks_per_arena) * blockDim.x + threadIdx.x;
    const int o0 = off[a];
    const int o = o0 + i;
    if (i < off[a + 1] - o0 && o < n_total) {
        const long gi = (long)a * E.grp[g].cap + i;
        switch (kind) {
            case INFO_ID: ((int *)buf)[o] = s.id[gi]; break;
            case INFO_POS:                // int[n][2] needs only 4-byte alignment: one 8-byte store where the buffer allows it
                if ((((size_t)buf) & 7) == 0) ((int2 *)buf)[o] = make_int2(s.x[gi], s.y[gi]);
                else { ((int *)buf)[2 * (size_t)o] = s.x[gi]; ((int *)buf)[2 * (size_t)o + 1] = s.y[gi]; }
                break;
            case INFO_ALIVE: ((unsigned char *)buf)[o] = (s.flags[gi] & FLAG_DEAD) ? 0 : 1; break;
            case INFO_REWARD: ((float *)buf)[o] = s.next_reward[gi] + E.hdr[a].grp_reward[g]; break;
            case INFO_HP: ((float *)buf)[o] = s.hp[gi]; break;
            case INFO_ACTION_SCATTER: s.act[gi] = ((const int *)buf)[o]; break;
        }
    }
}

void launch_info(Ctx *c, const EngineDev *dE, const EngineDev &hE, unsigned curmask, int kind, int group, void *buf, int n_total) {
    DeviceGuard guard(c);
    const int cap = hE.grp[group].cap;
    const int threads = cap >= 256 ? 256 : ((cap + 31) & ~31);
    const int cpa = (cap + threads - 1) / threads;
    info_kernel<<<(unsigned)((size_t)hE.A * cpa), threads, 0, c->stream>>>(dE, curmask, kind, group, buf, n_total, cpa);
    post_launch("info_kernel");
}

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

__global__ void __launch_bounds__(256) random_actions_kernel(const EngineDev *gE, unsigned curmask, int g,
                                                             unsigned long long seed, int n_total, int chunks_per_arena) {
    const EngineDev &E = *gE;
    const int *off = E.off + (size_t)g * (E.A + 1);
    const AgentSoA &s = E.grp[g].soa[(curmask >> g) & 1u];
    const unsigned na = (unsigned)E.grp[g].n_action;
    // the device-side step counter rides in the seed: a replayed CUDA graph (same kernel arguments) still draws fresh actions
    seed += (unsigned long long)E.counters[CNT_STEPS] * 0xA24BAED4963EE407ull;
    const int a = blockIdx.x / chunks_per_arena;
    const int i = (blockIdx.x - a * chunks_per_arena) * blockDim.x + threadIdx.x;
    const int o0 = off[a];
    const int o = o0 + i;
    if (i < off[a + 1] - o0 && o < n_total)
        s.act[(long)a * E.grp[g].cap + i] = (int)((splitmix64(seed ^ ((unsigned long long)o * 0xD1342543DE82EF95ull)) >> 33) % na);
}

void launch_random_actions(Ctx *c, const EngineDev *dE, const EngineDev &hE, unsigned curmask, int group,
                           unsigned long long seed, int n_total) {
    DeviceGuard guard(c);
    const int cap = hE.grp[group].cap;
    const int threads = cap >= 256 ? 256 : ((cap + 31) & ~31);
    const int cpa = (cap + threads - 1) / threads;
    random_actions_kernel<<<(unsigned)((size_t)hE.A * cpa), threads, 0, c->stream>>>(dE, curmask, group, seed, n_total, cpa);
    post_launch("random_actions_kernel");
}

// ------------------------------------------------------------------------------------------------
// obs_prepare: the minimap of one observation state (GridWorld.cc:328-357): per (arena, group) the number of agents in
// every coarse cell of the OBSERVER's view-sized grid, divided by the group's size.  Dead-but-unculled agents count,
// absorbed ones do not when the observer's type can absorb (:343-347).  (The hp_norm plane the render also needs is
// kept current by the step kernels, step_phases.h hpn_set.)
//
// minimap_small_kernel: one CTA per (arena, group) when a group of an arena is at most a few thousand agents --
// histogram in shared memory, normalised row written directly.  Larger groups: obs_prepare_kernel histograms chunks of
// 4096 agents into global counters, minimap_norm_kernel normalises.
__global__ void __launch_bounds__(256) minimap_small_kernel(const EngineDev *gE, unsigned curmask, int og, float *mm_val, int stride) {
    extern __shared__ int hist[];
    __shared__ int counted_s;
    const EngineDev &E = *gE;
    const int ag = blockIdx.x;               // a * G + j
    const int a = ag / E.G, j = ag - a * E.G;
    const int vw = E.grp[og].view_w, vh = E.grp[og].view_h, cells = vw * vh;
    const int n = E.n[j * E.A + a];
    for (int k = threadIdx.x; k < cells; k += blockDim.x) hist[k] = 0;
    if (threadIdx.x == 0) counted_s = 0;
    __syncthreads();
    const GroupDev &G = E.grp[j];
    const AgentSoA &s = G.soa[(curmask >> j) & 1u];
    const int scale_h = (E.H + vh - 1) / vh, scale_w = (E.W + vw - 1) / vw;
    const bool skip_absorbed = E.grp[og].can_absorb != 0;
    int counted = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const long gi = (long)a * G.cap + i;
        if (skip_absorbed && (s.flags[gi] & FLAG_ABSORBED)) continue;
        atomicAdd(&hist[(s.y[gi] / scale_h) * vw + s.x[gi] / scale_w], 1);
        ++counted;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) counted += __shfl_xor_sync(0xffffffffu, counted, d);
    if ((threadIdx.x & 31) == 0 && counted) atomicAdd(&counted_s, counted);
    __syncthreads();
    const int tot = counted_s;
    float *out = mm_val + (size_t)a * stride + (size_t)j * cells;
    // an empty (or fully absorbed) group is 0/0 in the reference: x86 divss yields the default quiet NaN 0xFFC00000
    for (int k = threadIdx.x; k < cells; k += blockDim.x)
        out[k] = tot ? (float)hist[k] / (float)tot : __int_as_float((int)0xFFC00000u);
}

__global__ void __launch_bounds__(256) obs_prepare_kernel(const EngineDev *gE, unsigned curmask, int og, int chunk) {
    extern __shared__ int hist[];
    const EngineDev &E = *gE;
    const int ag = blockIdx.y;               // a * G + j
    const int a = ag / E.G, j = ag - a * E.G;
    const int vw = E.grp[og].view_w, vh = E.grp[og].view_h, cells = vw * vh;
    const int n = E.n[j * E.A + a];
    const int lo = blockIdx.x * chunk;
    if (lo >= n) return;
    const int hi = min(n, lo + chunk);
    for (int k = threadIdx.x; k < cells; k += blockDim.x) hist[k] = 0;
    __syncthreads();
    const GroupDev &G = E.grp[j];
    const AgentSoA &s = G.soa[(curmask >> j) & 1u];
    const int scale_h = (E.H + vh - 1) / vh, scale_w = (E.W + vw - 1) / vw;
    const bool skip_absorbed = E.grp[og].can_absorb != 0;     // GridWorld.cc:343-347 (the OBSERVER's type decides)
    int counted = 0;
    for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        long gi = (long)a * G.cap + i;
        if (skip_absorbed && (s.flags[gi] & FLAG_ABSORBED)) continue;
        atomicAdd(&hist[(s.y[gi] / scale_h) * vw + s.x[gi] / scale_w], 1);
        ++counted;
    }
    if (counted) atomicAdd(&E.mm_total[ag], counted);
    __syncthreads();
    int *out = E.mm_count + (size_t)ag * cells;
    for (int k = threadIdx.x; k < cells; k += blockDim.x)
        if (hist[k]) atomicAdd(&out[k], hist[k]);
}

// normalised minimap, one padded row per arena: mm[a * stride + j * cells + cell]  (stride % 4 == 0 so that a row is a
// legal TMA bulk-copy source)
__global__ void __launch_bounds__(256) minimap_norm_kernel(const EngineDev *gE, int og, float *mm_val, int total, int stride) {
    const EngineDev &E = *gE;
    const int cells = E.grp[og].view_w * E.grp[og].view_h;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < total; k += gridDim.x * blockDim.x) {
        int ag = k / cells;
        // GridWorld.cc:350-357 (total_ct).  An empty (or fully absorbed) group is 0/0 in the reference: x86 divss
        // yields the default quiet NaN 0xFFC00000 whereas the GPU would give 0x7FFFFFFF, so emit the x86 payload.
        const int tot = E.mm_total[ag];
        const int a = ag / E.G;
        mm_val[(size_t)a * stride + (k - a * E.G * cells)] = tot ? (float)E.mm_count[k] / (float)tot : __int_as_float((int)0xFFC00000u);
    }
}

void launch_obs_prepare(Ctx *c, const EngineDev *dE, const EngineDev &hE, unsigned curmask, int og, float *mm_val) {
    if (!mm_val) return;                     // no minimap: nothing to prepare (the planes are kept current by the step)
    DeviceGuard guard(c);
    const int g_sms = c->sms;
    const int cells = hE.grp[og].view_w * hE.grp[og].view_h;
    const int total = hE.A * hE.G * cells;
    int cap_max = 0;
    for (int g = 0; g < hE.G; ++g) cap_max = cap_max > hE.grp[g].cap ? cap_max : hE.grp[g].cap;
    c->mm_stride = (hE.G * cells + 3) & ~3;
    const size_t need = (size_t)hE.A * c->mm_stride;
    if (need > c->mm_pad_n) {
        no_capture(c, "growing the minimap buffer");
        if (c->mm_pad) { CUDA_CHECK(cudaStreamSynchronize(c->stream)); CUDA_CHECK(cudaStreamSynchronize(c->copy)); cudaFree(c->mm_pad); }
        CUDA_CHECK(cudaMalloc(&c->mm_pad, need * sizeof(float)));
        CUDA_CHECK(cudaMemsetAsync(c->mm_pad, 0, need * sizeof(float), c->stream));
        c->mm_pad_n = need;
    }
    if (cap_max <= 8192 && (size_t)cells * sizeof(int) <= 48 * 1024) {
        minimap_small_kernel<<<hE.A * hE.G, 256, cells * sizeof(int), c->stream>>>(dE, curmask, og, c->mm_pad, c->mm_stride);
        post_launch("minimap_small_kernel");
        return;
    }
    CUDA_CHECK(cudaMemsetAsync(hE.mm_count, 0, (size_t)total * 4, c->stream));
    CUDA_CHECK(cudaMemsetAsync(hE.mm_total, 0, (size_t)hE.A * hE.G * 4, c->stream));
    const int chunk = 4096;
    dim3 grid((cap_max + chunk - 1) / chunk, hE.A * hE.G);
    obs_prepare_kernel<<<grid, 256, cells * sizeof(int), c->stream>>>(dE, curmask, og, chunk);
    post_launch("obs_prepare_kernel");
    int g2 = (total + 255) / 256;
    if (g2 > 8 * g_sms) g2 = 8 * g_sms;
    minimap_norm_kernel<<<g2, 256, 0, c->stream>>>(dE, og, c->mm_pad, total, c->mm_stride);
    post_launch("minimap_norm_kernel");
}

// ------------------------------------------------------------------------------------------------
// obs_render_kernel: the observation gather (GridWorld.cc:292-401 + Map::extract_view Map.cc:129-207).
//
// The kernel is a stream of 4.7 KB records (battle) whose content is ~97 % zeros + the dense minimap channels +
// a handful of values gathered from the map.  Two ceilings matter on B200 (profiles/README.md): the TMA
// bulk-store stream itself (6.3 TB/s measured for this tile size) and the L2 slice throughput (~12 TB/s summed
// over reads and writes) -- so every byte the kernel READS through L2 competes with the bytes it writes:
//   * tile = TA (4) consecutive agents of the ABI concatenation = ONE 128-thread CTA, one warp per agent, one
//     shared-memory tile (18.9 KB for battle), 8 CTAs = 32 warps per SM, tiles dealt round-robin so the whole
//     grid works inside a window of a few arenas (their planes / minimaps stay L1/L2-hot);
//   * the map is gathered from a ONE-BYTE kind plane (0 empty / 1 wall / 2+group; a view row is one 32-byte
//     sector) and only occupied cells (~5 %) take a second, dependent load from the hp_norm plane;
//   * the tile is composed entirely on the SM: each warp zero-fills its own record, copies the arena's
//     normalised minimap (G x cells floats, L1-resident) into the minimap channels, adds the self marker and
//     scatters the non-zero map values (n_channel-word stride => conflict-free for odd channel counts) --
//     no template tile is read through L2;
//   * the tile leaves the SM as ONE TMA bulk STORE (cp.async.bulk.global.shared::cta, SASS UBLKCP).  A tile's
//     byte range in the output is contiguous and 16-byte aligned because TA * sizeof(T) % 16 == 0.
// Algorithmic traffic per agent: sizeof(T)*(view_h*view_w*n_channel + feature) bytes written, plus one compulsory
// read of the occupancy plane per arena (DESIGN.md section 6).  No tensor cores: there is no contraction here.
#ifndef OBS_TA_N
#define OBS_TA_N 4
#endif
#ifndef OBS_ABLATE
#define OBS_ABLATE 0                 // profiling experiments only (profiles/README.md): 1 no plane gather, 2 no tile
#endif                               // init (zero + minimap), 4 no feature rows, 8 no bulk store -- results are WRONG

// output element type of the observation: float = the reference ABI (env_get_observation); __half = the compact
// hand-off format of magent_b200_get_observation_f16 (each value is the f32 value rounded to nearest-even).
// TA = agents per tile = warps per CTA; TA * sizeof(T) % 16 == 0 keeps every tile's byte range 16-byte aligned.
template <typename T> struct ObsOut;
template <> struct ObsOut<float> {
    static constexpr int TA = OBS_TA_N;
    static __device__ __forceinline__ float cv(float v) { return v; }
};
template <> struct ObsOut<__half> {
    static constexpr int TA = 2 * OBS_TA_N;
    static __device__ __forceinline__ __half cv(float v) {
        if (v != v) {                    // keep sign and top payload bits like a software f32->f16 cast does (numpy astype)
            const unsigned u = __float_as_uint(v);
            unsigned short r = (unsigned short)(0x7c00u + ((u & 0x7fffffu) >> 13));
            if (r == 0x7c00u) ++r;
            return __ushort_as_half((unsigned short)(r | ((u >> 16) & 0x8000u)));
        }
        return __float2half_rn(v);
    }
};

struct ObsParams {
    int A, W, H, G, C;
    int vw, vh, cells, rec, F;
    int ox, oy;                      // map offset of view cell (0,0) from the agent position
    int scale_w, scale_h, minimap;
    int cap, embedding, n_action, n_total;
    const unsigned char *mask;
    const int *off;
    const unsigned char *kind_plane; // [A][kplane] padded: 0 empty / 1 wall / 2+group (EngineDev::kind)
    const float *hpn_plane;          // [A][kplane] padded: hp / max_hp of the occupant (EngineDev::hpn)
    int kpad, kw;
    long kplane;
    int chunk;                       // consecutive tiles per CTA visit (<= OBS_CHUNK)
    int turn, body_w, body_l;        // turn_mode: 4 view LUTs (one per heading), the heading rides in the header
    const unsigned char *dir;
    const int *x, *y, *id, *act;
    const float *last_reward;
    const float *mm;                 // [A][mm_stride] normalised minimap rows (G x cells floats each), or nullptr
    int mm_stride;
    const int4 *hdr;                 // [n_total] per-agent header in ABI order (obs_headers_kernel)
    void *view, *feature;            // element type = the kernel's template argument
    int mm_ch[MG_MAX_GROUPS];        // observation channel of group j's minimap
    int grp_ch[MG_MAX_GROUPS];       // observation channel ('has'; hp is +1) of group j
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// pre-pass, one thread per observer, CTAs dealt per arena (no search for the arena: blockIdx says it):
//   * header h = {x, y, arena, self minimap cell | heading << 16}: everything the render kernel needs about the observer itself, so
//     that its only dependent loads are kind plane -> hp_norm plane;
//   * the complete non-spatial feature row (GridWorld.cc:386-396): id bits LSB first, one-hot last action, last
//     reward, and x/W, y/H with the minimap.  A fresh agent's last_action == n_action ("dangerous", GridWorld.h:140)
//     lands on the reward slot and is overwritten by it -- here the reward simply wins.  The rows of a CTA's observers are
//     one contiguous block of the output: composed in shared memory (zero fill, then every thread its own handful of
//     non-zeros), written out with coalesced stores.
template <typename T>
__global__ void __launch_bounds__(256) obs_headers_kernel(ObsParams P, int4 *hdr, int chunks_per_arena) {
    extern __shared__ __align__(16) unsigned char hdr_smem[];
    T *rows = (T *)hdr_smem;                                   // [blockDim.x][F]
    const int a = blockIdx.x / chunks_per_arena;
    const int i0 = (blockIdx.x - a * chunks_per_arena) * blockDim.x;
    const int o0 = P.off[a], n_a = P.off[a + 1] - o0;
    if (i0 >= n_a) return;
    int cnt = min((int)blockDim.x, n_a - i0);
    cnt = min(cnt, P.n_total - (o0 + i0));                     // never beyond the caller's buffers
    if (cnt <= 0) return;
    const int total = cnt * P.F;
    for (int q = threadIdx.x; q < total; q += blockDim.x) rows[q] = ObsOut<T>::cv(0.0f);
    __syncthreads();
    if ((int)threadIdx.x < cnt) {
        const int i = i0 + threadIdx.x;
        const long gi = (long)a * P.cap + i;
        const int x = P.x[gi], y = P.y[gi];
        const int self_cell = P.minimap ? (y / P.scale_h) * P.vw + x / P.scale_w : -1;  // GridWorld.cc:372-373
        const int heading = P.turn ? (int)P.dir[gi] : 0;
        hdr[o0 + i] = make_int4(x, y, a, (self_cell & 0xffff) | (heading << 16));
        T *f = rows + (size_t)threadIdx.x * P.F;
        unsigned id = (unsigned)P.id[gi];
        const int nbits = min(P.embedding, 31);
        id &= nbits >= 32 ? 0xffffffffu : ((1u << nbits) - 1u);
        while (id) {                                           // embedding: the set bits of the id, LSB first (GridWorld.h:155-164)
            const int bit = __ffs(id) - 1;
            f[bit] = ObsOut<T>::cv(1.0f);
            id &= id - 1;
        }
        T *g = f + P.embedding;
        const int act = P.act[gi];
        if (act >= 0 && act < P.n_action) g[act] = ObsOut<T>::cv(1.0f);
        g[P.n_action] = ObsOut<T>::cv(P.last_reward[gi]);       // also overwrites the "dangerous" fresh-agent one-hot slot
        if (P.minimap) {
            g[P.n_action + 1] = ObsOut<T>::cv((float)x / (float)P.W);               // GridWorld.cc:394-395
            g[P.n_action + 2] = ObsOut<T>::cv((float)y / (float)P.H);
        }
    }
    __syncthreads();
    T *out = (T *)P.feature + (size_t)(o0 + i0) * P.F;
    if (sizeof(T) == 4 && ((((size_t)out) & 15) == 0)) {       // 16-byte body, scalar tail
        const int v4 = total >> 2;
        for (int q = threadIdx.x; q < v4; q += blockDim.x) ((float4 *)out)[q] = ((const float4 *)rows)[q];
        for (int q = (v4 << 2) + threadIdx.x; q < total; q += blockDim.x) out[q] = rows[q];
    } else {
        for (int q = threadIdx.x; q < total; q += blockDim.x) out[q] = rows[q];
    }
}

#ifndef OBS_MIN_CTAS
#define OBS_MIN_CTAS 8
#endif
#ifndef OBS_CHUNK
#define OBS_CHUNK 4                  // consecutive tiles a CTA renders before it jumps ahead by grid * OBS_CHUNK tiles
#endif
// NIT = view cells per lane held in registers (NIT * 32 >= in-range cells of the view whenever that is <= 256;
// larger views take the unpipelined tail loop).
//
// The tile buffer is PERSISTENT: consecutive tiles of a CTA belong to the same arena (blocked tile assignment), so
// the zeros and the arena's minimap channels already in the buffer are still right for the next tile.  After the
// bulk store has read the buffer, each warp only UNDOES the few cells it marked for the previous observer (kinds
// remembered in one packed register) and restores the self-marker cell, then marks the new observer's cells.  A
// warp rebuilds its record (zero fill + minimap rows from L2) only when its observer's arena changes -- once or
// twice per launch.
template <typename T, int NIT, bool TURN>
__global__ void __launch_bounds__(32 * ObsOut<T>::TA, OBS_MIN_CTAS * OBS_TA_N / ObsOut<T>::TA)
obs_render_kernel(const __grid_constant__ ObsParams P) {
    const int n_total = min(P.n_total, __ldg(P.off + P.A));   // the host may hold pre-cull counts (upper bounds)
    constexpr int OBS_TA = ObsOut<T>::TA;
    constexpr int OBS_THREADS = 32 * OBS_TA;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T *buf = (T *)smem_raw;                                   // one tile: OBS_TA records
    // in-range view cells only: lut[k] = {word offset of the cell inside a record, offset of the map cell in the
    // padded planes relative to the observer's own cell}
    int2 *lut = (int2 *)(buf + OBS_TA * P.rec);
    __shared__ int n_in_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    const int lut_stride = (P.cells + 1) & ~1;
    if (warp == 0) {                                          // compact the view mask (Range.h:104-189)
        int k = 0;                                            // order-preserving: ballot prefix per 32 cells
        for (int base = 0; base < P.cells; base += 32) {
            const int cell = base + lane;
            const bool in = cell < P.cells && P.mask[cell];
            const unsigned bal = __ballot_sync(0xffffffffu, in);
            if (in) {
                const int vy = cell / P.vw, vx = cell - vy * P.vw;
                const int q = k + __popc(bal & ((1u << lane) - 1u));
                if (!TURN) lut[q] = make_int2(cell * P.C, (P.oy + vy) * P.kw + P.ox + vx);
                else {
                    // the window is laid out in the observer's frame: one LUT per heading (Map.cc:140-146, 515-560)
                    for (int d = 0; d < 4; ++d) {
                        int rx = 0, ry = 0, dx, dy;                     // save_to_real
                        if (d == DIR_SOUTH) { rx = P.body_w - 1; ry = P.body_l - 1; }
                        else if (d == DIR_WEST) ry = P.body_w - 1;
                        else if (d == DIR_EAST) rx = P.body_l - 1;
                        const int ex = P.ox + vx, ey = P.oy + vy;       // rela_to_abs
                        if (d == DIR_NORTH) { dx = ex; dy = ey; }
                        else if (d == DIR_SOUTH) { dx = -ex; dy = -ey; }
                        else if (d == DIR_WEST) { dx = ey; dy = -ex; }
                        else { dx = -ey; dy = ex; }
                        lut[d * lut_stride + q] = make_int2(cell * P.C, (ry + dy) * P.kw + rx + dx);
                    }
                }
            }
            k += __popc(bal);
        }
        if (lane == 0) n_in_s = k;
    }
    __syncthreads();
    const int n_in = n_in_s;
    const int n_tiles = (n_total + OBS_TA - 1) / OBS_TA;
    // this lane's slice of the view LUT never changes: small views keep it in registers, large ones re-read smem
    constexpr bool LUT_REGS = NIT <= 4 && !TURN;
    int2 lreg[LUT_REGS ? NIT : 1];
    if (LUT_REGS) {
#pragma unroll
        for (int it = 0; it < (LUT_REGS ? NIT : 1); ++it) lreg[it] = it * 32 + lane < n_in ? lut[it * 32 + lane] : make_int2(-1, 0);
    }
    // hd = heading of the observer (always 0 without turn_mode)
    auto lutv = [&](int it, int hd) -> int2 {
        if (TURN) return it * 32 + lane < n_in ? lut[hd * lut_stride + it * 32 + lane] : make_int2(-1, 0);
        return LUT_REGS ? lreg[LUT_REGS ? it : 0] : (it * 32 + lane < n_in ? lut[it * 32 + lane] : make_int2(-1, 0));
    };
    // position of an observer's own cell in the padded planes (header word h = {x, y, arena, self cell | heading << 16})
    auto plane_base = [&](const int4 &h) -> long { return h.z * P.kplane + (long)(h.y + P.kpad) * P.kw + h.x + P.kpad; };

    // issue the kind-plane loads of one observer; the pad makes every view cell addressable
    auto load_kinds = [&](const int4 &h, bool on, int (&kd)[NIT]) {
        const unsigned char *kp = P.kind_plane + plane_base(h);
        const int hd = TURN ? (h.w >> 16) & 3 : 0;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int2 l = lutv(it, hd);
            kd[it] = (on && l.x >= 0 && !(OBS_ABLATE & 1)) ? __ldg(kp + l.y) : 0;
        }
    };
    // write (on = true) or erase what an occupied view cell shows: wall / food flag, or a group's {1, hp / max_hp}
    // channel of every kind, one byte each in two registers (byte k of chpack = channel of group k): no constant-bank
    // lookup and no branch ladder per marked cell
    unsigned long long chpack = 0ull;
#pragma unroll
    for (int j = 0; j < MG_MAX_GROUPS; ++j) chpack |= (unsigned long long)(P.grp_ch[j] & 0xff) << (8 * j);
    auto mark = [&](T *px, int t, float hp, bool on) {
        const bool agent = kind_is_agent(t);
        const int ch = agent ? (int)((chpack >> (8 * kind_group(t))) & 0xffull) : (t == KIND_FOOD ? 1 : 0);
        px[ch] = ObsOut<T>::cv(on ? 1.0f : 0.0f);                          // wall / food flag or the group's 'has' channel
        if (agent) px[ch + 1] = ObsOut<T>::cv(on ? hp : 0.0f);             // hp / max_hp (Map.cc:197)
    };

    // tile assignment: chunks of OBS_CHUNK consecutive tiles, dealt round-robin over the CTAs.  Inside a chunk the
    // arena (almost) never changes, so the persistent tile needs no rebuild; across the grid all CTAs write inside one
    // window of grid * OBS_CHUNK tiles (~90 MB), which keeps the output stream inside the TLB reach (blocked
    // assignment -- one 4 MB region per CTA -- measured 20 % slower) and the planes of ~20 arenas L2-hot.
    // Software pipeline: while tile i is composed, the kind loads of tile i+1 and the header load of tile i+2 fly.
    const int chunk = P.chunk;                 // 1 when there are too few tiles to keep every CTA busy with longer chunks
    const int chunk_jump = ((int)gridDim.x - 1) * chunk;
    auto next_tile = [&](int t) -> int { return ((t + 1) % chunk) ? t + 1 : t + 1 + chunk_jump; };
    int tile = blockIdx.x * chunk;
    int tile1 = next_tile(tile), tile2 = next_tile(tile1);
    const int tile_end = n_tiles;
    const int4 zero4 = make_int4(0, 0, 0, 0);
    int4 hA = zero4, hA1 = zero4;             // headers of tile i and i+1
    int kind[NIT];
    // what this warp's record currently shows: the arena whose minimap rows it holds (-1: garbage), the previous
    // observer's heading, marked kinds (packed bytes; > 4 * 32 cells per lane never happens with NIT <= 8) and
    // self-marker cell with its unmarked minimap value per group lane
    int rec_arena = -1, prev_hd = 0, prev_self = -1;
    unsigned prev_kinds[(NIT + 3) / 4];
#pragma unroll
    for (int q = 0; q < (NIT + 3) / 4; ++q) prev_kinds[q] = 0u;
    float self_orig = 0.0f;
    bool prev_tail = false;                    // the previous observer had cells beyond NIT * 32 marked (large views)
    {
        const int o0 = tile * OBS_TA + warp, o1 = tile1 * OBS_TA + warp;
        const bool on0 = tile < tile_end && o0 < n_total;
        if (on0) hA = P.hdr[o0];
        if (o1 < n_total) hA1 = P.hdr[o1];
        load_kinds(hA, on0, kind);
    }
    for (; tile < tile_end; tile = tile1, tile1 = tile2, tile2 = next_tile(tile2)) {
        const int t0 = tile * OBS_TA;
        const int cnt = min(OBS_TA, n_total - t0);
        const bool active = warp < cnt;
        const int a = hA.z;
        // occupied cells only: the occupant's hp / max_hp (the kinds were loaded one tile ago)
        const float *hpnp = P.hpn_plane + plane_base(hA);
        const int hd = TURN ? (hA.w >> 16) & 3 : 0;
        float thp[NIT];
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            thp[it] = 0.0f;
            if (kind_is_agent(kind[it])) thp[it] = (kind[it] & KIND_FULL) ? 1.0f : __ldg(hpnp + lutv(it, hd).y);   // full hp: no load
        }
        // next tile's kinds, next-next tile's header
        int kind1[NIT];
        const long o1 = (long)tile1 * OBS_TA + warp;
        load_kinds(hA1, o1 < n_total, kind1);
        int4 hA2 = zero4;
        {
            const long o2 = (long)tile2 * OBS_TA + warp;
            if (o2 < n_total) hA2 = P.hdr[o2];
        }
        // the previous tile's bulk store must have finished READING the buffer before it is touched
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncthreads();
        if (active && !(OBS_ABLATE & 2)) {
            T *dst = buf + warp * P.rec;
            const int self = (int)(short)(hA.w & 0xffff);
            if (a != rec_arena) {
                // (re)build the record: zeros + the arena's minimap rows (GridWorld.cc:374-383), element stores because
                // f16 records share 32-bit words with their neighbours
                if (sizeof(T) == 4) {                              // 16-byte body, scalar head / tail
                    float *w = (float *)dst;
                    const int n = P.rec;
                    const int head = min(n, (int)((4u - ((unsigned)(warp * P.rec) & 3u)) & 3u));
                    const int body = (n - head) >> 2;
                    if (lane < head) w[lane] = 0.0f;
                    float4 *w4 = (float4 *)(w + head);
                    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    for (int q = lane; q < body; q += 32) w4[q] = z;
                    const int tail0 = head + (body << 2);
                    if (tail0 + lane < n) w[tail0 + lane] = 0.0f;
                } else {
                    for (int q = lane; q < P.rec; q += 32) dst[q] = ObsOut<T>::cv(0.0f);
                }
                __syncwarp();
                if (P.minimap) {
                    const float *rows = P.mm + (size_t)a * P.mm_stride;
                    for (int j = 0; j < P.G; ++j) {
                        T *d = dst + P.mm_ch[j];
                        for (int cell = lane; cell < P.cells; cell += 32) d[cell * P.C] = ObsOut<T>::cv(__ldg(rows + j * P.cells + cell));
                    }
                }
                rec_arena = a;
                __syncwarp();
            } else {
                // undo the previous observer: its marked cells and its self marker
#pragma unroll
                for (int it = 0; it < NIT; ++it) {
                    const int t = (prev_kinds[it >> 2] >> ((it & 3) * 8)) & 0xff;
                    if (t != 0) mark(dst + lutv(it, prev_hd).x, t, 0.0f, false);
                }
                if (prev_tail) {                                                   // large views: recompute which tail cells were marked
                    for (int k = NIT * 32 + lane; k < n_in; k += 32) {
                        T *px = dst + lut[(TURN ? prev_hd * lut_stride : 0) + k].x;
                        for (int ch = 0; ch < P.C; ++ch) {
                            bool mm_ch = false;
                            for (int j = 0; j < P.G; ++j) mm_ch |= P.minimap && ch == P.mm_ch[j];
                            if (!mm_ch) px[ch] = ObsOut<T>::cv(0.0f);
                        }
                    }
                }
                if (P.minimap && lane < P.G && prev_self >= 0) dst[prev_self * P.C + P.mm_ch[lane]] = ObsOut<T>::cv(self_orig);
                __syncwarp();
            }
            // the new observer: self marker (+1 at its coarse cell; NaN + 1 keeps the x86 payload in the reference)
            if (P.minimap && lane < P.G) {
                const float v = __ldg(P.mm + (size_t)a * P.mm_stride + lane * P.cells + self);
                self_orig = v;
                if (v == v) dst[self * P.C + P.mm_ch[lane]] = ObsOut<T>::cv(v + 1.0f);
            }
            prev_self = self;
            prev_hd = hd;
#pragma unroll
            for (int q = 0; q < (NIT + 3) / 4; ++q) prev_kinds[q] = 0u;
#pragma unroll
            for (int it = 0; it < NIT; ++it) {
                const int t = kind[it];
                prev_kinds[it >> 2] |= (unsigned)t << ((it & 3) * 8);
                if (t != 0) mark(dst + lutv(it, hd).x, t, thp[it], true);
            }
            prev_tail = false;
            const unsigned char *kindp = P.kind_plane + plane_base(hA);
            for (int k = NIT * 32 + lane; k < n_in; k += 32) {                          // views with > NIT * 32 in-range cells
                const int2 l = lut[(TURN ? hd * lut_stride : 0) + k];
                const int t = __ldg(kindp + l.y);
                if (t != 0) { mark(dst + l.x, t, kind_is_agent(t) ? ((t & KIND_FULL) ? 1.0f : __ldg(hpnp + l.y)) : 0.0f, true); }
                prev_tail = true;
            }
        }
        // make the generic-proxy writes visible to the async proxy, then one thread fires the bulk store
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        T *gout = (T *)P.view + (size_t)t0 * P.rec;
        const unsigned bytes = (unsigned)cnt * (unsigned)P.rec * (unsigned)sizeof(T);
        if ((bytes & 15u) == 0 && (((size_t)gout) & 15) == 0) {
            if (threadIdx.x == 0 && !(OBS_ABLATE & 8)) {
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                             :: "l"(gout), "r"(smem_u32(buf)), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        } else {                                   // ragged last tile / unaligned caller buffer
            for (int q = threadIdx.x; q < cnt * P.rec; q += OBS_THREADS) gout[q] = buf[q];
            __syncthreads();
        }
        // rotate the pipeline
        hA = hA1; hA1 = hA2;
#pragma unroll
        for (int it = 0; it < NIT; ++it) kind[it] = kind1[it];
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

template <typename T, int NIT, bool TURN>
static void launch_obs_typed(Ctx *c, int cfg_slot, const EngineDev &hE, ObsParams &P, int n_total,
                             bool with_headers = true, bool headers_only = false) {
    const int g_sms = c->sms;
    constexpr int TA = ObsOut<T>::TA;
    constexpr int THREADS = 32 * TA;
    const size_t tile_bytes = (size_t)TA * P.rec * sizeof(T);            // multiple of 16 by construction of TA
    const size_t smem = tile_bytes + (size_t)(P.turn ? 4 : 1) * ((P.cells + 1) & ~1) * sizeof(int2);
    if (smem > 227 * 1024) mg::fatal("observation record too large for the render kernel (%zu bytes of shared memory)", smem);
    const int tiles = (n_total + TA - 1) / TA;
    if ((size_t)n_total > c->obs_hdr_n) {                                // scratch owned by the context: per-agent headers
        no_capture(c, "growing the observation header table");
        if (c->obs_hdr) { CUDA_CHECK(cudaStreamSynchronize(c->stream)); cudaFree(c->obs_hdr); }
        c->obs_hdr_n = (size_t)n_total + n_total / 4 + 64;
        CUDA_CHECK(cudaMalloc(&c->obs_hdr, c->obs_hdr_n * sizeof(int4)));
    }
    P.hdr = c->obs_hdr;
    if (with_headers) {
        int threads = 256;                                               // as many observers per CTA as fit 48 KB of rows
        while (threads > 32 && (size_t)threads * P.F * sizeof(T) > 48 * 1024) threads >>= 1;
        const size_t hsm = (size_t)threads * P.F * sizeof(T);
        if (hsm > 48 * 1024) mg::fatal("feature row too long for the header kernel (%d elements)", P.F);
        const int cpa = (P.cap + threads - 1) / threads;
        obs_headers_kernel<T><<<(unsigned)((size_t)P.A * cpa), threads, hsm, c->stream>>>(P, c->obs_hdr, cpa);
        post_launch("obs_headers_kernel");
    }
    if (headers_only) return;
    Ctx::ObsCfg &cfg = c->obs_cfg[cfg_slot];
    ensure_dynamic_smem(c->device, ATTR_OBS0 + cfg_slot, obs_render_kernel<T, NIT, TURN>, smem);
    if (smem != cfg.smem) {
        CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cfg.ctas_per_sm, obs_render_kernel<T, NIT, TURN>, THREADS, smem));
        if (cfg.ctas_per_sm < 1) cfg.ctas_per_sm = 1;
        cfg.smem = smem;
    }
    const int ctas_per_sm = cfg.ctas_per_sm;
    const int grid = tiles < ctas_per_sm * g_sms ? tiles : ctas_per_sm * g_sms;
    P.chunk = tiles / (ctas_per_sm * g_sms);                            // keep every CTA busy before lengthening chunks
    if (P.chunk < 1) P.chunk = 1;
    const int max_chunk = sizeof(T) == 2 ? 2 * OBS_CHUNK : OBS_CHUNK;   // f16 tiles are rebuilt for 8 observers at once: longer chunks pay (measured)
    if (P.chunk > max_chunk) P.chunk = max_chunk;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    const bool timed = c->profile && !c->capturing;
    if (timed) { profile_pair(c, &e0, &e1); CUDA_CHECK(cudaEventRecord(e0, c->stream)); }
    obs_render_kernel<T, NIT, TURN><<<grid, THREADS, smem, c->stream>>>(P);
    post_launch("obs_render_kernel");
    if (timed) CUDA_CHECK(cudaEventRecord(e1, c->stream));
}

static void fill_obs_params(Ctx *c, const EngineDev &hE, const ObsArgs &O, const float *mm_val, int n_total, ObsParams &P) {
    const int g = O.group;
    const GroupDev &G = hE.grp[g];
    memset(&P, 0, sizeof P);
    P.A = hE.A; P.W = hE.W; P.H = hE.H; P.G = hE.G; P.C = hE.n_channel;
    P.vw = G.view_w; P.vh = G.view_h; P.cells = G.view_w * G.view_h; P.rec = P.cells * P.C; P.F = G.feature_size;
    P.ox = G.view_xoff + G.view_x1; P.oy = G.view_yoff + G.view_y1;
    P.scale_w = (hE.W + G.view_w - 1) / G.view_w; P.scale_h = (hE.H + G.view_h - 1) / G.view_h;
    P.minimap = mm_val != nullptr;
    P.cap = G.cap; P.embedding = hE.embedding_size; P.n_action = G.n_action; P.n_total = n_total;
    P.mask = G.view_mask;
    P.off = hE.off + (size_t)g * (hE.A + 1);
    P.kind_plane = hE.kind; P.hpn_plane = hE.hpn; P.kpad = hE.kpad; P.kw = hE.kw; P.kplane = hE.kplane;
    const AgentSoA &s = G.soa[(O.curmask >> g) & 1u];
    P.x = s.x; P.y = s.y; P.id = s.id; P.act = s.act; P.last_reward = s.last_reward; P.dir = s.dir;
    P.turn = hE.turn_mode; P.body_w = G.body_w; P.body_l = G.body_l;
    P.mm = mm_val ? c->mm_pad : nullptr; P.mm_stride = mm_val ? c->mm_stride : 0;
    P.view = O.view; P.feature = O.feature;
    const int stride = 2 + (hE.minimap_mode ? 1 : 0);
    for (int j = 0; j < hE.G; ++j) {
        int rel = j - g; if (rel < 0) rel += hE.G;
        const int ch = hE.channel_base + rel * stride;                 // make_channel_trans, GridWorld.cc:897-913
        P.mm_ch[j] = ch + 2;
        P.grp_ch[j] = ch;
    }
}

static void launch_obs_dispatch(Ctx *c, const EngineDev &hE, const ObsArgs &O, ObsParams &P, int n_total, bool with_headers, bool headers_only) {
    const bool small_view = hE.grp[O.group].view_count <= 4 * 32;   // in-range view cells held in registers: 4 or 8 per lane
    if (hE.turn_mode) {                                         // headings: per-heading LUTs in shared memory (NIT = 8 code path)
        if (O.half) launch_obs_typed<__half, 8, true>(c, 0, hE, P, n_total, with_headers, headers_only);
        else launch_obs_typed<float, 8, true>(c, 1, hE, P, n_total, with_headers, headers_only);
    } else if (O.half) {
        if (small_view) launch_obs_typed<__half, 4, false>(c, 2, hE, P, n_total, with_headers, headers_only);
        else launch_obs_typed<__half, 8, false>(c, 3, hE, P, n_total, with_headers, headers_only);
    } else {
        if (small_view) launch_obs_typed<float, 4, false>(c, 4, hE, P, n_total, with_headers, headers_only);
        else launch_obs_typed<float, 8, false>(c, 5, hE, P, n_total, with_headers, headers_only);
    }
}

void launch_obs(Ctx *c, const EngineDev *, const EngineDev &hE, const ObsArgs &O, const float *mm_val, int n_total) {
    DeviceGuard guard(c);
    ObsParams P;
    fill_obs_params(c, hE, O, mm_val, n_total, P);
    launch_obs_dispatch(c, hE, O, P, n_total, true, false);
}

// ------------------------------------------------------------------------------------------------
// env_step's done word
__global__ void __launch_bounds__(256) done_reduce_kernel(const EngineDev *gE, int *out) {
    __shared__ int all_s;
    if (threadIdx.x == 0) all_s = 1;
    __syncthreads();
    int all = 1;
    for (int a = threadIdx.x; a < gE->A; a += blockDim.x) all &= gE->done[a] & 1;
    if (!all) all_s = 0;
    __syncthreads();
    if (threadIdx.x == 0) *out = all_s;
}

void read_done(Ctx *c, const EngineDev &hE, int *done_words) {
    no_capture(c, "env_step with a host `done`");
    DeviceGuard guard(c);
    if ((size_t)hE.A > c->pin_done_n) {
        if (c->pin_done) cudaFreeHost(c->pin_done);
        c->pin_done_n = (size_t)hE.A + 64;
        CUDA_CHECK(cudaHostAlloc((void **)&c->pin_done, c->pin_done_n * sizeof(int), cudaHostAllocDefault));
    }
    CUDA_CHECK(cudaMemcpyAsync(c->pin_done, hE.done, (size_t)hE.A * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaStreamSynchronize(c->stream));
    memcpy(done_words, c->pin_done, (size_t)hE.A * sizeof(int));
}

void counts_fetch_begin(Ctx *c, const int *dev_off, size_t n_ints) {
    no_capture(c, "the asynchronous count fetch");
    DeviceGuard guard(c);
    if (n_ints > c->pin_counts_n) {
        if (c->pin_counts) { CUDA_CHECK(cudaStreamSynchronize(c->stream)); cudaFreeHost(c->pin_counts); }
        c->pin_counts_n = n_ints + 64;
        CUDA_CHECK(cudaHostAlloc((void **)&c->pin_counts, c->pin_counts_n * sizeof(int), cudaHostAllocDefault));
    }
    CUDA_CHECK(cudaMemcpyAsync(c->pin_counts, dev_off, n_ints * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaEventRecord(c->ev_counts, c->stream));
}
const int *counts_fetch_wait(Ctx *c) {
    DeviceGuard guard(c);
    CUDA_CHECK(cudaEventSynchronize(c->ev_counts));
    return c->pin_counts;
}

void launch_done_to_device(Ctx *c, const EngineDev *dE, const EngineDev &, int *dev_done) {
    DeviceGuard guard(c);
    done_reduce_kernel<<<1, 256, 0, c->stream>>>(dE, dev_done);
    post_launch("done_reduce_kernel");
}

// ------------------------------------------------------------------------------------------------
// Host-buffer observations: the wire format (backend.h WireHdr / WireMark, DESIGN.md 6b).
//
// The reference ABI wants one dense float32 record per observer in HOST memory (4732 B for battle, 97 % zeros).
// PCIe moves ~55 GB/s; the host's memory system takes several times that.  So the GPU does the gather -- which cells of
// the view window show something, and what (Map::extract_view, Map.cc:129-207) -- and ships the answer as a compact
// record of ~60 B per observer; host threads then write the dense bytes (host_expand.cc).
//
// obs_wire_kernel: one warp per observer, ABI order.  Lanes stride over the in-range view cells (same LUT as the render
// kernel), load the kind byte and, for occupied cells, hp / max_hp; a ballot compacts the non-empty cells into the
// observer's slot row (worst-case sized, written sparsely).  Lane 0 writes the header and adds the count to the
// observer's chunk total.  wire_scan_kernel turns chunk totals into chunk bases; wire_compact_kernel copies the slot
// rows of a chunk into the contiguous mark stream the host reads.
__global__ void __launch_bounds__(256) obs_wire_kernel(const __grid_constant__ ObsParams P, WireHdr *whdr, WireMark *slots,
                                                       int slot_stride, int *chunk_total) {
    extern __shared__ __align__(16) unsigned char wire_smem[];
    int2 *lut = (int2 *)wire_smem;
    __shared__ int n_in_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lut_stride = (P.cells + 1) & ~1;
    if (warp == 0) {                                          // compact the view mask (Range.h:104-189), as obs_render_kernel does
        int k = 0;
        for (int base = 0; base < P.cells; base += 32) {
            const int cell = base + lane;
            const bool in = cell < P.cells && P.mask[cell];
            const unsigned bal = __ballot_sync(0xffffffffu, in);
            if (in) {
                const int vy = cell / P.vw, vx = cell - vy * P.vw;
                const int q = k + __popc(bal & ((1u << lane) - 1u));
                if (!P.turn) lut[q] = make_int2(cell * P.C, (P.oy + vy) * P.kw + P.ox + vx);
                else {
                    for (int d = 0; d < 4; ++d) {                       // one LUT per heading (Map.cc:140-146, 515-560)
                        int rx = 0, ry = 0, dx, dy;
                        if (d == DIR_SOUTH) { rx = P.body_w - 1; ry = P.body_l - 1; }
                        else if (d == DIR_WEST) ry = P.body_w - 1;
                        else if (d == DIR_EAST) rx = P.body_l - 1;
                        const int ex = P.ox + vx, ey = P.oy + vy;
                        if (d == DIR_NORTH) { dx = ex; dy = ey; }
                        else if (d == DIR_SOUTH) { dx = -ex; dy = -ey; }
                        else if (d == DIR_WEST) { dx = ey; dy = -ex; }
                        else { dx = -ey; dy = ex; }
                        lut[d * lut_stride + q] = make_int2(cell * P.C, (ry + dy) * P.kw + rx + dx);
                    }
                }
            }
            k += __popc(bal);
        }
        if (lane == 0) n_in_s = k;
    }
    __syncthreads();
    const int n_in = n_in_s;
    const int warps = gridDim.x * (blockDim.x >> 5);
    for (int o = blockIdx.x * (blockDim.x >> 5) + warp; o < P.n_total; o += warps) {
        const int4 h = P.hdr[o];                              // {x, y, arena, self cell | heading << 16}
        const long pb = h.z * P.kplane + (long)(h.y + P.kpad) * P.kw + h.x + P.kpad;
        const unsigned char *kp = P.kind_plane + pb;
        const float *hpnp = P.hpn_plane + pb;
        const int2 *l = lut + (P.turn ? ((h.w >> 16) & 3) * lut_stride : 0);
        WireMark *row = slots + (size_t)o * slot_stride;
        int running = 0;
        for (int base = 0; base < n_in; base += 32) {
            const int k = base + lane;
            int t = 0;
            int2 lk = make_int2(0, 0);
            if (k < n_in) { lk = l[k]; t = __ldg(kp + lk.y); }
            const unsigned bal = __ballot_sync(0xffffffffu, t != 0);
            if (t != 0) {
                WireMark m;
                if (t == KIND_WALL) { m.off = (unsigned)lk.x; m.val = 0.0f; }
                else if (t == KIND_FOOD) { m.off = (unsigned)lk.x + 1u; m.val = 0.0f; }
                else { m.off = (unsigned)(lk.x + P.grp_ch[kind_group(t)]) | WIRE_HAS_HP; m.val = (t & KIND_FULL) ? 1.0f : __ldg(hpnp + lk.y); }
                row[running + __popc(bal & ((1u << lane) - 1u))] = m;
            }
            running += __popc(bal);
        }
        if (lane == 0) {
            WireHdr w;
            w.arena = h.z;
            w.self_cell = (unsigned short)(h.w & 0xffff);
            w.count = (unsigned short)running;
            whdr[o] = w;
            if (running) atomicAdd(&chunk_total[o / WIRE_CHUNK], running);
        }
    }
}

__global__ void __launch_bounds__(1024) wire_scan_kernel(const int *chunk_total, long long *base, int n_chunks) {
    __shared__ long long carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int tile = 0; tile < n_chunks; tile += blockDim.x) {
        const int cidx = tile + threadIdx.x;
        const int v = cidx < n_chunks ? chunk_total[cidx] : 0;
        int tot;
        const int ex = block_excl_scan(v, tot);
        const long long carry = carry_s;
        if (cidx < n_chunks) base[cidx] = carry + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) base[n_chunks] = carry_s;
}

__global__ void __launch_bounds__(256) wire_compact_kernel(const WireHdr *whdr, const WireMark *slots, int slot_stride,
                                                           const long long *base, WireMark *stream, int n_total, int n_chunks) {
    __shared__ int off_s[WIRE_CHUNK];
    __shared__ unsigned short cnt_s[WIRE_CHUNK];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
        const int o0 = ch * WIRE_CHUNK, cnt_obs = min(WIRE_CHUNK, n_total - o0);
        int running = 0;
        for (int tile = 0; tile < WIRE_CHUNK; tile += blockDim.x) {
            const int i = tile + threadIdx.x;
            const int v = i < cnt_obs ? (int)whdr[o0 + i].count : 0;
            int tot;
            const int ex = block_excl_scan(v, tot);
            off_s[i] = running + ex;
            cnt_s[i] = (unsigned short)v;
            running += tot;
        }
        __syncthreads();
        WireMark *dst = stream + base[ch];
        for (int i = warp; i < cnt_obs; i += nw) {
            const int n = cnt_s[i], off = off_s[i];
            const WireMark *src = slots + (size_t)(o0 + i) * slot_stride;
            for (int k = lane; k < n; k += 32) dst[off + k] = src[k];
        }
        __syncthreads();
    }
}

template <class T>
static void grow_dev(Ctx *c, T *&p, size_t &have, size_t need) {
    if (need <= have) return;
    if (p) { CUDA_CHECK(cudaStreamSynchronize(c->stream)); CUDA_CHECK(cudaStreamSynchronize(c->copy)); cudaFree(p); }
    have = need + need / 4 + 64;
    CUDA_CHECK(cudaMalloc((void **)&p, have * sizeof(T)));
}
template <class T>
static void grow_pinned(Ctx *c, T *&p, size_t &have, size_t need) {
    if (need <= have) return;
    if (p) { CUDA_CHECK(cudaStreamSynchronize(c->copy)); cudaFreeHost(p); }
    have = need + need / 2 + 1024;
    CUDA_CHECK(cudaHostAlloc((void **)&p, have * sizeof(T), cudaHostAllocDefault));
}

void obs_wire_begin(Ctx *c, const EngineDev *, const EngineDev &hE, const ObsArgs &O, const float *mm_val, int n_total,
                    WireDesc *out) {
    no_capture(c, "an observation into host memory");
    DeviceGuard guard(c);
    ObsParams P;
    fill_obs_params(c, hE, O, mm_val, n_total, P);
    launch_obs_dispatch(c, hE, O, P, n_total, true, true);               // headers + feature rows (into O.feature)
    const int n_in = hE.grp[O.group].view_count;
    const int n_chunks = (n_total + WIRE_CHUNK - 1) / WIRE_CHUNK;
    grow_dev(c, c->wire_slots, c->wire_slots_n, (size_t)n_total * n_in);
    grow_dev(c, c->wire_hdr, c->wire_hdr_n, (size_t)n_total);
    {
        size_t have = c->wire_base_n;
        grow_dev(c, c->wire_base, c->wire_base_n, (size_t)n_chunks + 1);
        if (c->wire_base_n != have) {
            if (c->wire_chunk_total) cudaFree(c->wire_chunk_total);
            CUDA_CHECK(cudaMalloc((void **)&c->wire_chunk_total, c->wire_base_n * sizeof(int)));
        }
    }
    CUDA_CHECK(cudaMemsetAsync(c->wire_chunk_total, 0, (size_t)n_chunks * sizeof(int), c->stream));
    {
        const size_t smem = (size_t)(P.turn ? 4 : 1) * ((P.cells + 1) & ~1) * sizeof(int2);
        if (smem > 48 * 1024) mg::fatal("view too large for the wire kernel (%zu bytes of shared memory)", smem);
        int grid = (n_total + 7) / 8;
        if (grid > 8 * c->sms) grid = 8 * c->sms;
        obs_wire_kernel<<<grid, 256, smem, c->stream>>>(P, c->wire_hdr, c->wire_slots, n_in, c->wire_chunk_total);
        post_launch("obs_wire_kernel");
        wire_scan_kernel<<<1, 1024, 0, c->stream>>>(c->wire_chunk_total, c->wire_base, n_chunks);
        post_launch("wire_scan_kernel");
    }
    grow_pinned(c, c->h_wire_base, c->h_wire_base_n, (size_t)n_chunks + 1);
    CUDA_CHECK(cudaMemcpyAsync(c->h_wire_base, c->wire_base, ((size_t)n_chunks + 1) * sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
    CUDA_CHECK(cudaEventRecord(c->ev_done, c->stream));                  // totals on their way
    if (mm_val) {
        grow_pinned(c, c->h_mm, c->h_mm_n, (size_t)hE.A * c->mm_stride);
        CUDA_CHECK(cudaMemcpyAsync(c->h_mm, c->mm_pad, (size_t)hE.A * c->mm_stride * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    }
    grow_pinned(c, c->h_wire_hdr, c->h_wire_hdr_n, (size_t)n_total);
    // the mark stream cannot be longer than every in-range cell of every observer; it is sized from the real total below
    CUDA_CHECK(cudaEventSynchronize(c->ev_done));
    const long long total_marks = c->h_wire_base[n_chunks];
    grow_dev(c, c->wire_stream, c->wire_stream_n, (size_t)total_marks + 1);
    grow_pinned(c, c->h_wire_marks, c->h_wire_marks_n, (size_t)total_marks + 1);
    {
        int grid = n_chunks < 8 * c->sms ? n_chunks : 8 * c->sms;
        wire_compact_kernel<<<grid, 256, 0, c->stream>>>(c->wire_hdr, c->wire_slots, n_in, c->wire_base, c->wire_stream, n_total, n_chunks);
        post_launch("wire_compact_kernel");
    }
    CUDA_CHECK(cudaEventRecord(c->ev_wire, c->stream));
    // queue the copies wave by wave on the copy stream
    CUDA_CHECK(cudaStreamWaitEvent(c->copy, c->ev_wire, 0));
    int cpw = (n_chunks + 7) / 8;
    if (cpw < 4) cpw = 4;
    const int n_waves = (n_chunks + cpw - 1) / cpw;
    while ((int)c->wave_events.size() < n_waves) {
        cudaEvent_t e; CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); c->wave_events.push_back(e);
    }
    for (int q = 0; q < n_waves; ++q) {
        const int half = (n_waves + 1) / 2;
        const int w = (q & 1) ? half + (q >> 1) : (q >> 1);             // 0, half, 1, half + 1, ...
        out->wave_order[q] = w;
        const int c0 = w * cpw, c1 = (c0 + cpw < n_chunks) ? c0 + cpw : n_chunks;
        const size_t o0 = (size_t)c0 * WIRE_CHUNK, o1 = (size_t)c1 * WIRE_CHUNK < (size_t)n_total ? (size_t)c1 * WIRE_CHUNK : (size_t)n_total;
        CUDA_CHECK(cudaMemcpyAsync(c->h_wire_hdr + o0, c->wire_hdr + o0, (o1 - o0) * sizeof(WireHdr), cudaMemcpyDeviceToHost, c->copy));
        const long long m0 = c->h_wire_base[c0], m1 = c->h_wire_base[c1];
        if (m1 > m0) CUDA_CHECK(cudaMemcpyAsync(c->h_wire_marks + m0, c->wire_stream + m0, (size_t)(m1 - m0) * sizeof(WireMark), cudaMemcpyDeviceToHost, c->copy));
        CUDA_CHECK(cudaEventRecord(c->wave_events[w], c->copy));
    }
    c->waves_queued = n_waves;
    out->hdr = c->h_wire_hdr; out->marks = c->h_wire_marks; out->chunk_base = c->h_wire_base;
    out->mm = mm_val ? c->h_mm : nullptr; out->mm_stride = mm_val ? c->mm_stride : 0;
    out->n_total = n_total; out->n_chunks = n_chunks; out->n_waves = n_waves; out->chunks_per_wave = cpw;
}

void obs_wire_wait(Ctx *c, int wave) {
    DeviceGuard guard(c);
    CUDA_CHECK(cudaEventSynchronize(c->wave_events[wave]));
}

void dma_d2h_async(Ctx *c, void *dst, const void *src, size_t bytes) {
    DeviceGuard guard(c);
    CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->copy));
    if (c->dma_events.size() < 64) {
        while (c->dma_events.size() < 64) { cudaEvent_t e; CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); c->dma_events.push_back(e); }
    }
    if (c->dma_tail - c->dma_head >= c->dma_events.size()) {             // ring full: retire the oldest
        CUDA_CHECK(cudaEventSynchronize(c->dma_events[c->dma_head % c->dma_events.size()]));
        ++c->dma_head;
    }
    CUDA_CHECK(cudaEventRecord(c->dma_events[c->dma_tail % c->dma_events.size()], c->copy));
    ++c->dma_tail;
}

void dma_wait(Ctx *c, int keep_in_flight) {
    DeviceGuard guard(c);
    while ((long long)(c->dma_tail - c->dma_head) > (long long)keep_in_flight) {
        CUDA_CHECK(cudaEventSynchronize(c->dma_events[c->dma_head % c->dma_events.size()]));
        ++c->dma_head;
    }
}

}  // namespace be
}  // namespace mg
