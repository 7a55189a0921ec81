// ab_api.cu -- host side of libaerobulk_gpu.so: the AEROBULK_MODEL session
// (reference src/mod_aerobulk.f90:24-269 + the SAVEd globals of src/mod_const.f90:22-33
// and the warm-layer module arrays of src/mod_skin_coare.f90:31-36 /
// src/mod_skin_ecmwf.f90:52-55) and the C ABI declared in include/aerobulk_gpu.h.
//
// Data layout in HBM: every field is one contiguous array of Ni*Nj points in the caller's
// (Fortran, column-major) order, FP64 -- or FP32 for the whole of an aerobulk_gpu_model*_f32
// call; a row block j0..j1 is the byte range [j0*Ni*es, j1*Ni*es) of each field (es = 8 or
// 4 bytes per element), so chunks and shards are plain pointer offsets.
// Host-array calls stage through 8 input + 6 output device arrays (grow-only) and are
// pipelined in row-block chunks over three streams (H2D | kernel | D2H).
// Warm-layer state never leaves the device between jt==1 and jt==nitend.
// the library is built with -fvisibility=hidden: only the declared C ABI is exported
#pragma GCC visibility push(default)
#include "../../include/aerobulk_gpu.h"
#pragma GCC visibility pop

#include <cuda_runtime.h>

#include <math.h>
#if defined(__linux__)
#include <sched.h>
#endif
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <condition_variable>
#include <fstream>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "ab_copy_pool.hpp"
#include "ab_kernels.cuh"

namespace {

constexpr int MAX_CHUNKS = 16;          // capacity of a chunk plan (plan_chunks)
// the staged pipelines (plan_chunks kinds 1 and 3): chunks of at least MIN_CHUNK_POINTS, at most STAGED_CHUNKS of them
// (6, measured best on B200) or SPEC_CHUNKS with the speculative AEROBULK_INIT
constexpr int STAGED_CHUNKS = 6, SPEC_CHUNKS = 12;
constexpr long long MIN_CHUNK_POINTS = 200000;
// Zero-copy host-array calls.  When EVERY array of a call is pinned host memory (cudaHostAlloc / cudaHostRegister: it has a
// device alias under unified virtual addressing) the flux kernel loads its inputs from and stores its outputs to the
// caller's arrays directly: each byte crosses PCIe once, both directions busy for the whole launch, no staging, no
// copy-engine granularity.  Measured 1.54 ms per 1 M-point skin call against 1.75-1.85 ms for the staged pipeline
// (tools/e2e_probe.py); one direction alone measured slower (outputs 1.77 ms, inputs 2.27 ms).  Not used at jt == 1 when
// AEROBULK_INIT needs the field statistics (the inputs would cross PCIe twice), nor together with the stability sort (a
// gather / scatter across PCIe: 4.7 ms).  AEROBULK_GPU_ZEROCOPY=0 turns it off, and with it the pinned slab of pageable
// arrays, which the kernel reads zero-copy too.
bool zerocopy_on()
{
    static bool v = [] { const char *e = getenv("AEROBULK_GPU_ZEROCOPY"); return e ? atoi(e) != 0 : true; }();
    return v;
}
// device alias of a pinned (page-locked, device-mapped) host pointer, or nullptr
template <class T>
T *device_alias(T *p)
{
    if (!p) return nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return (a.type == cudaMemoryTypeHost && a.devicePointer) ? static_cast<T *>(a.devicePointer) : nullptr;
}
// element i of an array of es-byte elements (aerobulk_model arrays are FP64 or FP32, see model_impl); NULL stays NULL
template <class T>
T *elem_at(T *p, long long i, size_t es)
{
    return p ? p + i * (long long)es : nullptr;
}


// ---------------------------------------------------------------------------
// Host bounce path for PAGEABLE caller arrays (the plain relink case: Fortran / numpy arrays nobody pinned).
// cudaMemcpyAsync from pageable memory is staged by the driver on ONE thread (measured 8.3 ms per 1 M-point skin call,
// 14 GB/s).  Instead a few persistent host threads move each row-block chunk between the caller's arrays and a pinned
// slab owned by the library, and the flux kernel works on that slab zero-copy: chunk c+1 is copied in and chunk c-1
// copied out while the kernel runs on chunk c.  AEROBULK_GPU_BOUNCE=0 restores the driver-staged copies,
// AEROBULK_GPU_HOST_THREADS sets the number of copy threads (default: 3/4 of the CPUs of the affinity mask, at most 12).
// ---------------------------------------------------------------------------
using abpool::CopyPiece;
using abpool::CopyPool;
int host_threads()
{
    static int v = [] {
        const char *e = getenv("AEROBULK_GPU_HOST_THREADS");
        int k;
        if (e) {
            k = atoi(e);
        } else {
            // the CPUs this process may run on (an MPI rank bound to a few cores must not spin 8 threads on them)
            int cpus = (int)std::thread::hardware_concurrency();
#if defined(__linux__)
            cpu_set_t set;
            if (sched_getaffinity(0, sizeof(set), &set) == 0) cpus = CPU_COUNT(&set);
#endif
            // three quarters of them, at most 12: measured on the 16-core GPU box (tools/pageable_jt1_probe.py, 9.3 M-point
            // jt == 1 skin call) 4 / 8 / 12 / 16 threads -> 32.1 / 25.4 / 23.1 / 22.2 ms; the 1 M-point jt > 1 call
            // (tools/pin_probe.py) 2.32 / 2.27 / 2.30 / 2.35 ms with 6 / 8 / 12 / 16
            k = cpus * 3 / 4;
            if (k > 12) k = 12;
        }
        return k < 1 ? 1 : (k > 64 ? 64 : k);
    }();
    return v;
}
CopyPool &copy_pool()
{
    static CopyPool *p = new CopyPool(host_threads(), [] { const char *e = getenv("AEROBULK_GPU_COPY_STREAMING"); return e ? atoi(e) != 0 : true; }());   // never destroyed: its threads outlive static destructors
    return *p;
}
// CopyPool::run has ONE caller at a time; the device threads of a split call take turns (the copies are bound by the
// host memory system, which they share anyway)
void pool_run(const CopyPiece *pieces, int np)
{
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    copy_pool().run(pieces, np);
}
bool bounce_on()
{
    static int v = [] { const char *e = getenv("AEROBULK_GPU_BOUNCE"); return e ? atoi(e) : 1; }();
    return v != 0;
}
long long bounce_chunk_points()
{
    static long long v = [] {
        const char *e = getenv("AEROBULK_GPU_BOUNCE_CHUNK_POINTS");
        long long k = e ? atoll(e) : 180224;
        return k < 2048 ? 2048 : k;
    }();
    return v;
}
size_t bounce_max_bytes()   // larger slabs are not worth pinning: the driver-staged copies take over
{
    static size_t v = [] {
        const char *e = getenv("AEROBULK_GPU_BOUNCE_MAX_MB");
        return (size_t)(e ? atoll(e) : 12288) << 20;   // 112 B per point: the 84 M-point grid of BASELINE C5 needs 9.4 GB
    }();
    return v;
}
constexpr long long BOUNCE_MIN_POINTS = 65536;   // below this the driver-staged copies are as fast
constexpr size_t COPY_PIECE_BYTES = 128 * 1024;

struct Session {
    // ---- module globals of mod_const.f90:22-33
    int nb_iter = 5;
    int nitend = 1;
    bool l_use_skin_schemes = false;
    int ihum = 0;   // 0 'sh', 1 'dp', 2 'rh'
    double rdt = 3600.;
    double gdept = 1.;
    // ---- plumbing
    int device = -1;
    bool device_ready = false;
    cudaStream_t own_stream = nullptr, user_stream = nullptr, in_stream = nullptr, out_stream = nullptr;
    bool use_user_stream = false;
    cudaEvent_t ev_in[MAX_CHUNKS] = {}, ev_k[MAX_CHUNKS] = {}, ev_out[MAX_CHUNKS] = {}, ev_bad = nullptr;
    int error_mode = 0;
    int verbose = 1;
    char errmsg[1024] = {0};
    int errcode = 0;
    bool preinit_done = false;
    // ---- warm-layer state (device)
    // n_* is the LOGICAL size (0: not allocated in the reference's sense); the device memory is kept
    // across sessions (cap_*) because cudaMalloc/cudaFree cost 5-600 ms per session otherwise
    long long n_coare = 0, n_ecmwf = 0, cap_coare = 0, cap_ecmwf = 0;
    double *c_state[4] = {nullptr, nullptr, nullptr, nullptr};   // dT_wl, Hz_wl, Qnt_ac, Tau_ac
    double *e_dT_wl = nullptr;
    // ---- staging for host-array calls: 14 rows of `cap` bytes (a multiple of ROW_ALIGN), for FP64 and FP32 calls alike
    long long cap = 0;
    char *d_in[8] = {}, *d_out[6] = {};
    // ---- pinned bounce slab for pageable caller arrays (14 rows, pitch cap_hb bytes: a multiple of ROW_ALIGN) and its device alias
    char *hb = nullptr, *hb_dev = nullptr;
    long long cap_hb = 0;
    // ---- the same for the other host-array entry points (turb, series, ice): arrays packed back to back
    double *hx = nullptr, *hx_dev = nullptr;
    long long cap_hx = 0;
    // ---- device slab of the other host-array entry points: staging and scratch (grow-only, see ensure_turb_slab)
    double *d_turb = nullptr;
    long long cap_turb = 0;
    // ---- stability-sort permutation (one uint16 per point, see classify_kernel)
    unsigned short *d_perm = nullptr;
    long long cap_perm = 0;
    int sort_points = 1;   // 0 never, 1 auto (where it measured faster), 2 always
    bool pitched_ok = true;       // pitched (2-D) staging copies allowed, see copy_fields
    int ice_form_per_point = 0;   // 0: LG15 form drag from the LAST point's ice fraction (reference), 1: per point
    // ---- statistics + deferred wind-stress flag
    double *d_partials = nullptr, *d_stats = nullptr;
    // ---- asynchronous AEROBULK_INIT of device-resident sessions: the stats-dependent verdict lives on the device
    // (d_init = {humidity type, error flag}, d_gstats = the combined statistics) until the host next synchronises
    int *d_init = nullptr;
    double *d_gstats = nullptr;
    // speculative AEROBULK_INIT of the staged host-array pipeline (see model_impl): per-chunk statistics, the running
    // combination after each chunk, and the running verdicts
    double *d_cstats = nullptr, *d_cgstats = nullptr;
    int *d_cinit = nullptr;
    bool init_pending = false;
    int pend_Nt = 0, pend_Ni = 0, pend_Nj = 0;
    bool pend_lsrad = false;
    char pend_algo[32] = {0};
    unsigned long long *d_bad = nullptr, *h_bad = nullptr;   // h_bad: pinned
    bool bad_pending = false;
    int pend_launches = 0;        // model calls whose flag has not been looked at yet
    int last_Ni = 0;
    const void *last_taux = nullptr, *last_tauy = nullptr;   // device pointers of the last launch
    size_t last_es = sizeof(double);                         // and the size of their elements
    long launches = 0;
    // ---- opt-in: device-pointer calls never synchronise, not even at jt == Nt (aerobulk_gpu_set_async)
    bool async_device = false;
    // ---- opt-in: CUDA events around every flux launch (aerobulk_gpu_set_kernel_timing): the roofline denominators of
    // bench.py are durations of the flux kernel ALONE, measured on the stream it runs on
    bool time_kernels = false;
    std::vector<cudaEvent_t> kt_ev;   // pairs
    size_t kt_used = 0;
    // ---- aerobulk_gpu_set_devices(n): this session's share of a call that the library split over several GPUs
    int shard = 0;                 // index of this session among the devices of the split
    long long flat_offset = 0;     // global flat index of the shard's first point (error messages, tau > 10 report)
    int report_Ni = 0, report_Nj = 0;   // the caller's (Ni,Nj): banner and (ji,jj) of error messages
    struct StatsHook *stats_hook = nullptr;   // jt == 1: row-block statistics -> global (AEROBULK_INIT sees the whole field)
};

// One session per GPU.  sess[0] is THE session of the single-device library (every entry point); with
// aerobulk_gpu_set_devices(n > 1) the host-array aerobulk_gpu_model call splits its points over sess[0..n-1], each
// driven by its own host thread whose `cur` points at its session.  `g` is "the session of the calling thread".
constexpr int MAX_DEVICES = 16;
Session sess[MAX_DEVICES];
thread_local Session *cur = &sess[0];
#define g (*cur)
int n_devices = 1;
std::mutex g_mu;

const char *HUM_NAMES[3] = {"sh", "dp", "rh"};

// Rendezvous of the per-device statistics of one split jt == 1 call (the reference computes AEROBULK_INIT's sums, minima
// and maxima over the WHOLE field, src/mod_aerobulk.f90:104-153): every shard contributes its 64-double vector, the last
// arrival combines them in shard order (deterministic), all leave with the global vector.  A shard that failed before
// reaching the rendezvous arrives with ok = false and everybody leaves with an error instead of waiting for ever.
struct StatsHook {
    std::mutex mu;
    std::condition_variable cv;
    int expected = 0, arrived = 0;
    bool failed = false;
    bool seen[MAX_DEVICES] = {};
    double part[MAX_DEVICES][abk::NSTATS];
    double global[abk::NSTATS];
    void reset(int n)
    {
        expected = n;
        arrived = 0;
        failed = false;
        for (int k = 0; k < MAX_DEVICES; ++k) seen[k] = false;
    }
    // returns false when some shard failed
    bool combine(int shard, const double *st, bool ok, double *out)
    {
        std::unique_lock<std::mutex> lk(mu);
        if (seen[shard]) return !failed;   // a shard arrives once (the failure path may call again)
        seen[shard] = true;
        if (ok) memcpy(part[shard], st, sizeof(double) * abk::NSTATS);
        else failed = true;
        if (++arrived == expected) {
            if (!failed) {
                for (int k = 0; k < abk::NSTATS; ++k) {
                    const int op = aerobulk_gpu_stats_reduce_op(k);
                    double r = part[0][k];
                    for (int d = 1; d < expected; ++d)
                        r = (op == 0) ? r + part[d][k] : (op == 1) ? fmin(r, part[d][k]) : fmax(r, part[d][k]);
                    global[k] = r;
                }
            }
            cv.notify_all();
        } else {
            cv.wait(lk, [&] { return arrived == expected; });
        }
        if (!failed && out) memcpy(out, global, sizeof(double) * abk::NSTATS);
        return !failed;
    }
};

// ---------------------------------------------------------------------------
// errors: ctl_stop semantics (mod_const.f90:238-278) or return codes
// ---------------------------------------------------------------------------
int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g.errmsg, sizeof(g.errmsg), fmt, ap);
    va_end(ap);
    g.errcode = code;
    if (g.error_mode == 0) {
        printf(" *** E R R O R :  \n %s\n\n", g.errmsg);
        fflush(stdout);
        exit(1);
    }
    return code;
}

#define CUDA_TRY(call)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            return fail(AEROBULK_GPU_ERR_CUDA, "CUDA error '%s' at %s:%d (%s)", cudaGetErrorString(e__), \
                        __FILE__, __LINE__, #call);                                                 \
    } while (0)

cudaStream_t compute_stream() { return g.use_user_stream ? g.user_stream : g.own_stream; }

int ensure_device()
{
    if (g.device_ready) {
        CUDA_TRY(cudaSetDevice(g.device));
        return 0;
    }
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0)
        return fail(AEROBULK_GPU_ERR_CUDA, "no CUDA device available (%s): libaerobulk_gpu has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (g.device < 0) {
        const char *env = getenv("AEROBULK_GPU_DEVICE");
        if (!env) env = getenv("LOCAL_RANK");
        g.device = env ? (atoi(env) % count) : 0;
    }
    if (g.device >= count) return fail(AEROBULK_GPU_ERR_CUDA, "device %d requested but only %d visible", g.device, count);
    CUDA_TRY(cudaSetDevice(g.device));
    CUDA_TRY(cudaStreamCreateWithFlags(&g.own_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&g.in_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&g.out_stream, cudaStreamNonBlocking));
    for (int i = 0; i < MAX_CHUNKS; ++i) {
        CUDA_TRY(cudaEventCreateWithFlags(&g.ev_in[i], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&g.ev_k[i], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&g.ev_out[i], cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventCreateWithFlags(&g.ev_bad, cudaEventDisableTiming));
    CUDA_TRY(cudaMalloc(&g.d_partials, sizeof(double) * abk::NSTATS * abk::stats_max_blocks()));
    CUDA_TRY(cudaMalloc(&g.d_stats, sizeof(double) * abk::NSTATS));
    CUDA_TRY(cudaMalloc(&g.d_gstats, sizeof(double) * abk::NSTATS));
    CUDA_TRY(cudaMalloc(&g.d_init, 2 * sizeof(int)));
    CUDA_TRY(cudaMemset(g.d_init, 0, 2 * sizeof(int)));
    CUDA_TRY(cudaMalloc(&g.d_cstats, sizeof(double) * abk::NSTATS * MAX_CHUNKS));
    CUDA_TRY(cudaMalloc(&g.d_cgstats, sizeof(double) * abk::NSTATS * MAX_CHUNKS));
    CUDA_TRY(cudaMalloc(&g.d_cinit, 2 * sizeof(int) * MAX_CHUNKS));
    // word 0: wind stress > 10 N/m^2; word 1 (sea-ice calls only): rough_leng_tq fail-stop
    CUDA_TRY(cudaMalloc(&g.d_bad, 2 * sizeof(unsigned long long)));
    CUDA_TRY(cudaHostAlloc(&g.h_bad, 2 * sizeof(unsigned long long), cudaHostAllocDefault));
    g.h_bad[0] = g.h_bad[1] = ~0ull;
    CUDA_TRY(cudaMemset(g.d_bad, 0xFF, 2 * sizeof(unsigned long long)));
    g.device_ready = true;
    return 0;
}

// *_EXIT of the reference: the state stops existing; the device memory stays cached
void release_coare_state() { g.n_coare = 0; }
void release_ecmwf_state() { g.n_ecmwf = 0; }
void free_coare_state()
{
    for (int k = 0; k < 4; ++k) {
        if (g.c_state[k]) cudaFree(g.c_state[k]);
        g.c_state[k] = nullptr;
    }
    g.n_coare = g.cap_coare = 0;
}
void free_ecmwf_state()
{
    if (g.e_dT_wl) cudaFree(g.e_dT_wl);
    g.e_dT_wl = nullptr;
    g.n_ecmwf = g.cap_ecmwf = 0;
}
int alloc_coare_state(long long n)
{
    if (n > g.cap_coare) {
        free_coare_state();
        for (int k = 0; k < 4; ++k) CUDA_TRY(cudaMalloc(&g.c_state[k], sizeof(double) * (size_t)n));
        g.cap_coare = n;
    }
    g.n_coare = n;
    return 0;
}
int alloc_ecmwf_state(long long n)
{
    if (n > g.cap_ecmwf) {
        free_ecmwf_state();
        CUDA_TRY(cudaMalloc(&g.e_dT_wl, sizeof(double) * (size_t)n));
        g.cap_ecmwf = n;
    }
    g.n_ecmwf = n;
    return 0;
}
// kt == nit000 -> *_INIT allocates the warm-layer state (mod_blk_coare3p6.f90:250,68-95; mod_blk_ecmwf.f90:189); the
// state is shared by aerobulk_model and TURB_*, like the module arrays of the reference
int init_wl_state(int ialgo, long long n)
{
    if (ialgo == abd::ECMWF) {
        if (g.n_ecmwf) return fail(AEROBULK_GPU_ERR_STATE, " ECMWF_INIT => allocation of dT_wl & Hz_wl failed!");
        return alloc_ecmwf_state(n);
    }
    if (g.n_coare) return fail(AEROBULK_GPU_ERR_STATE, " COARE_INIT => allocation of Tau_ac, Qnt_ac, dT_wl & Hz_wl failed!");
    return alloc_coare_state(n);
}
// points the warm-layer state of a FluxArgs / TurbArgs at the row block that starts at point s0
template <class Args>
void bind_wl_state(Args &a, int ialgo, long long s0)
{
    if (ialgo == abd::ECMWF) {
        a.dT_wl = g.e_dT_wl + s0;
    } else {
        a.dT_wl = g.c_state[0] + s0; a.Hz_wl = g.c_state[1] + s0;
        a.Qnt_ac = g.c_state[2] + s0; a.Tau_ac = g.c_state[3] + s0;
    }
}

// Moves elements [s0, s0+len) of `nf` fields of es-byte elements between host and device staging (dev_pitch: bytes
// between device rows).  Consecutive fields whose HOST arrays are equally spaced in memory (a caller that keeps its
// fields in one slab) go in ONE pitched copy: with H2D and D2H running concurrently in 0.4-3 MB pieces the DMA engines
// reach 62 GB/s aggregate, with one pitched copy per chunk 72 GB/s (tools/probes/duplex_probe.cu on this pool's B200:
// 1.86 -> 1.62 ms per 1 M-point skin call).
int copy_fields(int nf, char *const *dev, char *const *host, long long dev_pitch, long long s0, long long len, size_t es,
                bool h2d, cudaStream_t st)
{
    const long long MAX_PITCH_BYTES = 0x7fffffffLL;   // cudaDevAttrMaxPitch
    const long long o = s0 * (long long)es, bytes = len * (long long)es;
    int k = 0;
    while (k < nf) {
        if (!host[k]) { ++k; continue; }
        int run = 1;
        if (k + 1 < nf && host[k + 1]) {
            const long long d = host[k + 1] - host[k];   // bytes
            if (d >= bytes && d <= MAX_PITCH_BYTES && dev_pitch <= MAX_PITCH_BYTES)
                while (k + run < nf && host[k + run] && host[k + run] - host[k + run - 1] == d) ++run;
        }
        if (run > 1 && g.pitched_ok) {
            const size_t hp = (size_t)(host[k + 1] - host[k]), dp = (size_t)dev_pitch, w = (size_t)bytes;
            const cudaError_t e =
                h2d ? cudaMemcpy2DAsync(dev[k] + o, dp, host[k] + o, hp, w, (size_t)run, cudaMemcpyHostToDevice, st)
                    : cudaMemcpy2DAsync(host[k] + o, hp, dev[k] + o, dp, w, (size_t)run, cudaMemcpyDeviceToHost, st);
            if (e == cudaErrorInvalidValue) {
                // equally spaced but SEPARATE pinned allocations: the driver refuses a pitched copy that spans them.
                // Nothing was enqueued; use plain copies from now on.
                cudaGetLastError();
                g.pitched_ok = false;
                continue;
            }
            CUDA_TRY(e);
        } else if (run > 1) {
            for (int j = k; j < k + run; ++j) {
                if (h2d) CUDA_TRY(cudaMemcpyAsync(dev[j] + o, host[j] + o, (size_t)bytes, cudaMemcpyHostToDevice, st));
                else CUDA_TRY(cudaMemcpyAsync(host[j] + o, dev[j] + o, (size_t)bytes, cudaMemcpyDeviceToHost, st));
            }
        } else {
            if (h2d) CUDA_TRY(cudaMemcpyAsync(dev[k] + o, host[k] + o, (size_t)bytes, cudaMemcpyHostToDevice, st));
            else CUDA_TRY(cudaMemcpyAsync(host[k] + o, dev[k] + o, (size_t)bytes, cudaMemcpyDeviceToHost, st));
        }
        k += run;
    }
    return 0;
}

// Row pitch of the staging arrays and of the pinned slab: the bytes of one field (points x element size) rounded up to
// ROW_ALIGN.  Both are grow-only and shared by FP64 and FP32 calls, so a row sized for an odd number of floats must not
// leave a later, smaller FP64 call with rows that are not 8-byte aligned; 256 bytes also keeps every row on a whole
// number of 128-byte lines for coalesced access.
constexpr long long ROW_ALIGN = 256;
long long aligned_row(long long bytes) { return (bytes + ROW_ALIGN - 1) / ROW_ALIGN * ROW_ALIGN; }

// `row`: bytes per field (points x element size)
int ensure_staging(long long row)
{
    row = aligned_row(row);
    if (row <= g.cap) return 0;
    // one slab, fields equally spaced (pitch = cap bytes): a run of equally spaced caller arrays then moves with ONE
    // pitched copy per chunk (see copy_fields)
    if (g.d_in[0]) cudaFree(g.d_in[0]);
    for (int k = 0; k < 8; ++k) g.d_in[k] = nullptr;
    for (int k = 0; k < 6; ++k) g.d_out[k] = nullptr;
    g.cap = 0;
    char *slab = nullptr;
    CUDA_TRY(cudaMalloc(&slab, (size_t)row * 14));
    for (int k = 0; k < 8; ++k) g.d_in[k] = slab + (long long)k * row;
    for (int k = 0; k < 6; ++k) g.d_out[k] = slab + (long long)(8 + k) * row;
    g.cap = row;
    return 0;
}

void free_bounce()
{
    if (g.hb) cudaFreeHost(g.hb);
    g.hb = g.hb_dev = nullptr;
    g.cap_hb = 0;
    if (g.hx) cudaFreeHost(g.hx);
    g.hx = g.hx_dev = nullptr;
    g.cap_hx = 0;
}
// Grows a mapped pinned slab to `rows` rows of n elements of type T (cap counts n).  False, with the slab released, when
// the host has no pinned memory to spare: the session stays usable and the caller keeps the driver-staged copies.
template <class T>
bool grow_mapped(T *&h, T *&d, long long &cap, long long n, int rows)
{
    if (n <= cap) return true;
    if (h) cudaFreeHost(h);
    h = d = nullptr;
    cap = 0;
    if (cudaHostAlloc(&h, sizeof(T) * (size_t)n * rows, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer(&d, h, 0) != cudaSuccess) {
        cudaGetLastError();
        if (h) cudaFreeHost(h);
        h = d = nullptr;
        return false;
    }
    cap = n;
    return true;
}
// `row`: bytes per field (points x element size)
bool ensure_bounce(long long row)
{
    row = aligned_row(row);
    if (row <= g.cap_hb) return true;
    if ((size_t)row * 14 > bounce_max_bytes()) return false;
    free_bounce();
    return grow_mapped(g.hb, g.hb_dev, g.cap_hb, row, 14);
}
// appends the copy of `bytes` bytes from src to dst, cut into COPY_PIECE_BYTES pieces for the copy threads
void add_pieces(std::vector<CopyPiece> &pieces, void *dst, const void *src, size_t bytes)
{
    char *d = static_cast<char *>(dst);
    const char *s = static_cast<const char *>(src);
    for (size_t o = 0; o < bytes; o += COPY_PIECE_BYTES)
        pieces.push_back(CopyPiece{d + o, s + o, bytes - o < COPY_PIECE_BYTES ? bytes - o : COPY_PIECE_BYTES});
}
// copy points [s0, s0+len) of nf fields of es-byte elements between the caller's arrays and the bounce slab rows
// row0.., on the copy threads
void bounce_copy(int nf, char *const *user, int row0, long long s0, long long len, size_t es, bool to_slab)
{
    static thread_local std::vector<CopyPiece> pieces;
    pieces.clear();
    const long long o = s0 * (long long)es;
    const size_t bytes = (size_t)len * es;
    for (int k = 0; k < nf; ++k) {
        if (!user[k]) continue;
        char *u = user[k] + o, *b = g.hb + (long long)(row0 + k) * g.cap_hb + o;
        if (to_slab) add_pieces(pieces, b, u, bytes);
        else add_pieces(pieces, u, b, bytes);
    }
    pool_run(pieces.data(), (int)pieces.size());
}

int algo_id(const char *calgo)
{
    if (!strcmp(calgo, "coare3p0")) return abd::COARE3P0;
    if (!strcmp(calgo, "coare3p6")) return abd::COARE3P6;
    if (!strcmp(calgo, "ncar")) return abd::NCAR;
    if (!strcmp(calgo, "ecmwf")) return abd::ECMWF;
    if (!strcmp(calgo, "andreas")) return abd::ANDREAS;
    return 0;
}

// COARE 3.0, COARE 3.6 and ECMWF have cool-skin / warm-layer schemes; NCAR and ANDREAS have none
bool has_skin_schemes(int ialgo) { return ialgo == abd::COARE3P0 || ialgo == abd::COARE3P6 || ialgo == abd::ECMWF; }

// l_zt_equal_zu of the TURB_* routines: the ZTEQ kernels when the two heights are less than 1 cm apart
bool zt_eq_zu(double zt, double zu) { return fabs(zu - zt) < 0.01; }

// ---------------------------------------------------------------------------
// AEROBULK_INIT from field statistics (mod_aerobulk.f90:24-160)
// ---------------------------------------------------------------------------
struct FieldCheck {
    const char *name, *unit;
    double zmin, zmax;
};
// order of the statistics vector: sst t_air slp u10 v10 wnd hum rad_sw(=rad_lw) rad_lw
const FieldCheck CHECKS[9] = {
    {"sst", "K", 270., 320.},      {"t_air", "K", 180., 330.},   {"slp", "Pa", 80000., 110000.},
    {"u10", "m/s", -50., 50.},     {"v10", "m/s", -50., 50.},    {"wnd", "m/s", 0., 50.},
    {"hum", "kg/kg", 0., 0.},      {"rad_sw", "W/m^2", 0., 1500.}, {"rad_lw", "W/m^2", 0., 750.}};

int check_units(const char *name, const char *unit, double zmin, double zmax, const double *st5, double np)
{
    // check_unit_consistency, mod_phymbl.f90:1851-1954
    const double zmean = st5[0] / np;
    const bool bad = (st5[2] > zmax) || (st5[1] < zmin) || (zmean < zmin) || (zmean > zmax);
    if (bad)
        return fail(AEROBULK_GPU_ERR_UNITS,
                    "*** ERROR (check_unit_consistency@mod_phymbl): field `%s` does not seem to be in %s !\n"
                    " min value = %10.3E max value = %10.3E mean value = %10.3E",
                    name, unit, st5[3], st5[4], zmean);
    return 0;
}

// AEROBULK_INIT, first half (mod_aerobulk.f90:56-99): what depends on the ARGUMENTS only -- skin flag, nitend
int init_flags(int Nt, const char *calgo, bool lskin, bool lsrad)
{
    if (g.verbose) {
        printf(" \n ===================================================================\n");
        printf("                    ----- AeroBulk_init -----\n \n");
        printf("     *** Bulk parameterization to be used => \"%s\"\n", calgo);
    }
    if (lskin) {
        if (!(strncmp(calgo, "coar", 4) == 0 || strcmp(calgo, "ecmwf") == 0))
            return fail(AEROBULK_GPU_ERR_SKIN_ALGO,
                        "AEROBULK_INIT => Only `COARE*` and `ECMWF` algorithms support cool-skin & warm/layer schemes");
        if (!lsrad)
            return fail(AEROBULK_GPU_ERR_SKIN_NORAD,
                        "AEROBULK_INIT => provide SW and LW rad. input if you want to use skin schemes");
        g.l_use_skin_schemes = true;   // :74 -- sticky
        if (g.verbose) printf("        ==> will use the Cool-skin & Warm-layer scheme of `%s` !\n", calgo);
    } else if (g.verbose) {
        printf("     *** Cool-skin & Warm-layer schemes will NOT be used!\n");
    }
    g.nitend = Nt;   // :99
    return 0;
}

// AEROBULK_INIT, second half (mod_aerobulk.f90:100-160): what depends on the field STATISTICS -- mask, humidity type, units
int init_checks(bool lsrad, const double *st, int Ni, int Nj)
{
    if (g.verbose) {
        if (Ni > 0) printf("     *** Computational domain shape: Ni x Nj = %05d x %05d\n", Ni, Nj);
        printf("     *** Number of time records that will be treated: %11d\n", g.nitend);
        printf("     *** Number of iterations in bulk algos: nb_iter  = %4d\n", g.nb_iter);
        printf("     *** Filling the `mask` array...\n");
    }
    const double np = st[0], ntot = st[1];
    if (np == ntot) {
        if (g.verbose) printf("         ==> no points need to be masked! :)\n");
    } else if (np > 0.) {
        if (g.verbose) printf("         ==> number of points to mask: %.0f (out of %.0f)\n", ntot - np, ntot);
    } else {
        return fail(AEROBULK_GPU_ERR_ALL_MASKED, "the whole domain is masked!\n check unit consistency of input fields");
    }
    // type_of_humidity, mod_phymbl.f90:1957-2007
    const double *h = st + 2 + 5 * 6;
    const double zmean = h[0] / np, zmin = h[1], zmax = h[2];
    const char *ln;
    if (zmean >= 0. && zmean < 0.08 && zmin >= 0. && zmax < 0.08) { g.ihum = 0; ln = "specific humidity [kg/kg]"; }
    else if (zmean >= 150. && zmean < 330. && zmin >= 150. && zmax < 330.) { g.ihum = 1; ln = "dew-point temperature [K]"; }
    else if (zmean >= 0. && zmean <= 100. && zmin >= 0. && zmax <= 100.) { g.ihum = 2; ln = "relative humidity [%]"; }
    else
        return fail(AEROBULK_GPU_ERR_HUMIDITY,
                    "ERROR: type_of_humidity()@mod_aerobulk_compute => un-identified humidity type!\n"
                    "   ==> we could not identify the humidity type based on the mean, min & max of the field:\n"
                    "     * mean = %g\n     * min  = %g\n     * max  = %g", zmean, zmin, zmax);
    if (g.verbose) printf("     *** Type of prescribed air humidity  `%s`\n", ln);

    for (int f = 0; f < (lsrad ? 9 : 7); ++f) {
        FieldCheck c = CHECKS[f];
        if (f == 6) {
            // check_unit_consistency(ctype_humidity, pha): note the reference's unit label is 'kg/kg' for all three
            c.unit = "kg/kg";
            if (g.ihum == 0) { c.name = "sh"; c.zmin = 0.; c.zmax = 0.08; }
            else if (g.ihum == 1) { c.name = "dp"; c.zmin = 150.; c.zmax = 330.; }
            else { c.name = "rh"; c.zmin = 0.; c.zmax = 100.; }
        }
        int rc = check_units(c.name, c.unit, c.zmin, c.zmax, st + 2 + 5 * f, np);
        if (rc) return rc;
    }
    if (g.verbose) {
        printf(" ===================================================================\n");
        fflush(stdout);
    }
    return 0;
}

int init_from_stats(int Nt, const char *calgo, bool lskin, bool lsrad, const double *st, int Ni, int Nj)
{
    const int rc = init_flags(Nt, calgo, lskin, lsrad);
    return rc ? rc : init_checks(lsrad, st, Ni, Nj);
}

// Asynchronous AEROBULK_INIT (device-resident sessions, banners off): the argument-only half runs now, the statistics
// are combined and judged by init_decide_kernel on the compute stream, and the kernels that follow read the humidity
// type (and the stop flag) from device memory.  The host catches up in resolve_init() at its next synchronisation.
int init_async(int Nt, const char *calgo, bool lskin, bool lsrad, const double *d_all, int nranks, int Ni, int Nj, cudaStream_t s)
{
    int rc = init_flags(Nt, calgo, lskin, lsrad);
    if (rc) return rc;
    CUDA_TRY(abk::launch_init_decide(d_all, nranks, lsrad ? 1 : 0, g.d_gstats, g.d_init, s));
    g.launches += 1;
    g.init_pending = true;
    g.pend_Nt = Nt;
    g.pend_Ni = Ni;
    g.pend_Nj = Nj;
    g.pend_lsrad = lsrad;
    snprintf(g.pend_algo, sizeof(g.pend_algo), "%s", calgo);
    return 0;
}

// The host half of an asynchronous AEROBULK_INIT: waits for the stream, reads the combined statistics back and runs the
// reference's checks on them (same verdict as the device, with the reference's messages).  Cheap no-op otherwise.
int resolve_init()
{
    if (!g.init_pending) return 0;
    g.init_pending = false;
    double st[abk::NSTATS];
    CUDA_TRY(cudaMemcpyAsync(st, g.d_gstats, sizeof(st), cudaMemcpyDeviceToHost, compute_stream()));
    CUDA_TRY(cudaStreamSynchronize(compute_stream()));
    return init_checks(g.pend_lsrad, st, g.pend_Ni, g.pend_Nj);
}

// stats_fast_kernel + stats_fix_kernel + stats_final (their *_io_kernel<float> twins for es == sizeof(float)) on stream
// s; the 64-double vector lands in `d_out` (device memory)
int launch_local_stats(long long n, size_t es, const void *sst, const void *t_zt, const void *hum, const void *U,
                       const void *V, const void *slp, const void *rad_lw, cudaStream_t s, double *d_out)
{
    abk::StatsArgs a;
    a.sst = sst; a.t_zt = t_zt; a.hum_zt = hum; a.U_zu = U; a.V_zu = V; a.slp = slp; a.rad_lw = rad_lw;
    a.n = n;
    a.partials = g.d_partials;
    a.out = d_out;
    long long want = (n + 255) / 256;
    int nblocks = (int)(want < 1 ? 1 : (want > abk::stats_max_blocks() ? abk::stats_max_blocks() : want));
    CUDA_TRY(abk::launch_stats(es, a, nblocks, s));
    g.launches += 3;   // stats_fast_kernel, stats_fix_kernel, stats_final
    return 0;
}
int local_stats(long long n, size_t es, const void *sst, const void *t_zt, const void *hum, const void *U,
                const void *V, const void *slp, const void *rad_lw, cudaStream_t s, double *host_stats)
{
    const int rc = launch_local_stats(n, es, sst, t_zt, hum, U, V, slp, rad_lw, s, g.d_stats);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(host_stats, g.d_stats, sizeof(double) * abk::NSTATS, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return 0;
}

abd::Uniform make_uniform(double zt, double zu)
{
    abd::Uniform u;
    u.zt = zt;
    u.zu = zu;
    u.log_zt = log(zt);
    u.log_zu = log(zu);
    u.log_ztu = log(zt / zu);
    u.log_zu10 = log(zu / 10.);
    u.log_10 = log(10.);
    const double zz0 = 0.0001;
    u.fg_c_a = 0.035 * log(10. / zz0) / log(zu / zz0);        // mod_common_coare.f90:107
    const double zc_b = 0.004 * 600. * 1.2 * 1.2 * 1.2;         // :108
    u.fg_1_o_Ribcu = -zc_b / zu;                               // :140
    u.rdt = g.rdt;
    u.gdept = g.gdept;
    u.nb_iter = g.nb_iter;
    u.wl_commit_mask = 0ull;
    for (int jit = 1; jit < 64 && jit <= g.nb_iter; ++jit)
        if (g.nb_iter % jit == 0) u.wl_commit_mask |= 1ull << jit;
    u.isd = 12;   // aerobulk_compute passes isecday_utc=12 (seconds), mod_aerobulk_compute.f90:136,146
    u.dawn = abd::wl_coare_dawn(0., u.isd) ? 1 : 0;   // longitude fixed to 0, mod_aerobulk_compute.f90:126
    return u;
}

// element i of an array of es-byte elements, widened to double; `on_device`: p is device memory (false on a failed copy)
bool read_elem(const void *p, long long i, size_t es, bool on_device, double *v)
{
    const char *q = static_cast<const char *>(p) + i * (long long)es;
    float f = 0.f;
    void *dst = es == sizeof(float) ? static_cast<void *>(&f) : static_cast<void *>(v);
    if (on_device) {
        if (cudaMemcpy(dst, q, es, cudaMemcpyDeviceToHost) != cudaSuccess) return false;
    } else {
        memcpy(dst, q, es);
    }
    if (es == sizeof(float)) *v = f;
    return true;
}

// reports a wind stress > 10 N/m^2 found by earlier launches (mod_phymbl.f90:1250-1253); h_taux / h_tauy: the host
// output arrays of the last call (elements of g.last_es bytes), or NULL
int check_bad_flag(const void *h_taux, const void *h_tauy)
{
    if (!g.bad_pending) return 0;
    // the flag copy of an asynchronous device-pointer call may still be in flight (entry points that did not wait)
    cudaEventSynchronize(g.ev_bad);
    g.bad_pending = false;
    const int flagged_launches = g.pend_launches;
    g.pend_launches = 0;
    const unsigned long long bad = *g.h_bad;
    if (bad == ~0ull) return 0;
    *g.h_bad = ~0ull;
    // ordered after every kernel that may still be updating the word, unlike a memset on the legacy stream
    cudaMemsetAsync(g.d_bad, 0xFF, sizeof(unsigned long long), compute_stream());
    // (ji, jj) of the CALLER's grid: a shard of a split call reports through its global flat index
    const long long Ni = g.report_Ni > 0 ? g.report_Ni : (g.last_Ni > 0 ? g.last_Ni : 1);
    const long long idx = (long long)bad + g.flat_offset;
    double tx = 0., ty = 0.;
    bool have_tau = false;
    if (h_taux && h_tauy) {
        have_tau = read_elem(h_taux, (long long)bad, g.last_es, false, &tx) && read_elem(h_tauy, (long long)bad, g.last_es, false, &ty);
    } else if (g.last_taux && g.last_tauy && flagged_launches == 1) {
        // the buffers of the ONE call the flag can come from; with several asynchronous calls behind the flag the
        // offending call (and its output arrays and shape) is not known any more and only the index is reported
        have_tau = read_elem(g.last_taux, (long long)bad, g.last_es, true, &tx) && read_elem(g.last_tauy, (long long)bad, g.last_es, true, &ty);
    }
    if (have_tau)
        return fail(AEROBULK_GPU_ERR_TAU,
                    "BULK_FORMULA_VCTR()@mod_phymbl: wind stress too strong!\n  => %8.2f N/m^2 ! At ji, jj = %04lld, %04lld",
                    sqrt(tx * tx + ty * ty), idx % Ni + 1, idx / Ni + 1);
    return fail(AEROBULK_GPU_ERR_TAU,
                "BULK_FORMULA_VCTR()@mod_phymbl: wind stress too strong!\n  => above 10 N/m^2 in one of the last %d asynchronous "
                "calls, first at flat index %lld of that call",
                flagged_launches, idx);
}

// entry points other than aerobulk_gpu_model*: everything an earlier asynchronous call still owes the caller
int deferred_errors()
{
    const int rc = resolve_init();
    return rc ? rc : check_bad_flag(nullptr, nullptr);
}

// Row-block chunk plan of a host-array call: cstart[0..nchunks], boundaries on multiples of 2048 points (whole sort
// windows / thread blocks).
//   kind 0: one chunk (device arrays, zero-copy on pinned arrays);
//   kind 1: staged H2D | kernel | D2H pipeline.  It is H2D-bound (PCIe ~50 GB/s per direction measured, vs. >150 GB/s
//           consumed by the kernel), so its length is H2D(all) + kernel(last chunk) + D2H(last chunk): sizes decrease
//           linearly (weights K..1) to keep the exposed tail short while the early pieces stay large enough for full
//           PCIe efficiency.  (Two copy-in streams were measured slower: 2.3 vs 2.0 ms per 1M-point call.)
//   kind 2: pageable arrays through the pinned slab: small first and last chunks (weights 1,2,3,..,3,2,1) for a short
//           fill and drain, 2.26-2.34 ms per 1 M-point skin call against 2.45 ms with equal chunks;
//   kind 3: staged pipeline with the speculative AEROBULK_INIT (jt == 1): H2D and D2H overlap, up to 12 equal pieces
//           with half-size first and last ones.
int plan_chunks(long long n, int kind, long long *cstart)
{
    int nchunks = 1;
    if (kind == 2) {
        nchunks = (int)((n + bounce_chunk_points() - 1) / bounce_chunk_points());
        nchunks = nchunks < 1 ? 1 : (nchunks > MAX_CHUNKS ? MAX_CHUNKS : nchunks);
    } else if (kind == 1) {
        nchunks = (int)(n / MIN_CHUNK_POINTS);
        nchunks = nchunks < 1 ? 1 : (nchunks > STAGED_CHUNKS ? STAGED_CHUNKS : nchunks);
    } else if (kind == 3) {
        nchunks = (int)(n / MIN_CHUNK_POINTS);
        nchunks = nchunks < 1 ? 1 : (nchunks > SPEC_CHUNKS ? SPEC_CHUNKS : nchunks);
    }
    double w[MAX_CHUNKS], wsum = 0.;
    for (int c = 0; c < nchunks; ++c) {
        if (kind == 2) w[c] = (double)((c + 1 < nchunks - c) ? c + 1 : nchunks - c);
        else if (kind == 3) w[c] = (c == 0 || c == nchunks - 1) ? 0.5 : 1.;   // both directions busy: equal pieces, short fill and drain
        else w[c] = (double)(nchunks - c);
        wsum += w[c];
    }
    double acc = 0.;
    cstart[0] = 0;
    for (int c = 0; c < nchunks; ++c) {
        acc += w[c];
        long long s0 = (long long)((double)n * acc / wsum);
        s0 = (s0 + 2047) / 2048 * 2048;
        cstart[c + 1] = s0 > n ? n : s0;
    }
    cstart[nchunks] = n;
    return nchunks;
}

// ---------------------------------------------------------------------------
// AEROBULK_MODEL (mod_aerobulk.f90:176-269) + aerobulk_compute dispatch
// ---------------------------------------------------------------------------
// the argument checks that come before any device work (:244), for one device and for a split call alike
int check_model_args(int jt, const char *calgo, int Ni, int Nj, const void *sst, const void *t_zt, const void *hum_zt,
                     const void *U_zu, const void *V_zu, const void *slp, const void *QL, const void *QH,
                     const void *Tau_x, const void *Tau_y, const void *Evap)
{
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!calgo || !sst || !t_zt || !hum_zt || !U_zu || !V_zu || !slp || !QL || !QH || !Tau_x || !Tau_y || !Evap)
        return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_model: NULL mandatory argument");
    if (Ni < 0 || Nj < 0) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_model: negative shape %d x %d", Ni, Nj);
    if (jt < 1) return fail(AEROBULK_GPU_ERR_JT, "AEROBULK_MODEL => jt < 1 !??\n we are in a Fortran world here...");
    return 0;
}

// `es`: bytes per element of every array of the call, sizeof(double) (aerobulk_gpu_model*) or sizeof(float)
// (aerobulk_gpu_model*_f32).  Only the kernels (abk::ELEM_F64 / ELEM_F32) and the byte counts of the copies depend on it:
// the transport path, the chunk plan, AEROBULK_INIT and the warm-layer state (always FP64) do not.
int model_impl(bool device_ptrs, size_t es, int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj,
               const void *sst, const void *t_zt, const void *hum_zt, const void *U_zu,
               const void *V_zu, const void *slp, void *QL, void *QH, void *Tau_x, void *Tau_y,
               void *Evap, const int *Niter, const int *l_use_skin, const void *rad_sw,
               const void *rad_lw, void *T_s)
{
    int rc = check_model_args(jt, calgo, Ni, Nj, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x, Tau_y, Evap);
    if (rc) return rc;
    if (Niter) g.nb_iter = *Niter;   // :236 sticky
    const bool lskin = l_use_skin ? (*l_use_skin != 0) : false;
    const bool lsrad = (rad_sw != nullptr) && (rad_lw != nullptr);

    rc = ensure_device();
    if (rc) return rc;
    const long long n = (long long)Ni * (long long)Nj;
    cudaStream_t cs = compute_stream();
    if (g.init_pending && !device_ptrs) {   // a host-array call is blocking anyway: catch up with an asynchronous AEROBULK_INIT
        rc = resolve_init();
        if (rc) return rc;
    }

    // a deferred wind-stress error of earlier asynchronous launches surfaces as soon as its flag
    // copy has landed (no synchronisation here: device-resident calls stay asynchronous)
    if (g.bad_pending && cudaEventQuery(g.ev_bad) == cudaSuccess) {
        rc = check_bad_flag(nullptr, nullptr);
        if (rc) return rc;
    }

    // rad_lw before rad_sw: a caller slab [sst .. slp, rad_lw] with a per-step rad_sw elsewhere is one run + one array
    auto in_p = [](const void *p) { return static_cast<const char *>(p); };
    auto out_p = [](void *p) { return static_cast<char *>(p); };
    const char *in_h[8] = {in_p(sst), in_p(t_zt), in_p(hum_zt), in_p(U_zu), in_p(V_zu), in_p(slp),
                           lsrad ? in_p(rad_lw) : nullptr, lsrad ? in_p(rad_sw) : nullptr};
    char *out_h[6] = {out_p(QL), out_p(QH), out_p(Tau_x), out_p(Tau_y), out_p(Evap), lsrad ? out_p(T_s) : nullptr};
    const char *in_d[8] = {};   // what the kernels read and write
    char *out_d[6] = {};
    const long long row = n * (long long)es;   // bytes per field

    // How the arrays reach the kernel, chosen once per call, in this order:
    //   DEVICE  device pointers (aerobulk_gpu_model_device): one launch on them;
    //   ALIAS   jt > 1 or AEROBULK_INIT already done, every array pinned: one launch on their device aliases, no sort;
    //   BOUNCE  jt > 1, pageable arrays of BOUNCE_MIN_POINTS or more, and the pinned slab fits: the copy threads move kind-2
    //           chunks between the caller's arrays and the slab, the kernel works on the slab zero-copy, no sort, and the
    //           outputs go home two chunks behind the GPU;
    //   STAGED  anything else: H2D | kernel | D2H through the device staging arrays, kind-1 chunks.
    // At jt == 1 with AEROBULK_INIT still to run the path is STAGED whatever the arrays, with kind-3 chunks; `spec_init`:
    // there are two or more of them and AEROBULK_INIT runs speculatively chunk by chunk (below), otherwise the statistics
    // are taken once all inputs are in.  `slab_first`: the arrays are pageable, BOUNCE_MIN_POINTS or more, and the pinned
    // slab fits, so the pipeline copies from / to the slab and the copy threads feed it -- chunk by chunk under
    // spec_init, otherwise whole.
    enum Path { DEVICE, ALIAS, BOUNCE, STAGED } path = device_ptrs ? DEVICE : STAGED;
    const bool init_stats = jt == 1 && !g.preinit_done;   // this call takes AEROBULK_INIT's field statistics
    const bool slab_ok = bounce_on() && zerocopy_on() && n >= BOUNCE_MIN_POINTS;   // the kernel reads the slab zero-copy
    auto alias_all = [&] {   // device aliases of every array into in_d / out_d; false at the first array without one
        for (int k = 0; k < 8; ++k)
            if (in_h[k] && !(in_d[k] = device_alias(in_h[k]))) return false;
        for (int k = 0; k < 6; ++k)
            if (out_h[k] && !(out_d[k] = device_alias(out_h[k]))) return false;
        return true;
    };
    bool slab_first = false;
    if (!device_ptrs && init_stats) {
        slab_first = slab_ok && !alias_all() && ensure_bounce(row);
    } else if (!device_ptrs) {
        if (n > 0 && zerocopy_on() && alias_all()) path = ALIAS;
        else if (slab_ok && ensure_bounce(row)) path = BOUNCE;
    }
    long long cstart[MAX_CHUNKS + 1];
    const int nchunks = plan_chunks(n, path == BOUNCE ? 2 : path == STAGED ? (init_stats ? 3 : 1) : 0, cstart);
    // Speculative AEROBULK_INIT (jt == 1 of a staged host-array call with >= 2 chunks).  The reference judges the WHOLE
    // fields before it computes anything, which would hold the first flux launch -- and every byte of D2H -- back until the
    // last input byte has arrived: H2D and D2H one after the other.  Instead each chunk's statistics are taken as it lands,
    // combined with those of the chunks before it and judged on the device (init_decide_kernel), and the chunk's flux
    // launch runs on that RUNNING verdict (humidity type; stop flag).  When the last chunk is in, the verdict is the
    // reference's; the few chunks (normally none) whose running verdict differed from it are recomputed from the staged
    // inputs, and an AEROBULK_INIT error is raised exactly as before -- the arrays the reference would never have
    // written are then undefined.  Same results, H2D and D2H overlapped: C5 end to end 0.54 -> ~1 Gpt/s.
    const bool spec_init = path == STAGED && init_stats && nchunks >= 2;

    // through the slab: the caller's arrays move to user_in / user_out, in_h / out_h name the slab rows
    char *user_in[8] = {}, *user_out[6] = {};
    if (slab_first || path == BOUNCE) {
        for (int k = 0; k < 8; ++k) {
            user_in[k] = const_cast<char *>(in_h[k]);
            in_h[k] = in_h[k] ? g.hb + (long long)k * g.cap_hb : nullptr;
        }
        for (int k = 0; k < 6; ++k) {
            user_out[k] = out_h[k];
            out_h[k] = out_h[k] ? g.hb + (long long)(8 + k) * g.cap_hb : nullptr;
        }
    }
    if (path == STAGED) {
        rc = ensure_staging(row);
        if (rc) return rc;
    }
    for (int k = 0; k < 8; ++k) {
        if (!in_h[k] || path == DEVICE) in_d[k] = in_h[k];
        else if (path == BOUNCE) in_d[k] = g.hb_dev + (long long)k * g.cap_hb;
        else if (path == STAGED) in_d[k] = g.d_in[k];
    }
    for (int k = 0; k < 6; ++k) {
        if (!out_h[k] || path == DEVICE) out_d[k] = out_h[k];
        else if (path == BOUNCE) out_d[k] = g.hb_dev + (long long)(8 + k) * g.cap_hb;
        else if (path == STAGED) out_d[k] = g.d_out[k];
    }

    if (slab_first && !spec_init) bounce_copy(8, user_in, 0, 0, n, es, true);
    // H2D of chunk c on the copy-in stream (preceded by its way into the slab on the copy threads where that applies)
    auto enqueue_h2d = [&](int c) -> int {
        const long long s0 = cstart[c], len = cstart[c + 1] - s0;
        if (len > 0 && path == STAGED) {
            if (slab_first && spec_init) bounce_copy(8, user_in, 0, s0, len, es, true);
            const int r = copy_fields(8, g.d_in, const_cast<char *const *>(in_h), g.cap, s0, len, es, true, g.in_stream);
            if (r) return r;
        }
        CUDA_TRY(cudaEventRecord(g.ev_in[c], g.in_stream));
        return 0;
    };
    int h2d_next = 0;   // first chunk whose H2D is not enqueued yet
    if (!device_ptrs) {
        // all of them up front, except where the copy threads feed the slab: there chunk c + 1 follows the launch of chunk c
        for (; h2d_next < (slab_first && spec_init ? 1 : nchunks); ++h2d_next) {
            rc = enqueue_h2d(h2d_next);
            if (rc) return rc;
        }
    }

    // ---- jt == 1: AEROBULK_INIT (needs global field statistics before any flux is computed)
    if (jt == 1) {
        if (g.preinit_done) {
            g.preinit_done = false;   // aerobulk_gpu_init_from_stats() already ran the global init
        } else {
            double st[abk::NSTATS];
            if (spec_init) {
                // staged host-array pipeline: see the chunk loop -- only the argument-dependent half runs here
                rc = init_flags(Nt, calgo, lskin, lsrad);
                if (rc) return rc;
            } else {
            if (!device_ptrs) CUDA_TRY(cudaStreamWaitEvent(cs, g.ev_in[nchunks - 1], 0));
            if (device_ptrs && !g.verbose && !g.stats_hook && n > 0) {
                // device-resident session, banners off: no host round trip -- the statistics stay on the device, are judged
                // there, and the flux kernel reads the verdict from device memory (init_async / resolve_init)
                rc = launch_local_stats(n, es, in_d[0], in_d[1], in_d[2], in_d[3], in_d[4], in_d[5], lsrad ? in_d[6] : nullptr, cs, g.d_stats);
                if (rc) return rc;
                rc = init_async(Nt, calgo, lskin, lsrad, g.d_stats, 1, Ni, Nj, cs);
                if (rc) return rc;
            } else {
            if (n > 0) {
                // :248 -- prsw=rad_lw: rad_lw is checked against both radiation ranges, rad_sw never
                rc = local_stats(n, es, in_d[0], in_d[1], in_d[2], in_d[3], in_d[4], in_d[5], lsrad ? in_d[6] : nullptr, cs, st);
                if (rc) return rc;
            } else {
                memset(st, 0, sizeof(st));
            }
            // aerobulk_gpu_set_devices(n): this session holds one shard; AEROBULK_INIT judges the whole field
            if (g.stats_hook && !g.stats_hook->combine(g.shard, st, true, st))
                return fail(AEROBULK_GPU_ERR_STATE, "AEROBULK_INIT => another device of the split call failed");
            rc = init_from_stats(Nt, calgo, lskin, lsrad, st, g.report_Ni > 0 ? g.report_Ni : Ni, g.report_Ni > 0 ? g.report_Nj : Nj);
            if (rc) return rc;
            }
            }
        }
    }

    // ---- aerobulk_compute (mod_aerobulk_compute.f90:22-213)
    const int ialgo = algo_id(calgo);
    if (!ialgo)
        return fail(AEROBULK_GPU_ERR_ALGO, "ERROR: mod_aerobulk_compute.f90 => bulk algorithm %s is unknown!!!", calgo);
    const bool use_skin = g.l_use_skin_schemes && has_skin_schemes(ialgo);
    if (use_skin && !lsrad)
        return fail(AEROBULK_GPU_ERR_SKIN_NORAD,
                    "skin schemes are active (l_use_skin_schemes is sticky, mod_aerobulk.f90:74) but rad_sw/rad_lw are absent");

    if (use_skin && jt == 1) {
        rc = init_wl_state(ialgo, n);
        if (rc) return rc;
    }
    if (use_skin) {
        const long long have = (ialgo == abd::ECMWF) ? g.n_ecmwf : g.n_coare;
        if (have != n || (jt > 1 && have == 0 && n > 0))
            return fail(AEROBULK_GPU_ERR_STATE, "warm-layer state missing or of another size at jt=%d (no jt==1 call for this session?)", jt);
    }

    // Stability sort (classify_kernel).  Auto policy = where it measured faster on B200 (kbench with KBENCH_SORT=1/2,
    // profiles/exp_sort_r02d.txt, 4320x2160): everything but NCAR (too little work per point: 0.97 -> 1.06 ms).  Since the
    // proxy follows the skin temperature (T_s starts 0.25 K below the SST and carries the warm-layer increment) and keeps
    // the doubtful points to themselves, ECMWF + skin gains the most (5.01 -> 4.54 ms by day, 4.46 -> 3.88 ms by night;
    // with the round-1 proxy it lost 1 %).
    // (never with zero-copy inputs: the gather through the permutation would cross PCIe at sector granularity)
    const bool do_sort = (path == DEVICE || path == STAGED) && (g.sort_points == 2 || (g.sort_points == 1 && ialgo != abd::NCAR));
    if (do_sort) {
        // every chunk is padded to whole sort windows
        const long long need = n + (long long)(nchunks + 1) * abk::sort_window();
        if (need > g.cap_perm) {
            if (g.d_perm) cudaFree(g.d_perm);
            g.d_perm = nullptr;
            g.cap_perm = 0;
            CUDA_TRY(cudaMalloc(&g.d_perm, sizeof(unsigned short) * (size_t)need));
            g.cap_perm = need;
        }
    }

    abk::FluxArgs a;
    memset(&a, 0, sizeof(a));
    a.u = make_uniform(zt, zu);
    a.ihum = g.ihum;
    a.init_dev = g.init_pending ? g.d_init : nullptr;
    a.first_step = (jt == 1);
    a.bad_index = g.d_bad;
    const bool zteq = zt_eq_zu(zt, zu);

    // the kernels of chunk c on the compute stream: classify (when sorting) and flux, on the chunk's row block of every
    // array and of the warm-layer state; `timed`: the flux launch between a pair of aerobulk_gpu_set_kernel_timing events
    auto launch_chunk = [&](int c, bool timed) -> int {
        const long long s0 = cstart[c];
        a.sst = elem_at(in_d[0], s0, es); a.t_zt = elem_at(in_d[1], s0, es); a.hum_zt = elem_at(in_d[2], s0, es);
        a.U_zu = elem_at(in_d[3], s0, es); a.V_zu = elem_at(in_d[4], s0, es); a.slp = elem_at(in_d[5], s0, es);
        a.rad_lw = elem_at(in_d[6], s0, es);
        a.rad_sw = elem_at(in_d[7], s0, es);
        a.QL = elem_at(out_d[0], s0, es); a.QH = elem_at(out_d[1], s0, es); a.Tau_x = elem_at(out_d[2], s0, es);
        a.Tau_y = elem_at(out_d[3], s0, es); a.Evap = elem_at(out_d[4], s0, es);
        a.T_s = elem_at(out_d[5], s0, es);
        if (use_skin) bind_wl_state(a, ialgo, s0);
        a.n = cstart[c + 1] - s0;
        a.index_offset = s0;
        a.perm = nullptr;
        if (do_sort) {
            unsigned short *perm = g.d_perm + s0 + (long long)c * abk::sort_window();
            CUDA_TRY(abk::launch_classify(es, a, perm, use_skin, cs));
            g.launches += 1;
            a.perm = perm;
        }
        cudaEvent_t kt0 = nullptr, kt1 = nullptr;
        if (timed && g.time_kernels) {
            if (g.kt_used + 2 > g.kt_ev.size()) {
                cudaEvent_t e0, e1;
                CUDA_TRY(cudaEventCreate(&e0));
                CUDA_TRY(cudaEventCreate(&e1));
                g.kt_ev.push_back(e0);
                g.kt_ev.push_back(e1);
            }
            kt0 = g.kt_ev[g.kt_used];
            kt1 = g.kt_ev[g.kt_used + 1];
            g.kt_used += 2;
            CUDA_TRY(cudaEventRecord(kt0, cs));
        }
        CUDA_TRY(abk::launch_flux(ialgo, use_skin, zteq, es, a, cs));
        g.launches += 1;
        if (kt1) CUDA_TRY(cudaEventRecord(kt1, cs));
        return 0;
    };
    // D2H of chunk c on the copy-out stream once its kernel is done (the zero-copy kernels have written the host already)
    auto enqueue_d2h = [&](int c) -> int {
        CUDA_TRY(cudaEventRecord(g.ev_k[c], cs));
        CUDA_TRY(cudaStreamWaitEvent(g.out_stream, g.ev_k[c], 0));
        if (path != STAGED) return 0;
        return copy_fields(6, g.d_out, out_h, g.cap, cstart[c], cstart[c + 1] - cstart[c], es, false, g.out_stream);
    };

    int launched[MAX_CHUNKS], n_launched = 0, n_home = 0;
    bool home[MAX_CHUNKS] = {};   // pageable jt == 1: chunk already copied back to the caller's arrays
    for (int c = 0; c < nchunks; ++c) {
        const long long s0 = cstart[c], len = cstart[c + 1] - s0;
        if (len <= 0) continue;
        if (path == BOUNCE) bounce_copy(8, user_in, 0, s0, len, es, true);
        while (slab_first && spec_init && h2d_next <= c) {   // (normally enqueued one iteration ahead, below)
            rc = enqueue_h2d(h2d_next++);
            if (rc) return rc;
        }
        if (!device_ptrs) CUDA_TRY(cudaStreamWaitEvent(cs, g.ev_in[c], 0));
        if (spec_init) {
            rc = launch_local_stats(len, es, elem_at(in_d[0], s0, es), elem_at(in_d[1], s0, es), elem_at(in_d[2], s0, es),
                                    elem_at(in_d[3], s0, es), elem_at(in_d[4], s0, es), elem_at(in_d[5], s0, es),
                                    lsrad ? elem_at(in_d[6], s0, es) : nullptr, cs, g.d_cstats + (long long)c * abk::NSTATS);
            if (rc) return rc;
            CUDA_TRY(abk::launch_init_decide(g.d_cstats, c + 1, lsrad ? 1 : 0, g.d_cgstats + (long long)c * abk::NSTATS,
                                             g.d_cinit + 2 * c, cs));
            g.launches += 1;
            a.init_dev = g.d_cinit + 2 * c;
        }
        rc = launch_chunk(c, true);
        if (rc) return rc;
        if (device_ptrs) continue;
        rc = enqueue_d2h(c);
        if (rc) return rc;
        if (slab_first && spec_init) {
            CUDA_TRY(cudaEventRecord(g.ev_out[c], g.out_stream));
            launched[n_launched++] = c;
            // the next chunk goes into the slab (and on to the device) while the GPU works on this one ...
            while (h2d_next < nchunks && h2d_next <= c + 1) {
                rc = enqueue_h2d(h2d_next++);
                if (rc) return rc;
            }
            // ... and the chunks whose results have landed in the slab go home
            while (n_home < n_launched && cudaEventQuery(g.ev_out[launched[n_home]]) == cudaSuccess) {
                const int h = launched[n_home++];
                bounce_copy(6, user_out, 8, cstart[h], cstart[h + 1] - cstart[h], es, false);
                home[h] = true;
            }
        }
        if (path == BOUNCE) {   // results of an earlier chunk go home while the GPU has two chunks queued
            launched[n_launched++] = c;
            if (n_launched - n_home > 2) {
                const int h = launched[n_home++];
                CUDA_TRY(cudaEventSynchronize(g.ev_k[h]));
                bounce_copy(6, user_out, 8, cstart[h], cstart[h + 1] - cstart[h], es, false);
            }
        }
    }
    if (spec_init) {
        // the reference's verdict (all chunks), then the chunks that ran on a different running verdict once more
        int cinit[2 * MAX_CHUNKS];
        double st[abk::NSTATS];
        CUDA_TRY(cudaMemcpyAsync(cinit, g.d_cinit, 2 * sizeof(int) * nchunks, cudaMemcpyDeviceToHost, cs));
        CUDA_TRY(cudaMemcpyAsync(st, g.d_cgstats + (long long)(nchunks - 1) * abk::NSTATS, sizeof(st), cudaMemcpyDeviceToHost, cs));
        CUDA_TRY(cudaStreamSynchronize(cs));
        // aerobulk_gpu_set_devices(n): the shards ran on their LOCAL running verdicts; the reference's verdict is the one
        // of the whole field -- the statistics of all devices, combined here
        if (g.stats_hook && !g.stats_hook->combine(g.shard, st, true, st)) {
            cudaStreamSynchronize(g.out_stream);
            return fail(AEROBULK_GPU_ERR_STATE, "AEROBULK_INIT => another device of the split call failed");
        }
        rc = init_checks(lsrad, st, g.report_Ni > 0 ? g.report_Ni : Ni, g.report_Ni > 0 ? g.report_Nj : Nj);
        if (rc) {
            cudaStreamSynchronize(g.out_stream);   // nothing may still be writing the caller's arrays when the call returns
            return rc;
        }
        a.init_dev = nullptr;
        a.ihum = g.ihum;
        for (int c = 0; c < nchunks; ++c) {
            if (cstart[c + 1] <= cstart[c] || (cinit[2 * c] == g.ihum && cinit[2 * c + 1] == 0)) continue;
            rc = launch_chunk(c, false);
            if (!rc) rc = enqueue_d2h(c);
            if (rc) return rc;
            home[c] = false;   // recomputed: what went home earlier is stale
        }
    }
    while (path == BOUNCE && n_home < n_launched) {
        const int h = launched[n_home++];
        CUDA_TRY(cudaEventSynchronize(g.ev_k[h]));
        bounce_copy(6, user_out, 8, cstart[h], cstart[h + 1] - cstart[h], es, false);
    }
    CUDA_TRY(cudaMemcpyAsync(g.h_bad, g.d_bad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaEventRecord(g.ev_bad, cs));
    g.bad_pending = true;
    g.pend_launches += 1;
    g.last_Ni = Ni;
    g.last_taux = out_d[2];
    g.last_tauy = out_d[3];
    g.last_es = es;

    const bool last = (jt == g.nitend);
    const bool never_sync = device_ptrs && g.async_device;   // the caller collects errors with aerobulk_gpu_synchronize()
    if (!never_sync && (!device_ptrs || last || (jt == 1 && !g.init_pending))) {
        CUDA_TRY(cudaStreamSynchronize(cs));
        if (!device_ptrs) CUDA_TRY(cudaStreamSynchronize(g.out_stream));
        if (slab_first) {   // what is not home yet (everything, without the chunk-wise feed)
            for (int c = 0; c < nchunks; ++c) {
                const long long s0 = cstart[c], len = cstart[c + 1] - s0;
                if (len > 0 && !home[c]) bounce_copy(6, user_out, 8, s0, len, es, false);
            }
        }
        rc = resolve_init();   // an asynchronous AEROBULK_INIT of this session reports first, as in the reference
        if (!rc) rc = check_bad_flag(device_ptrs ? nullptr : Tau_x, device_ptrs ? nullptr : Tau_y);
    }

    // kt == nitend -> *_EXIT frees the state (mod_blk_coare3p6.f90:411); jt == Nt -> AEROBULK_BYE (:267)
    if (use_skin && last) {
        if (ialgo == abd::ECMWF) release_ecmwf_state();
        else release_coare_state();
    }
    if (rc) return rc;
    if (jt == Nt && g.verbose) {
        printf(" ===================================================================\n");
        printf("                    ----- AeroBulk_bye -----\n");
        printf(" ===================================================================\n \n");
        fflush(stdout);
    }
    return 0;
}


// ---------------------------------------------------------------------------
// aerobulk_gpu_set_devices(n): ONE aerobulk_model call split over n GPUs inside the library (SURVEY.md 8b / 8e).
// The caller makes the reference's call -- whole (Ni,Nj) fields, host arrays, src/mod_aerobulk.f90:176-269 -- and the
// library partitions the flat point range into n contiguous shards (boundaries on multiples of 2048 points; for a
// 2-D field these are latitude row blocks up to that rounding), one per GPU, each with its own session: streams,
// staging, pinned bounce slab, warm-layer state, tau > 10 flag.  Points are independent, so there is no data-path
// exchange; the only combine is AEROBULK_INIT's field statistics at jt == 1 (StatsHook, in host memory: the devices
// belong to one process).  Device 0's shard runs on the calling thread, the others on persistent host threads.
// ---------------------------------------------------------------------------
class DeviceThreads
{
  public:
    // runs job(d) for d = 1 .. n-1 on the worker of session d and job(0) on the caller; returns when all are done
    template <class F>
    void run(int n, F &&job)
    {
        while ((int)started_ < n - 1) {
            const int d = ++started_;
            std::thread([this, d] { work(d); }).detach();   // never joined: the library is linked -z nodelete
        }
        {
            std::lock_guard<std::mutex> lk(mu_);
            job_ = [&job](int d) { job(d); };
            active_ = n;
            pending_ = n - 1;
            ++gen_;
        }
        cv_.notify_all();
        job(0);
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [&] { return pending_ == 0; });
        job_ = nullptr;
    }

  private:
    void work(int d)
    {
        cur = &sess[d];
        unsigned long long seen = 0;
        for (;;) {
            std::function<void(int)> job;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return gen_ != seen; });
                seen = gen_;
                if (d >= active_) continue;
                job = job_;
            }
            job(d);
            {
                std::lock_guard<std::mutex> lk(mu_);
                --pending_;
            }
            done_.notify_all();
        }
    }
    std::mutex mu_;
    std::condition_variable cv_, done_;
    std::function<void(int)> job_;
    unsigned long long gen_ = 0;
    int active_ = 0, pending_ = 0;
    int started_ = 0;
};
DeviceThreads &device_threads()
{
    static DeviceThreads *t = new DeviceThreads();   // never destroyed, like the copy threads
    return *t;
}

// shard boundaries of the last split call (state get / set, tests)
int split_nd = 1;
long long split_start[MAX_DEVICES + 1] = {0, 0};

int plan_shards(long long n, int nd_max, long long *start)
{
    int nd = nd_max < 1 ? 1 : (nd_max > MAX_DEVICES ? MAX_DEVICES : nd_max);
    long long per = (n + nd - 1) / nd;
    per = (per + 2047) / 2048 * 2048;
    if (per < 2048) per = 2048;
    nd = (int)((n + per - 1) / per);
    if (nd < 1) nd = 1;
    for (int d = 0; d <= nd; ++d) start[d] = (long long)d * per < n ? (long long)d * per : n;
    start[nd] = n;
    return nd;
}

int model_multi(size_t es, int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj, const void *sst,
                const void *t_zt, const void *hum_zt, const void *U_zu, const void *V_zu, const void *slp,
                void *QL, void *QH, void *Tau_x, void *Tau_y, void *Evap, const int *Niter,
                const int *l_use_skin, const void *rad_sw, const void *rad_lw, void *T_s)
{
    Session &s0 = sess[0];
    int rc = check_model_args(jt, calgo, Ni, Nj, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x, Tau_y, Evap);
    if (rc) return rc;
    rc = ensure_device();   // session 0: resolves its device id
    if (rc) return rc;
    int count = 0;
    CUDA_TRY(cudaGetDeviceCount(&count));
    const long long n = (long long)Ni * Nj;
    long long start[MAX_DEVICES + 1];
    const int nd = plan_shards(n, n_devices < count ? n_devices : count, start);
    for (int d = 0; d < nd; ++d)
        if (start[d + 1] - start[d] > 0x7fffffffLL) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_model: shard %d has more than 2^31 points", d);
    if (s0.use_user_stream)
        return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_set_devices(n > 1) and aerobulk_gpu_set_stream are exclusive: each device runs on a stream of the library");
    // a session keeps the shard it was given at jt == 1
    if (jt > 1 && (s0.n_coare || s0.n_ecmwf) && nd != split_nd)
        return fail(AEROBULK_GPU_ERR_STATE, "the number of devices changed inside a warm-layer session");
    // session-wide settings (the SAVEd module variables of mod_const.f90:22-33 exist once) follow session 0
    for (int d = 1; d < nd; ++d) {
        Session &sd = sess[d];
        const int want = (s0.device + d) % count;
        if (sd.device_ready && sd.device != want)
            return fail(AEROBULK_GPU_ERR_ARG, "device %d of the split is bound to GPU %d, not %d: call aerobulk_gpu_reset()", d, sd.device, want);
        sd.device = want;
        sd.nb_iter = s0.nb_iter; sd.nitend = s0.nitend; sd.l_use_skin_schemes = s0.l_use_skin_schemes; sd.ihum = s0.ihum;
        sd.rdt = s0.rdt; sd.gdept = s0.gdept; sd.error_mode = s0.error_mode; sd.verbose = 0; sd.sort_points = s0.sort_points;
        sd.preinit_done = s0.preinit_done;
    }
    static StatsHook hook;
    const bool need_stats = (jt == 1) && !s0.preinit_done;
    if (need_stats) hook.reset(nd);
    int rcs[MAX_DEVICES] = {};
    device_threads().run(nd, [&](int d) {
        Session &sd = sess[d];
        sd.shard = d;
        sd.flat_offset = start[d];
        sd.report_Ni = Ni;
        sd.report_Nj = Nj;
        sd.stats_hook = need_stats ? &hook : nullptr;
        const long long o = start[d];
        const int len = (int)(start[d + 1] - o);
        auto in = [&](const void *p) { return elem_at(static_cast<const char *>(p), o, es); };
        auto out = [&](void *p) { return elem_at(static_cast<char *>(p), o, es); };
        rcs[d] = model_impl(false, es, jt, Nt, calgo, zt, zu, len, 1, in(sst), in(t_zt), in(hum_zt), in(U_zu), in(V_zu), in(slp),
                            out(QL), out(QH), out(Tau_x), out(Tau_y), out(Evap), Niter, l_use_skin, in(rad_sw), in(rad_lw),
                            out(T_s));
        if (need_stats && rcs[d]) hook.combine(d, nullptr, false, nullptr);   // failed before the rendezvous: release the others
        sd.stats_hook = nullptr;
    });
    split_nd = nd;
    for (int d = 0; d <= nd; ++d) split_start[d] = start[d];
    // the reference would have stopped at the first error: report the one of the lowest shard that is not the echo of another's
    int first = -1;
    for (int d = 0; d < nd && first < 0; ++d)
        if (rcs[d] && !(rcs[d] == AEROBULK_GPU_ERR_STATE && strstr(sess[d].errmsg, "another device of the split call failed"))) first = d;
    for (int d = 0; d < nd && first < 0; ++d)
        if (rcs[d]) first = d;
    for (int d = 0; d < nd; ++d) {
        sess[d].report_Ni = sess[d].report_Nj = 0;
        sess[d].flat_offset = 0;
    }
    if (first < 0) return 0;
    if (first != 0) {
        memcpy(s0.errmsg, sess[first].errmsg, sizeof(s0.errmsg));
        s0.errcode = sess[first].errcode;
    }
    return rcs[first];
}


// Return-code mode only (the default fail-stop mode never gets here: fail() has ended the process).  The reference
// would have STOPped: whatever session was open is over.  The warm-layer state is released on every device and a skin
// flag switched on by the failed jt == 1 call is rolled back, so that the next jt == 1 call starts clean.
void end_session_after_error(int jt, bool skin_before)
{
    for (int d = 0; d < MAX_DEVICES; ++d) {
        sess[d].n_coare = sess[d].n_ecmwf = 0;
        sess[d].preinit_done = false;
        sess[d].init_pending = false;
        if (jt == 1) sess[d].l_use_skin_schemes = skin_before;
    }
}

// host-array AEROBULK_MODEL: one device, or split over aerobulk_gpu_set_devices(n) of them
int model_host(size_t es, int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj, const void *sst,
               const void *t_zt, const void *hum_zt, const void *U_zu, const void *V_zu, const void *slp,
               void *QL, void *QH, void *Tau_x, void *Tau_y, void *Evap, const int *Niter,
               const int *l_use_skin, const void *rad_sw, const void *rad_lw, void *T_s)
{
    const bool skin_before = sess[0].l_use_skin_schemes;
    int rc;
    if (n_devices > 1) {
        rc = model_multi(es, jt, Nt, calgo, zt, zu, Ni, Nj, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x, Tau_y, Evap,
                         Niter, l_use_skin, rad_sw, rad_lw, T_s);
    } else {
        split_nd = 1;
        rc = model_impl(false, es, jt, Nt, calgo, zt, zu, Ni, Nj, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x, Tau_y, Evap,
                        Niter, l_use_skin, rad_sw, rad_lw, T_s);
    }
    if (rc) end_session_after_error(jt, skin_before);
    return rc;
}

// device-pointer AEROBULK_MODEL (one device)
int model_device(size_t es, int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj, const void *sst,
                 const void *t_zt, const void *hum_zt, const void *U_zu, const void *V_zu, const void *slp,
                 void *QL, void *QH, void *Tau_x, void *Tau_y, void *Evap, const int *Niter,
                 const int *l_use_skin, const void *rad_sw, const void *rad_lw, void *T_s)
{
    const bool skin_before = sess[0].l_use_skin_schemes;
    const int rc = model_impl(true, es, jt, Nt, calgo, zt, zu, Ni, Nj, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x,
                              Tau_y, Evap, Niter, l_use_skin, rad_sw, rad_lw, T_s);
    if (rc) end_session_after_error(jt, skin_before);
    return rc;
}

// device slab of the staged host-array calls and of device-only scratch (grow-only)
int ensure_turb_slab(long long need)
{
    if (need > g.cap_turb) {
        if (g.d_turb) cudaFree(g.d_turb);
        g.d_turb = nullptr;
        g.cap_turb = 0;
        if (need > 0) CUDA_TRY(cudaMalloc(&g.d_turb, sizeof(double) * (size_t)need));
        g.cap_turb = need;
    }
    return 0;
}

// ---------------------------------------------------------------------------
// Caller arrays of the entry points other than aerobulk_gpu_model (turb, series, turb_ice, oce_ice, series_ice).  The
// entry point registers each array with its length and role and asks for device-only scratch; open() stores a device
// pointer in every registered slot, close() brings the outputs home.  open() picks the first mode that applies:
//   DEVICE  the caller passed device pointers: they pass through, nothing moves, close() does nothing;
//   ALIAS   every array is pinned (cudaHostAlloc / cudaHostRegister) and zerocopy_on(): the kernel works on the
//           caller's memory through its device aliases;
//   BOUNCE  from BOUNCE_MIN_POINTS elements up, the copy threads pack the inputs into the pinned slab g.hx, the kernel
//           works on the slab zero-copy and the copy threads bring the outputs home (pageable cudaMemcpy is staged by
//           the driver on one thread at ~14 GB/s; the copy threads move 55-70 GB/s);
//   STAGED  cudaMemcpyAsync through the device slab g.d_turb on the compute stream.
// The three host modes block in close().  Scratch lives in g.d_turb in every mode.
// ---------------------------------------------------------------------------
struct HostTransport {
    enum Mode { DEVICE, ALIAS, BOUNCE, STAGED };
    struct Array {
        double **slot;          // receives the device pointer
        double *host;           // the caller's pointer; NULL: absent (the slot gets NULL)
        long long len, off;     // elements; offset in the packed slab
        bool in, home;          // copied in before the launch / home after it
        double *dev;            // what open() stores in the slot
    };
    std::vector<Array> arrays, scratch_rows;
    Mode mode = DEVICE;

    void in(const double **slot, const double *h, long long len)
    {
        arrays.push_back({const_cast<double **>(slot), const_cast<double *>(h), len, 0, true, false, nullptr});
    }
    void out(double **slot, double *h, long long len, bool home = true) { arrays.push_back({slot, h, len, 0, false, home, nullptr}); }
    void inout(double **slot, double *h, long long len, bool home) { arrays.push_back({slot, h, len, 0, true, home, nullptr}); }
    void scratch(double **slot, long long len) { scratch_rows.push_back({slot, nullptr, len, 0, false, false, nullptr}); }

    Mode pick(long long total, long long longest)
    {
        if (!zerocopy_on()) return STAGED;
        bool pinned = true;
        for (Array &a : arrays)
            if (a.host && !(a.dev = device_alias(a.host))) {
                pinned = false;
                break;
            }
        if (pinned) return ALIAS;
        if (!bounce_on() || longest < BOUNCE_MIN_POINTS || sizeof(double) * (size_t)total > bounce_max_bytes() ||
            !grow_mapped(g.hx, g.hx_dev, g.cap_hx, total, 1))
            return STAGED;
        return BOUNCE;
    }
    // the copy threads move every array with `in` (to the slab) or `home` (from it)
    void bounce(bool to_slab)
    {
        std::vector<CopyPiece> pieces;
        for (const Array &a : arrays)
            if (a.host && (to_slab ? a.in : a.home)) {
                if (to_slab) add_pieces(pieces, g.hx + a.off, a.host, sizeof(double) * (size_t)a.len);
                else add_pieces(pieces, a.host, g.hx + a.off, sizeof(double) * (size_t)a.len);
            }
        pool_run(pieces.data(), (int)pieces.size());
    }
    int open(int on_device)
    {
        long long total = 0, longest = 0;
        for (Array &a : arrays) {
            const long long m = (a.host && a.len > 0) ? a.len : 0;
            a.off = total;
            total += (m + 63) / 64 * 64;   // rows start on 512-byte boundaries
            longest = m > longest ? m : longest;
        }
        mode = on_device ? DEVICE : pick(total, longest);
        long long need = mode == STAGED ? total : 0;
        for (Array &s : scratch_rows) {
            s.off = need;
            need += (s.len + 63) / 64 * 64;
        }
        const int rc = ensure_turb_slab(need);
        if (rc) return rc;
        for (Array &s : scratch_rows) *s.slot = g.d_turb + s.off;
        for (Array &a : arrays) {
            if (!a.host || mode == DEVICE) a.dev = a.host;
            else if (mode == BOUNCE) a.dev = g.hx_dev + a.off;
            else if (mode == STAGED) a.dev = g.d_turb + a.off;
            if (mode == STAGED && a.host && a.in && a.len > 0)
                CUDA_TRY(cudaMemcpyAsync(a.dev, a.host, sizeof(double) * (size_t)a.len, cudaMemcpyHostToDevice, compute_stream()));
            *a.slot = a.dev;
        }
        if (mode == BOUNCE) bounce(true);
        return 0;
    }
    int close()
    {
        if (mode == DEVICE) return 0;
        if (mode == STAGED)
            for (const Array &a : arrays)
                if (a.host && a.home && a.len > 0)
                    CUDA_TRY(cudaMemcpyAsync(a.host, a.dev, sizeof(double) * (size_t)a.len, cudaMemcpyDeviceToHost, compute_stream()));
        CUDA_TRY(cudaStreamSynchronize(compute_stream()));
        if (mode == BOUNCE) bounce(false);
        return 0;
    }
};

// ---------------------------------------------------------------------------
// TURB_* (SURVEY.md 8f row 1)
// ---------------------------------------------------------------------------
int turb_impl(const char *calgo, int kt, double zt, double zu, int Ni, int Nj, double *T_s, const double *t_zt,
              double *q_s, const double *q_zt, const double *U_zu, int l_use_cs, int l_use_wl, double *Cd, double *Ch,
              double *Ce, double *t_zu, double *q_zu, double *Ubzu, const double *Qsw, const double *rad_lw,
              const double *slp, int isecday_utc, const double *plong, const aerobulk_gpu_turb_optional *opt,
              int on_device)
{
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!calgo || !T_s || !t_zt || !q_s || !q_zt || !U_zu || !Cd || !Ch || !Ce || !t_zu || !q_zu || !Ubzu)
        return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_turb: NULL mandatory argument");
    const int ialgo = algo_id(calgo);
    if (!ialgo) return fail(AEROBULK_GPU_ERR_ALGO, "aerobulk_gpu_turb: bulk algorithm %s is unknown!!!", calgo);
    if (!has_skin_schemes(ialgo) && (l_use_cs || l_use_wl))
        return fail(AEROBULK_GPU_ERR_SKIN_ALGO, "aerobulk_gpu_turb: TURB_%s has no cool-skin / warm-layer option", calgo);
    const bool cs = l_use_cs != 0, wl = l_use_wl != 0;
    // mod_blk_coare3p6.f90:263-269, mod_blk_ecmwf.f90:202-206
    if (cs && !(Qsw && rad_lw && slp))
        return fail(AEROBULK_GPU_ERR_SKIN_NORAD, "[turb_%s] => you need to provide Qsw, rad_lw & slp to use cool-skin param!", calgo);
    if (wl && !(Qsw && rad_lw && slp && (ialgo == abd::ECMWF || plong)))
        return fail(AEROBULK_GPU_ERR_SKIN_NORAD,
                    "[turb_%s] => you need to provide Qsw, rad_lw, slp, isecday_utc & plong to use warm-layer param!", calgo);
    int rc = ensure_device();
    if (rc) return rc;
    rc = resolve_init();
    if (rc) return rc;
    const long long n = (long long)Ni * Nj;
    cudaStream_t cs_ = compute_stream();

    if (wl && kt == 1) {
        rc = init_wl_state(ialgo, n);
        if (rc) return rc;
    }
    if (wl) {
        const long long have = (ialgo == abd::ECMWF) ? g.n_ecmwf : g.n_coare;
        if (have != n || n == 0) return fail(AEROBULK_GPU_ERR_STATE, "warm-layer state missing or of another size at kt=%d", kt);
    }

    abk::TurbArgs a;
    memset(&a, 0, sizeof(a));
    a.u = make_uniform(zt, zu);
    a.u.isd = isecday_utc;
    a.u.dawn = abd::wl_coare_dawn(0., isecday_utc) ? 1 : 0;
    a.n = n;
    a.first_step = (kt == 1);
    double *optp[10] = {nullptr};
    static_assert(sizeof(aerobulk_gpu_turb_optional) == 10 * sizeof(double *), "10 optional outputs");
    if (opt) memcpy(optp, opt, sizeof(*opt));
    HostTransport t;
    t.inout(&a.T_s, T_s, n, cs || wl);   // T_s, q_s come back only from the skin schemes
    t.inout(&a.q_s, q_s, n, cs || wl);
    t.in(&a.t_zt, t_zt, n); t.in(&a.q_zt, q_zt, n); t.in(&a.U_zu, U_zu, n);
    t.in(&a.Qsw, Qsw, n); t.in(&a.rad_lw, rad_lw, n); t.in(&a.slp, slp, n); t.in(&a.lon, plong, n);
    t.out(&a.Cd, Cd, n); t.out(&a.Ch, Ch, n); t.out(&a.Ce, Ce, n); t.out(&a.t_zu, t_zu, n); t.out(&a.q_zu, q_zu, n);
    t.out(&a.Ubzu, Ubzu, n);
    for (int k = 0; k < 10; ++k) t.out(&a.opt[k], optp[k], n);
    rc = t.open(on_device);
    if (rc) return rc;
    if (wl) bind_wl_state(a, ialgo, 0);
    CUDA_TRY(abk::launch_turb(ialgo, cs, wl, zt_eq_zu(zt, zu), a, cs_));
    g.launches += 1;
    rc = t.close();
    if (rc) return rc;
    // kt == nitend -> *_EXIT
    if (wl && kt == g.nitend) {
        CUDA_TRY(cudaStreamSynchronize(cs_));
        if (ialgo == abd::ECMWF) release_ecmwf_state();
        else release_coare_state();
    }
    return 0;
}

// ---------------------------------------------------------------------------
// station time series (SURVEY.md 8f row 3): one launch for the whole series
// ---------------------------------------------------------------------------
int series_impl(const char *calgo, int Nt, long long S, double zt, double zu, const int *isd, const double *lon,
                const double *sst, const double *t_zt, const double *hum_zt, int hum_kind, const double *wind,
                const double *slp, const double *rad_sw, const double *rad_lw, int l_use_skin,
                const aerobulk_gpu_series_out *out, int on_device)
{
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!calgo || !isd || !lon || !sst || !t_zt || !hum_zt || !wind || !slp || !rad_sw || !rad_lw || !out)
        return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_series: NULL mandatory argument");
    if (Nt < 0 || S < 0 || hum_kind < 0 || hum_kind > 2)
        return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_series: bad Nt=%d, S=%lld or hum_kind=%d", Nt, S, hum_kind);
    const int ialgo = algo_id(calgo);
    if (!ialgo) return fail(AEROBULK_GPU_ERR_ALGO, "aerobulk_gpu_series: bulk algorithm %s is unknown!!!", calgo);
    const bool skin = l_use_skin && has_skin_schemes(ialgo);
    int rc = ensure_device();
    if (rc) return rc;
    const long long n = (long long)Nt * S;
    if (n == 0) return 0;
    cudaStream_t cs_ = compute_stream();
    rc = deferred_errors();   // of earlier asynchronous aerobulk_gpu_model_device calls
    if (rc) return rc;

    double *const hout[abk::NSERIES_OUT] = {
        out->rho_zu, out->QL, out->QH, out->Qlw, out->QNS, out->Qsw, out->dT_cs, out->dT_wl, out->TAU, out->dT,
        out->Hz_wl, out->Qnt_ac, out->Tau_ac, out->Cd, out->Ce, out->Ch, out->theta_zu, out->q_zu, out->t_zu,
        out->RiB, out->z0, out->u_star, out->L, out->UN10, out->Ts, out->Evap, out->q_zt, out->theta_zt};

    abk::SeriesArgs a;
    memset(&a, 0, sizeof(a));
    a.S = S;
    a.Nt = Nt;
    a.hum_kind = hum_kind;
    a.u = make_uniform(zt, zu);
    a.bad_index = g.d_bad;

    HostTransport t;
    double *d_isd;   // isecday_utc is a host array in every mode
    t.scratch(&d_isd, ((long long)Nt * (long long)sizeof(int) + 7) / 8);
    t.in(&a.lon, lon, S);
    t.in(&a.sst, sst, n); t.in(&a.t_zt, t_zt, n); t.in(&a.hum_zt, hum_zt, n); t.in(&a.wnd, wind, n); t.in(&a.slp, slp, n);
    t.in(&a.rad_sw, rad_sw, n); t.in(&a.rad_lw, rad_lw, n);
    for (int k = 0; k < abk::NSERIES_OUT; ++k) t.out(&a.out[k], hout[k], n);
    rc = t.open(on_device);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(d_isd, isd, sizeof(int) * (size_t)Nt, cudaMemcpyHostToDevice, cs_));
    a.isd = reinterpret_cast<const int *>(d_isd);
    CUDA_TRY(abk::launch_series(ialgo, skin, zt_eq_zu(zt, zu), a, cs_));
    g.launches += 1;
    CUDA_TRY(cudaMemcpyAsync(g.h_bad, g.d_bad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, cs_));
    rc = t.close();
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(cs_));
    const unsigned long long bad = *g.h_bad;
    if (bad != ~0ull) {
        *g.h_bad = ~0ull;
        cudaMemsetAsync(g.d_bad, 0xFF, sizeof(unsigned long long), cs_);
        return fail(AEROBULK_GPU_ERR_TAU,
                    "BULK_FORMULA_VCTR()@mod_phymbl: wind stress too strong!\n  => at record %lld, station %lld",
                    (long long)(bad / (unsigned long long)S) + 1, (long long)(bad % (unsigned long long)S) + 1);
    }
    return 0;
}

// ---------------------------------------------------------------------------
// one station, CSV in / CSV out: src/tests/test_aerobulk_buoy_series_oce.f90 with text files for NetCDF
// ---------------------------------------------------------------------------
std::vector<std::string> split_csv(const std::string &line)
{
    std::vector<std::string> out;
    std::string cur;
    for (char ch : line) {
        if (ch == ',') {
            out.push_back(cur);
            cur.clear();
        } else if (ch != '\r' && ch != '\n' && ch != '"') {
            cur.push_back(ch);
        }
    }
    out.push_back(cur);
    for (auto &f : out) {
        size_t b = f.find_first_not_of(" \t"), e = f.find_last_not_of(" \t");
        f = (b == std::string::npos) ? std::string() : f.substr(b, e - b + 1);
    }
    return out;
}

// "YYYY?MM?DD?hh?mm[?ss]" with any non-digit separators -> hh*3600 + mm*60 (the program drops the seconds, :373)
bool parse_isecday(const std::string &t, int *isd)
{
    int f[6] = {0, 0, 0, 0, 0, 0}, nf = 0;
    size_t i = 0;
    while (i < t.size() && nf < 6) {
        if (t[i] >= '0' && t[i] <= '9') {
            long v = 0;
            while (i < t.size() && t[i] >= '0' && t[i] <= '9') v = v * 10 + (t[i++] - '0');
            f[nf++] = (int)v;
        } else {
            ++i;
        }
    }
    if (nf < 5 || f[3] > 23 || f[4] > 59) return false;
    *isd = f[3] * 3600 + f[4] * 60;
    return true;
}

// TO_KELVIN_3D, src/mod_phymbl.f90:1826-1847
int to_kelvin(std::vector<double> &v, const char *name)
{
    double sum = 0.;
    for (double x : v) sum += x;
    const double zm = sum / (double)v.size();
    if (zm < 50. && zm > -80.) {
        for (double &x : v) x = x + 273.15;
        return 0;
    }
    if (zm > 200. && zm < 320.) return 0;
    return fail(AEROBULK_GPU_ERR_UNITS, " *** PROBLEM: cannot figure out unit of variable %s !!!", name);
}

int series_csv_impl(const char *path_in, const char *path_out, const char *calgo, double zt, double zu, int l_use_skin)
{
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!path_in || !path_out || !calgo) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_series_csv: NULL argument");
    if (!algo_id(calgo)) return fail(AEROBULK_GPU_ERR_ALGO, "aerobulk_gpu_series_csv: bulk algorithm %s is unknown!!!", calgo);
    std::ifstream in(path_in);
    if (!in) return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: cannot open %s", path_in);
    std::string line;
    do {
        if (!std::getline(in, line)) return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: %s is empty", path_in);
    } while (line.empty() || line[0] == '#');
    std::vector<std::string> names = split_csv(line);
    auto col = [&](const char *nm) {
        for (size_t k = 0; k < names.size(); ++k) {
            std::string low = names[k];
            for (char &c : low) c = (char)tolower((unsigned char)c);
            if (low == nm) return (int)k;
        }
        return -1;
    };
    // the reference's default variable names, src/mod_const.f90:208-220
    const int c_time = col("time"), c_lon = col("lon"), c_sst = col("sst"), c_ta = col("t_air"), c_q = col("q_air"),
              c_rh = col("rh_air"), c_dp = col("dp_air"), c_w = col("wndspd"), c_u = col("u10"), c_v = col("v10"),
              c_p = col("msl"), c_sw = col("ssrd"), c_lw = col("strd");
    if (c_time < 0 || c_sst < 0 || c_ta < 0 || c_p < 0 || c_sw < 0 || c_lw < 0)
        return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: %s needs the columns time, sst, t_air, msl, ssrd, strd", path_in);
    const int hum_kind = (c_q >= 0) ? 0 : (c_rh >= 0) ? 2 : (c_dp >= 0) ? 1 : -1;
    if (hum_kind < 0) return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: %s needs one of q_air, rh_air, dp_air", path_in);
    const int c_hum = hum_kind == 0 ? c_q : hum_kind == 2 ? c_rh : c_dp;
    if (c_w < 0 && (c_u < 0 || c_v < 0))
        return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: %s needs wndspd, or u10 and v10", path_in);

    std::vector<std::string> stamp;
    std::vector<int> isd;
    std::vector<double> sst, ta, hum, wnd, slp, rsw, rlw;
    double lon = 0.;
    long lineno = 1;
    while (std::getline(in, line)) {
        ++lineno;
        if (line.empty() || line[0] == '#' || line.find_first_not_of(" \t\r") == std::string::npos) continue;
        std::vector<std::string> f = split_csv(line);
        if (f.size() < names.size())
            return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: %s line %ld has %zu fields, header has %zu", path_in,
                        lineno, f.size(), names.size());
        int sd = 0;
        if (!parse_isecday(f[c_time], &sd))
            return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: %s line %ld: cannot read the time '%s'", path_in, lineno,
                        f[c_time].c_str());
        bool ok = true;
        auto num = [&](int c) {
            char *end = nullptr;
            const double v = strtod(f[c].c_str(), &end);
            if (end == f[c].c_str()) ok = false;
            return v;
        };
        stamp.push_back(f[c_time]);
        isd.push_back(sd);
        sst.push_back(num(c_sst));
        ta.push_back(num(c_ta));
        hum.push_back(num(c_hum));
        if (c_w >= 0) {
            wnd.push_back(num(c_w));
        } else {
            const double u = num(c_u), v = num(c_v);
            wnd.push_back(sqrt(u * u + v * v));   // :206 (no FMA on the host build: -ffp-contract is off for .cu host code)
        }
        slp.push_back(num(c_p));
        rsw.push_back(num(c_sw));
        rlw.push_back(num(c_lw));
        if (stamp.size() == 1 && c_lon >= 0) lon = num(c_lon);
        if (!ok) return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: %s line %ld: not a number", path_in, lineno);
    }
    const int Nt = (int)stamp.size();
    if (Nt == 0) return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: %s holds no record", path_in);
    int rc = to_kelvin(ta, "t_air");   // :212
    if (rc) return rc;
    rc = to_kelvin(sst, "sst");        // :299
    if (rc) return rc;

    std::vector<std::vector<double>> o(abk::NSERIES_OUT, std::vector<double>((size_t)Nt));
    aerobulk_gpu_series_out out = {o[0].data(), o[1].data(), o[2].data(), o[3].data(), o[4].data(), o[5].data(), o[6].data(),
                                   o[7].data(), o[8].data(), o[9].data(), o[10].data(), o[11].data(), o[12].data(),
                                   o[13].data(), o[14].data(), o[15].data(), o[16].data(), o[17].data(), o[18].data(),
                                   o[19].data(), o[20].data(), o[21].data(), o[22].data(), o[23].data(), o[24].data(),
                                   o[25].data(), o[26].data(), o[27].data()};
    rc = series_impl(calgo, Nt, 1, zt, zu, isd.data(), &lon, sst.data(), ta.data(), hum.data(), hum_kind, wnd.data(),
                     slp.data(), rsw.data(), rlw.data(), l_use_skin, &out, 0);
    if (rc) return rc;

    FILE *fo = fopen(path_out, "w");
    if (!fo) return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: cannot write %s", path_out);
    // names of src/tests/test_aerobulk_buoy_series_oce.f90:539-577, then the extras
    static const char *onames[abk::NSERIES_OUT] = {"rho_a", "Qlat", "Qsen", "Qlw", "QNS", "Qsw", "dTcs", "dTwl", "Tau", "dT",
                                                    "H_wl", "Qnt_ac", "Tau_ac", "Cd", "Ce", "Ch", "theta_zu", "q_zu",
                                                    "t_zu", "RiB", "z0", "u_star", "L", "UN10", "Ts", "Evap", "q_zt",
                                                    "theta_zt"};
    fprintf(fo, "time,isecday_utc,Wind");
    for (int k = 0; k < abk::NSERIES_OUT; ++k) fprintf(fo, ",%s", onames[k]);
    fprintf(fo, "\n");
    for (int jt = 0; jt < Nt; ++jt) {
        fprintf(fo, "%s,%d,%.17g", stamp[jt].c_str(), isd[jt], wnd[jt]);
        for (int k = 0; k < abk::NSERIES_OUT; ++k) fprintf(fo, ",%.17g", o[k][jt]);
        fprintf(fo, "\n");
    }
    if (fclose(fo) != 0) return fail(AEROBULK_GPU_ERR_IO, "aerobulk_gpu_series_csv: error writing %s", path_out);
    return 0;
}

// ---------------------------------------------------------------------------
// sea ice (SURVEY.md 8f row 4)
// ---------------------------------------------------------------------------
int ice_algo_id(const char *c)
{
    if (!strcmp(c, "nemo")) return abd::ICE_NEMO;
    if (!strcmp(c, "easy")) return abd::ICE_EASY;
    if (!strcmp(c, "an05")) return abd::ICE_AN05;
    if (!strcmp(c, "lu12")) return abd::ICE_LU12;
    if (!strcmp(c, "lg15") || !strcmp(c, "lg15_io")) return abd::ICE_LG15;
    return 0;
}

abd::IceUniform make_ice_uniform(double zt, double zu, const double *cxn)
{
    abd::IceUniform u;
    memset(&u, 0, sizeof(u));
    u.zt = zt;
    u.zu = zu;
    u.log_zu = log(zu);
    u.log_ztu = log(zt / zu);
    u.log_zu10 = log(zu / 10.);
    if (cxn) {
        u.cxn[0] = cxn[0]; u.cxn[1] = cxn[1]; u.cxn[2] = cxn[2];
        u.sqrt_cdn = sqrt(cxn[0]);
    }
    const double r = 1. / log(zu / abd::RZ0_I_S_0);                 // Cd_from_z0, mod_phymbl.f90:1396-1414
    u.cdn_s = abd::VKARMN2 * r * r;
    u.chn_s = abd::VKARMN2 / (log(zu / abd::RZ0_I_S_0) * log(zu / (abd::RALPHA_0 * abd::RZ0_I_S_0)));   // LG15 Eq.11-12
    const double t = 1. / abd::RZ0_I_F_0;
    u.lg15_log_ratio = log(10. * t) / log(zu * t);                 // mod_cdn_form_ice.f90:322
    u.an05_us_c = 0.035 * log(10. / 8.0E-4) / log(zu / 8.0E-4);    // mod_blk_ice_an05.f90:151
    u.nb_iter = g.nb_iter;
    return u;
}

// copies both flag words back, synchronises, reports
int finish_ice_call(cudaStream_t cs_, const char *what)
{
    CUDA_TRY(cudaMemcpyAsync(g.h_bad, g.d_bad, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, cs_));
    CUDA_TRY(cudaStreamSynchronize(cs_));
    const unsigned long long bad_tau = g.h_bad[0], bad_rough = g.h_bad[1];
    if (bad_tau != ~0ull || bad_rough != ~0ull) {
        g.h_bad[0] = g.h_bad[1] = ~0ull;
        cudaMemsetAsync(g.d_bad, 0xFF, 2 * sizeof(unsigned long long), cs_);
        if (bad_rough != ~0ull)
            return fail(AEROBULK_GPU_ERR_ICE_ROUGH,
                        " rough_leng_tq@mod_blk_ice_an05.f90 => something wrong with zsmoot, ztrans, zrough!\n  (%s, point %lld)",
                        what, (long long)bad_rough + 1);
        return fail(AEROBULK_GPU_ERR_TAU, "BULK_FORMULA_VCTR()@mod_phymbl: wind stress too strong!\n  (%s, point %lld)", what,
                    (long long)bad_tau + 1);
    }
    return 0;
}

int turb_ice_impl(const char *calgo, double zt, double zu, int Ni, int Nj, const double *Ts_i, const double *t_zt,
                  const double *qs_i, const double *q_zt, const double *U_zu, const double *frice, const double *cxn,
                  double *Cd, double *Ch, double *Ce, double *t_zu, double *q_zu, double *Ubzu,
                  const aerobulk_gpu_turb_ice_optional *opt, int on_device)
{
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!calgo || !Ts_i || !t_zt || !qs_i || !q_zt || !U_zu || !Cd || !Ch || !Ce || !t_zu || !q_zu || !Ubzu)
        return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_turb_ice: NULL mandatory argument");
    const int ialgo = ice_algo_id(calgo);
    if (!ialgo) return fail(AEROBULK_GPU_ERR_ALGO, "aerobulk_gpu_turb_ice: sea-ice bulk algorithm %s is unknown!!!", calgo);
    const bool need_frice = (ialgo == abd::ICE_LU12 || ialgo == abd::ICE_LG15);
    if (need_frice && !frice) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_turb_ice: turb_ice_%s needs frice", calgo);
    if (ialgo == abd::ICE_EASY && !cxn) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_turb_ice: turb_ice_easy needs CdN, ChN, CeN");
    if (Ni < 0 || Nj < 0) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_turb_ice: negative shape %d x %d", Ni, Nj);
    int rc = ensure_device();
    if (rc) return rc;
    const long long n = (long long)Ni * Nj;
    if (n == 0) return 0;
    cudaStream_t cs_ = compute_stream();
    rc = deferred_errors();
    if (rc) return rc;

    double *optp[8] = {nullptr};
    static_assert(sizeof(aerobulk_gpu_turb_ice_optional) == 8 * sizeof(double *), "8 optional outputs");
    if (opt) memcpy(optp, opt, sizeof(*opt));
    abk::IceTurbArgs a;
    memset(&a, 0, sizeof(a));
    HostTransport t;
    t.in(&a.Ts_i, Ts_i, n); t.in(&a.t_zt, t_zt, n); t.in(&a.qs_i, qs_i, n); t.in(&a.q_zt, q_zt, n); t.in(&a.U_zu, U_zu, n);
    t.in(&a.frice, need_frice ? frice : nullptr, n);
    t.out(&a.Cd, Cd, n); t.out(&a.Ch, Ch, n); t.out(&a.Ce, Ce, n); t.out(&a.t_zu, t_zu, n); t.out(&a.q_zu, q_zu, n);
    t.out(&a.Ubzu, Ubzu, n);
    for (int k = 0; k < 8; ++k) t.out(&a.opt[k], optp[k], n);
    rc = t.open(on_device);
    if (rc) return rc;
    a.n = n;
    a.form_index = g.ice_form_per_point ? -1 : n - 1;
    a.u = make_ice_uniform(zt, zu, cxn);
    a.bad_rough = g.d_bad + 1;
    CUDA_TRY(abk::launch_ice_turb(ialgo, zt_eq_zu(zt, zu), a, cs_));
    g.launches += 1;
    rc = t.close();
    if (rc) return rc;
    return finish_ice_call(cs_, "aerobulk_gpu_turb_ice");
}

int oce_ice_impl(const char *calgo_ice, const char *calgo_oce, double zt, double zu, long long n, const double *sit,
                 const double *sst, const double *t_zt, const double *hum_zt, int hum_kind, const double *wind,
                 const double *slp, const double *frice, const double *cxn, const aerobulk_gpu_oce_ice_out *out, int on_device)
{
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!calgo_ice || !sit || !t_zt || !hum_zt || !wind || !slp || !frice || !out)
        return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_oce_ice: NULL mandatory argument");
    const int ialgo = ice_algo_id(calgo_ice);
    if (!ialgo) return fail(AEROBULK_GPU_ERR_ALGO, "aerobulk_gpu_oce_ice: sea-ice bulk algorithm %s is unknown!!!", calgo_ice);
    const int oalgo = calgo_oce ? algo_id(calgo_oce) : 0;
    if (calgo_oce && !oalgo) return fail(AEROBULK_GPU_ERR_ALGO, "aerobulk_gpu_oce_ice: bulk algorithm %s is unknown!!!", calgo_oce);
    if (oalgo && !sst) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_oce_ice: the leads need sst");
    if (ialgo == abd::ICE_EASY && !cxn) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_oce_ice: turb_ice_easy needs CdN, ChN, CeN");
    if (n < 0 || hum_kind < 0 || hum_kind > 2) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_oce_ice: bad n or hum_kind");
    int rc = ensure_device();
    if (rc) return rc;
    if (n == 0) return 0;
    cudaStream_t cs_ = compute_stream();
    rc = deferred_errors();
    if (rc) return rc;

    double *const hout[abk::NOCEICE_OUT] = {
        out->Cd_i, out->Ch_i, out->Ce_i, out->theta_zu_i, out->q_zu_i, out->t_zu_i, out->Ub_i, out->RiB_i, out->z0_i,
        out->u_star_i, out->L_i, out->UN10_i, out->rho_zu_i, out->Tau_i, out->QH_i, out->QL_i, out->Evap_i,
        out->Cd_w, out->Ch_w, out->Ce_w, out->theta_zu_w, out->q_zu_w, out->Ub_w, out->z0_w, out->u_star_w, out->L_w,
        out->UN10_w, out->Tau_w, out->QH_w, out->QL_w, out->Evap_w, out->Tau, out->QH, out->QL, out->Evap};
    abk::OceIceArgs a;
    memset(&a, 0, sizeof(a));
    HostTransport t;
    t.in(&a.sit, sit, n); t.in(&a.sst, oalgo ? sst : nullptr, n); t.in(&a.t_zt, t_zt, n); t.in(&a.hum_zt, hum_zt, n);
    t.in(&a.wnd, wind, n); t.in(&a.slp, slp, n); t.in(&a.frice, frice, n);
    // the leads kernel writes out[17..34]: without leads they stay as the caller passed them
    for (int k = 0; k < abk::NOCEICE_OUT; ++k) t.out(&a.out[k], hout[k], n, oalgo || k < 17);
    // scratch for the four ice fluxes the cell means need when the caller does not want them
    for (int k = 0; k < 4 && oalgo; ++k)
        if (!hout[13 + k]) t.scratch(&a.ice_flux[k], n);
    rc = t.open(on_device);
    if (rc) return rc;
    for (int k = 0; k < 4 && oalgo; ++k)
        if (hout[13 + k]) a.ice_flux[k] = a.out[13 + k];
    a.n = n;
    a.form_index = g.ice_form_per_point ? -1 : n - 1;
    a.hum_kind = hum_kind;
    a.ui = make_ice_uniform(zt, zu, cxn);
    a.uo = make_uniform(zt, zu);
    a.bad_tau = g.d_bad;
    a.bad_rough = g.d_bad + 1;
    const bool zteq = zt_eq_zu(zt, zu);
    CUDA_TRY(abk::launch_ice_flux(ialgo, zteq, a, cs_));
    g.launches += 1;
    if (oalgo) {
        CUDA_TRY(abk::launch_leads(oalgo, zteq, a, cs_));
        g.launches += 1;
    }
    rc = t.close();
    if (rc) return rc;
    return finish_ice_call(cs_, "aerobulk_gpu_oce_ice");
}

// ---------------------------------------------------------------------------
// sea-ice station series (src/ice/test_aerobulk_buoy_series_ice.f90): one launch for all records
// ---------------------------------------------------------------------------
int series_ice_impl(const char *calgo, double zt, double zu, long long n, const double *sic, const double *sit,
                    const double *t_zt, const double *hum_zt, int hum_kind, const double *wind, const double *slp,
                    const double *rad_sw, const double *rad_lw, const aerobulk_gpu_series_ice_out *out, int on_device)
{
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!calgo || !sic || !sit || !t_zt || !hum_zt || !wind || !slp || !rad_sw || !rad_lw || !out)
        return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_series_ice: NULL mandatory argument");
    const int ialgo = ice_algo_id(calgo);
    if (ialgo != abd::ICE_NEMO && ialgo != abd::ICE_AN05 && ialgo != abd::ICE_LU12 && ialgo != abd::ICE_LG15)
        return fail(AEROBULK_GPU_ERR_ALGO, "UNKNOWN algo: %s !!!", calgo);   // test_aerobulk_buoy_series_ice.f90:413-415
    if (n < 0 || hum_kind < 0 || hum_kind > 2) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_series_ice: bad n or hum_kind");
    int rc = ensure_device();
    if (rc) return rc;
    if (n == 0) return 0;
    cudaStream_t cs_ = compute_stream();
    rc = deferred_errors();
    if (rc) return rc;

    static_assert(sizeof(aerobulk_gpu_series_ice_out) == abk::NICESERIES_OUT * sizeof(double *), "21 output pointers");
    double *hout[abk::NICESERIES_OUT];
    memcpy(hout, out, sizeof(hout));
    abk::IceSeriesArgs a;
    memset(&a, 0, sizeof(a));
    HostTransport t;
    t.in(&a.sic, sic, n); t.in(&a.sit, sit, n); t.in(&a.t_zt, t_zt, n); t.in(&a.hum_zt, hum_zt, n); t.in(&a.wnd, wind, n);
    t.in(&a.slp, slp, n); t.in(&a.rad_sw, rad_sw, n); t.in(&a.rad_lw, rad_lw, n);
    for (int k = 0; k < abk::NICESERIES_OUT; ++k) t.out(&a.out[k], hout[k], n);
    rc = t.open(on_device);
    if (rc) return rc;
    a.n = n;
    a.hum_kind = hum_kind;
    a.ui = make_ice_uniform(zt, zu, nullptr);
    a.bad_tau = g.d_bad;
    a.bad_rough = g.d_bad + 1;
    CUDA_TRY(abk::launch_ice_series(ialgo, zt_eq_zu(zt, zu), a, cs_));
    g.launches += 1;
    rc = t.close();
    if (rc) return rc;
    return finish_ice_call(cs_, "aerobulk_gpu_series_ice");
}

// ---------------------------------------------------------------------------
// flux diagnostics (SURVEY.md 8e: the optional global reduction)
// ---------------------------------------------------------------------------
int diag_impl(long long n, const double *const *fields, double *stats, int on_device)
{
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!stats || n < 0) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_flux_diagnostics: bad argument");
    int rc = ensure_device();
    if (rc) return rc;
    cudaStream_t cs_ = compute_stream();
    abk::DiagArgs a;
    memset(&a, 0, sizeof(a));
    a.n = n;
    a.partials = g.d_partials;
    a.out = g.d_stats;
    if (on_device) {
        for (int f = 0; f < abk::NDIAG_FIELDS; ++f) a.field[f] = fields[f];
    } else {
        int nf = 0;
        for (int f = 0; f < abk::NDIAG_FIELDS; ++f) nf += fields[f] ? 1 : 0;
        rc = ensure_turb_slab(n * nf);
        if (rc) return rc;
        double *p = g.d_turb;
        for (int f = 0; f < abk::NDIAG_FIELDS; ++f) {
            if (!fields[f] || n == 0) continue;
            CUDA_TRY(cudaMemcpyAsync(p, fields[f], sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, cs_));
            a.field[f] = p;
            p += n;
        }
    }
    const long long want = (n + 255) / 256;
    const int nblocks = (int)(want < 1 ? 1 : (want > abk::stats_max_blocks() ? abk::stats_max_blocks() : want));
    CUDA_TRY(abk::launch_diag(a, nblocks, cs_));
    g.launches += 2;
    CUDA_TRY(cudaMemcpyAsync(stats, g.d_stats, sizeof(double) * abk::NDIAG, cudaMemcpyDeviceToHost, cs_));
    CUDA_TRY(cudaStreamSynchronize(cs_));
    return 0;
}

}  // namespace

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

int aerobulk_gpu_model(int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj, const double *sst,
                       const double *t_zt, const double *hum_zt, const double *U_zu, const double *V_zu,
                       const double *slp, double *QL, double *QH, double *Tau_x, double *Tau_y, double *Evap,
                       const int *Niter, const int *l_use_skin, const double *rad_sw, const double *rad_lw, double *T_s)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return model_host(sizeof(double), jt, Nt, calgo, zt, zu, Ni, Nj, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x,
                      Tau_y, Evap, Niter, l_use_skin, rad_sw, rad_lw, T_s);
}

int aerobulk_gpu_model_device(int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj,
                              const double *sst, const double *t_zt, const double *hum_zt, const double *U_zu,
                              const double *V_zu, const double *slp, double *QL, double *QH, double *Tau_x,
                              double *Tau_y, double *Evap, const int *Niter, const int *l_use_skin,
                              const double *rad_sw, const double *rad_lw, double *T_s)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return model_device(sizeof(double), jt, Nt, calgo, zt, zu, Ni, Nj, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x,
                        Tau_y, Evap, Niter, l_use_skin, rad_sw, rad_lw, T_s);
}

int aerobulk_gpu_model_f32(int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj, const float *sst,
                           const float *t_zt, const float *hum_zt, const float *U_zu, const float *V_zu,
                           const float *slp, float *QL, float *QH, float *Tau_x, float *Tau_y, float *Evap,
                           const int *Niter, const int *l_use_skin, const float *rad_sw, const float *rad_lw, float *T_s)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return model_host(sizeof(float), jt, Nt, calgo, zt, zu, Ni, Nj, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x,
                      Tau_y, Evap, Niter, l_use_skin, rad_sw, rad_lw, T_s);
}

int aerobulk_gpu_model_device_f32(int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj,
                                  const float *sst, const float *t_zt, const float *hum_zt, const float *U_zu,
                                  const float *V_zu, const float *slp, float *QL, float *QH, float *Tau_x,
                                  float *Tau_y, float *Evap, const int *Niter, const int *l_use_skin,
                                  const float *rad_sw, const float *rad_lw, float *T_s)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return model_device(sizeof(float), jt, Nt, calgo, zt, zu, Ni, Nj, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x,
                        Tau_y, Evap, Niter, l_use_skin, rad_sw, rad_lw, T_s);
}

static void copy_algo(char *dst, size_t cap, const char *calgo, int l)
{
    size_t n = (l < 0) ? 0 : (size_t)l;
    if (n >= cap) n = cap - 1;
    memcpy(dst, calgo, n);
    dst[n] = 0;
    // TRIM(): the Fortran side compares the blank-trimmed string
    while (n > 0 && dst[n - 1] == ' ') dst[--n] = 0;
}

void aerobulk_cxx_skin(const int *jt, const int *Nt, const char *calgo, const double *zt, const double *zu,
                       const double *sst, const double *t_zt, const double *hum_zt, const double *U_zu,
                       const double *V_zu, const double *slp, double *QL, double *QH, double *Tau_x, double *Tau_y,
                       double *Evap, const int *Niter, const bool *l_skin, const double *rad_sw, const double *rad_lw,
                       double *T_s, const int *l, const int *m)
{
    char algo[64];
    copy_algo(algo, sizeof(algo), calgo, *l);
    const int lskin = (*(const unsigned char *)l_skin) != 0;
    std::lock_guard<std::mutex> lk(g_mu);
    model_host(sizeof(double), *jt, *Nt, algo, *zt, *zu, *m, 1, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x, Tau_y, Evap,
               Niter, &lskin, rad_sw, rad_lw, T_s);
}

void aerobulk_cxx_no_skin(const int *jt, const int *Nt, const char *calgo, const double *zt, const double *zu,
                          const double *sst, const double *t_zt, const double *hum_zt, const double *U_zu,
                          const double *V_zu, const double *slp, double *QL, double *QH, double *Tau_x,
                          double *Tau_y, double *Evap, const int *Niter, const int *l, const int *m)
{
    char algo[64];
    copy_algo(algo, sizeof(algo), calgo, *l);
    std::lock_guard<std::mutex> lk(g_mu);
    model_host(sizeof(double), *jt, *Nt, algo, *zt, *zu, *m, 1, sst, t_zt, hum_zt, U_zu, V_zu, slp, QL, QH, Tau_x, Tau_y, Evap,
               Niter, nullptr, nullptr, nullptr, nullptr);
}

int aerobulk_gpu_turb(const char *calgo, int kt, double zt, double zu, int Ni, int Nj, double *T_s, const double *t_zt,
                      double *q_s, const double *q_zt, const double *U_zu, int l_use_cs, int l_use_wl, double *Cd,
                      double *Ch, double *Ce, double *t_zu, double *q_zu, double *Ubzu, const double *Qsw,
                      const double *rad_lw, const double *slp, int isecday_utc, const double *plong,
                      const aerobulk_gpu_turb_optional *opt, int on_device)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return turb_impl(calgo, kt, zt, zu, Ni, Nj, T_s, t_zt, q_s, q_zt, U_zu, l_use_cs, l_use_wl, Cd, Ch, Ce, t_zu, q_zu,
                     Ubzu, Qsw, rad_lw, slp, isecday_utc, plong, opt, on_device);
}

int aerobulk_gpu_series(const char *calgo, int Nt, long long S, double zt, double zu, const int *isecday_utc,
                        const double *lon, const double *sst, const double *t_zt, const double *hum_zt, int hum_kind,
                        const double *wind, const double *slp, const double *rad_sw, const double *rad_lw,
                        int l_use_skin, const aerobulk_gpu_series_out *out, int on_device)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return series_impl(calgo, Nt, S, zt, zu, isecday_utc, lon, sst, t_zt, hum_zt, hum_kind, wind, slp, rad_sw, rad_lw,
                       l_use_skin, out, on_device);
}

int aerobulk_gpu_series_csv(const char *path_in, const char *path_out, const char *calgo, double zt, double zu,
                            int l_use_skin)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return series_csv_impl(path_in, path_out, calgo, zt, zu, l_use_skin);
}

int aerobulk_gpu_turb_ice(const char *calgo, double zt, double zu, int Ni, int Nj, const double *Ts_i, const double *t_zt,
                          const double *qs_i, const double *q_zt, const double *U_zu, const double *frice,
                          const double *CxN_easy, double *Cd, double *Ch, double *Ce, double *t_zu, double *q_zu,
                          double *Ubzu, const aerobulk_gpu_turb_ice_optional *opt, int on_device)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return turb_ice_impl(calgo, zt, zu, Ni, Nj, Ts_i, t_zt, qs_i, q_zt, U_zu, frice, CxN_easy, Cd, Ch, Ce, t_zu, q_zu, Ubzu,
                         opt, on_device);
}

int aerobulk_gpu_oce_ice(const char *calgo_ice, const char *calgo_oce, double zt, double zu, long long n,
                         const double *sit, const double *sst, const double *t_zt, const double *hum_zt, int hum_kind,
                         const double *wind, const double *slp, const double *frice, const double *CxN_easy,
                         const aerobulk_gpu_oce_ice_out *out, int on_device)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return oce_ice_impl(calgo_ice, calgo_oce, zt, zu, n, sit, sst, t_zt, hum_zt, hum_kind, wind, slp, frice, CxN_easy, out,
                        on_device);
}

int aerobulk_gpu_series_ice(const char *calgo, double zt, double zu, long long n, const double *sic, const double *sit,
                            const double *t_zt, const double *hum_zt, int hum_kind, const double *wind, const double *slp,
                            const double *rad_sw, const double *rad_lw, const aerobulk_gpu_series_ice_out *out, int on_device)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return series_ice_impl(calgo, zt, zu, n, sic, sit, t_zt, hum_zt, hum_kind, wind, slp, rad_sw, rad_lw, out, on_device);
}

void aerobulk_gpu_set_ice_form_drag_per_point(int on) { std::lock_guard<std::mutex> lk(g_mu); g.ice_form_per_point = on ? 1 : 0; }

int aerobulk_gpu_flux_diagnostics(long long n, const double *QL, const double *QH, const double *Tau_x, const double *Tau_y,
                                  const double *Evap, const double *T_s, double *stats, int on_device)
{
    std::lock_guard<std::mutex> lk(g_mu);
    const double *fields[abk::NDIAG_FIELDS] = {QL, QH, Tau_x, Tau_y, Evap, T_s};
    return diag_impl(n, fields, stats, on_device);
}

int aerobulk_gpu_diag_reduce_op(int i) { return (i <= 0 || i >= abk::NDIAG) ? 0 : (i - 1) % 3; }

int aerobulk_gpu_chunk_plan(long long n, int kind, long long *cstart)
{
    if (n < 0 || kind < 0 || kind > 3 || !cstart) return -1;
    return plan_chunks(n, kind, cstart);
}

int aerobulk_gpu_selftest_host_copy(long long n, int rounds)
{
    // no device needed: exercises the copy threads of the pageable-array path on host memory alone
    if (n < 1 || rounds < 1) return -1;
    std::vector<double> src((size_t)n), mid((size_t)n), dst((size_t)n);
    int bad = 0;
    for (int r = 0; r < rounds; ++r) {
        for (long long i = 0; i < n; ++i) src[(size_t)i] = (double)(i * 31 + r);
        std::vector<CopyPiece> there, back;
        add_pieces(there, mid.data(), src.data(), sizeof(double) * (size_t)n);
        add_pieces(back, dst.data(), mid.data(), sizeof(double) * (size_t)n);
        copy_pool().run(there.data(), (int)there.size());
        copy_pool().run(back.data(), (int)back.size());
        bad += memcmp(src.data(), dst.data(), sizeof(double) * (size_t)n) != 0;
    }
    return bad;
}

int aerobulk_gpu_host_register(void *ptr, size_t bytes)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!ptr || bytes == 0) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_host_register: NULL pointer or empty range");
    int rc = ensure_device();
    if (rc) return rc;
    const cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped);
    if (e != cudaSuccess) {
        cudaGetLastError();   // not sticky: the session stays usable
        return fail(AEROBULK_GPU_ERR_CUDA, "aerobulk_gpu_host_register: %s", cudaGetErrorString(e));
    }
    return 0;
}

int aerobulk_gpu_host_unregister(void *ptr)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!ptr) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_host_unregister: NULL pointer");
    int rc = ensure_device();
    if (rc) return rc;
    cudaSetDevice(g.device);
    cudaDeviceSynchronize();   // nothing in flight may still touch the range
    const cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(AEROBULK_GPU_ERR_CUDA, "aerobulk_gpu_host_unregister: %s", cudaGetErrorString(e));
    }
    return 0;
}

void aerobulk_gpu_set_nitend(int nitend) { std::lock_guard<std::mutex> lk(g_mu); g.nitend = nitend; }

int aerobulk_gpu_synchronize(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    for (int d = MAX_DEVICES - 1; d >= 1; --d) {   // the other devices of a split call (their calls are blocking: nothing pending)
        if (!sess[d].device_ready) continue;
        CUDA_TRY(cudaSetDevice(sess[d].device));
        CUDA_TRY(cudaStreamSynchronize(sess[d].own_stream));
        CUDA_TRY(cudaStreamSynchronize(sess[d].out_stream));
    }
    if (!g.device_ready) return 0;
    CUDA_TRY(cudaSetDevice(g.device));
    CUDA_TRY(cudaStreamSynchronize(compute_stream()));
    CUDA_TRY(cudaStreamSynchronize(g.out_stream));
    const bool skin_before = g.l_use_skin_schemes;
    int rc = resolve_init();
    if (!rc) rc = check_bad_flag(nullptr, nullptr);
    if (rc) end_session_after_error(0, skin_before);
    return rc;
}

int aerobulk_gpu_set_devices(int n)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (n < 1 || n > MAX_DEVICES) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_set_devices(%d): 1 .. %d devices", n, MAX_DEVICES);
    for (int d = 0; d < MAX_DEVICES; ++d)
        if (sess[d].n_coare || sess[d].n_ecmwf)
            return fail(AEROBULK_GPU_ERR_STATE, "aerobulk_gpu_set_devices(%d): a warm-layer session is open (finish it at jt == Nt or call aerobulk_gpu_reset)", n);
    if (n > 1) {
        int count = 0;
        const cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count <= 0)
            return fail(AEROBULK_GPU_ERR_CUDA, "no CUDA device available (%s): libaerobulk_gpu has no CPU fallback",
                        e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        if (n > count) return fail(AEROBULK_GPU_ERR_CUDA, "aerobulk_gpu_set_devices(%d): only %d device(s) visible", n, count);
    }
    n_devices = n;
    if (n == 1) split_nd = 1;
    return 0;
}
int aerobulk_gpu_get_devices(void) { return n_devices; }

int aerobulk_gpu_shard_plan(long long n, int n_dev, long long *start)
{
    if (n < 0 || n_dev < 1 || !start) return -1;
    return plan_shards(n, n_dev, start);
}

int aerobulk_gpu_init_local_stats(int Ni, int Nj, const double *sst, const double *t_zt, const double *hum_zt,
                                  const double *U_zu, const double *V_zu, const double *slp, const double *rad_lw,
                                  double *stats)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (!stats || !sst || !t_zt || !hum_zt || !U_zu || !V_zu || !slp) return fail(AEROBULK_GPU_ERR_ARG, "init_local_stats: NULL argument");
    int rc = ensure_device();
    if (rc) return rc;
    const long long n = (long long)Ni * Nj;
    if (n <= 0) {
        for (int k = 0; k < abk::NSTATS; ++k) {
            const int op = aerobulk_gpu_stats_reduce_op(k);
            stats[k] = op == 0 ? 0. : op == 1 ? 1.79769313486231570e308 : -1.79769313486231570e308;
        }
        return 0;
    }
    return local_stats(n, sizeof(double), sst, t_zt, hum_zt, U_zu, V_zu, slp, rad_lw, compute_stream(), stats);
}

int aerobulk_gpu_stats_reduce_op(int i)
{
    if (i < 2 || i >= 2 + 5 * abk::NFIELDS) return 0;
    const int r = (i - 2) % 5;
    return (r == 0) ? 0 : (r == 1 || r == 3) ? 1 : 2;
}

int aerobulk_gpu_init_from_stats(int Nt, const char *calgo, const int *l_use_skin, int have_rad, const double *stats)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!calgo || !stats) return fail(AEROBULK_GPU_ERR_ARG, "init_from_stats: NULL argument");
    const bool lskin = l_use_skin ? (*l_use_skin != 0) : false;
    int rc = init_from_stats(Nt, calgo, lskin, have_rad != 0, stats, 0, 0);
    if (rc) return rc;
    g.preinit_done = true;
    return 0;
}

int aerobulk_gpu_init(int Nt, const char *calgo, int Ni, int Nj, const double *sst, const double *t_zt, const double *hum_zt,
                      const double *U_zu, const double *V_zu, const double *slp, const int *l_use_skin, const double *rad_sw,
                      const double *rad_lw)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!calgo || !sst || !t_zt || !hum_zt || !U_zu || !V_zu || !slp) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_init: NULL mandatory argument");
    if (Ni < 0 || Nj < 0) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_init: negative shape %d x %d", Ni, Nj);
    int rc = ensure_device();
    if (rc) return rc;
    rc = resolve_init();
    if (rc) return rc;
    const long long n = (long long)Ni * Nj;
    const bool lskin = l_use_skin ? (*l_use_skin != 0) : false;
    const bool lsrad = rad_sw && rad_lw;
    double st[abk::NSTATS];
    memset(st, 0, sizeof(st));
    if (n > 0) {
        rc = ensure_staging(n * (long long)sizeof(double));
        if (rc) return rc;
        cudaStream_t cs = compute_stream();
        const double *h[7] = {sst, t_zt, hum_zt, U_zu, V_zu, slp, lsrad ? rad_lw : nullptr};
        for (int k = 0; k < 7; ++k)
            if (h[k]) CUDA_TRY(cudaMemcpyAsync(g.d_in[k], h[k], sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, cs));
        rc = local_stats(n, sizeof(double), g.d_in[0], g.d_in[1], g.d_in[2], g.d_in[3], g.d_in[4], g.d_in[5], lsrad ? g.d_in[6] : nullptr, cs, st);
        if (rc) return rc;
    }
    const bool skin_before = g.l_use_skin_schemes;
    rc = init_from_stats(Nt, calgo, lskin, lsrad, st, Ni, Nj);
    if (rc) end_session_after_error(1, skin_before);
    return rc;
}

void aerobulk_gpu_bye(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (g.verbose) {
        printf(" ===================================================================\n");
        printf("                    ----- AeroBulk_bye -----\n");
        printf(" ===================================================================\n \n");
        fflush(stdout);
    }
}

int aerobulk_gpu_init_local_stats_device(int Ni, int Nj, const double *sst, const double *t_zt, const double *hum_zt,
                                         const double *U_zu, const double *V_zu, const double *slp, const double *rad_lw,
                                         double *d_stats)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!d_stats || !sst || !t_zt || !hum_zt || !U_zu || !V_zu || !slp)
        return fail(AEROBULK_GPU_ERR_ARG, "init_local_stats_device: NULL argument");
    const long long n = (long long)Ni * Nj;
    if (n <= 0) return fail(AEROBULK_GPU_ERR_ARG, "init_local_stats_device: empty row block (give it the identity vector instead)");
    int rc = ensure_device();
    if (rc) return rc;
    return launch_local_stats(n, sizeof(double), sst, t_zt, hum_zt, U_zu, V_zu, slp, rad_lw, compute_stream(), d_stats);
}

int aerobulk_gpu_init_from_gathered_stats(int Nt, const char *calgo, const int *l_use_skin, int have_rad,
                                          const double *d_all, int nranks)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (!calgo || !d_all || nranks < 1) return fail(AEROBULK_GPU_ERR_ARG, "init_from_gathered_stats: bad argument");
    int rc = ensure_device();
    if (rc) return rc;
    const bool lskin = l_use_skin ? (*l_use_skin != 0) : false;
    const int verbose = g.verbose;
    g.verbose = 0;   // the banner needs the statistics on the host: this path never brings them back in time
    rc = init_async(Nt, calgo, lskin, have_rad != 0, d_all, nranks, 0, 0, compute_stream());
    g.verbose = verbose;
    if (rc) return rc;
    g.preinit_done = true;
    return 0;
}

void aerobulk_gpu_set_rdt(double v) { std::lock_guard<std::mutex> lk(g_mu); g.rdt = v; }
void aerobulk_gpu_set_gdept(double v) { std::lock_guard<std::mutex> lk(g_mu); g.gdept = v; }
void aerobulk_gpu_set_nb_iter(int v) { std::lock_guard<std::mutex> lk(g_mu); g.nb_iter = v; }
int aerobulk_gpu_get_nb_iter(void) { return g.nb_iter; }
int aerobulk_gpu_get_use_skin(void) { return g.l_use_skin_schemes ? 1 : 0; }
const char *aerobulk_gpu_get_humidity_type(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (g.init_pending && g.device_ready && cudaSetDevice(g.device) == cudaSuccess) {
        // asynchronous AEROBULK_INIT: the device has decided, the host has not caught up -- read the device's verdict
        // (the checks and their error, if any, still surface at the next synchronising call, where they belong)
        int v[2] = {g.ihum, 0};
        if (cudaStreamSynchronize(compute_stream()) == cudaSuccess &&
            cudaMemcpy(v, g.d_init, sizeof(v), cudaMemcpyDeviceToHost) == cudaSuccess && v[0] >= 0 && v[0] <= 2)
            return HUM_NAMES[v[0]];
    }
    return HUM_NAMES[g.ihum];
}

int aerobulk_gpu_set_device(int device)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (g.device_ready && device != g.device)
        return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_set_device(%d): session already bound to device %d (call aerobulk_gpu_reset first)", device, g.device);
    g.device = device;
    return 0;
}
int aerobulk_gpu_get_device(void) { return g.device; }

int aerobulk_gpu_set_stream(void *stream)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.user_stream = (cudaStream_t)stream;
    g.use_user_stream = (stream != nullptr);
    return 0;
}

void aerobulk_gpu_set_error_mode(int m) { g.error_mode = m ? 1 : 0; }
void aerobulk_gpu_set_verbose(int on) { g.verbose = on ? 1 : 0; }
void aerobulk_gpu_set_sort(int mode) { g.sort_points = mode < 0 ? 0 : (mode > 2 ? 2 : mode); }
const char *aerobulk_gpu_last_error(void) { return g.errmsg; }
int aerobulk_gpu_last_error_code(void) { return g.errcode; }

static void reset_session()   // the session of `cur`
{
    if (g.device_ready) {
        cudaSetDevice(g.device);
        cudaDeviceSynchronize();
        free_coare_state();
        free_ecmwf_state();
        free_bounce();
        if (g.d_in[0]) cudaFree(g.d_in[0]);   // one slab, see ensure_staging
        for (int k = 0; k < 8; ++k) g.d_in[k] = nullptr;
        for (int k = 0; k < 6; ++k) g.d_out[k] = nullptr;
        g.cap = 0;
        if (g.d_perm) cudaFree(g.d_perm);
        g.d_perm = nullptr;
        g.cap_perm = 0;
        if (g.d_turb) cudaFree(g.d_turb);
        g.d_turb = nullptr;
        g.cap_turb = 0;
        if (g.h_bad) g.h_bad[0] = g.h_bad[1] = ~0ull;
        if (g.d_bad) cudaMemset(g.d_bad, 0xFF, 2 * sizeof(unsigned long long));
    }
    g.n_coare = g.n_ecmwf = 0;
    g.ice_form_per_point = 0;
    g.pitched_ok = true;
    g.nb_iter = 5;
    g.nitend = 1;
    g.l_use_skin_schemes = false;
    g.ihum = 0;
    g.rdt = 3600.;
    g.gdept = 1.;
    g.preinit_done = false;
    g.init_pending = false;
    g.bad_pending = false;
    g.pend_launches = 0;
    g.async_device = false;
    g.time_kernels = false;
    g.kt_used = 0;
    g.errcode = 0;
    g.errmsg[0] = 0;
    g.shard = 0;
    g.flat_offset = 0;
    g.report_Ni = g.report_Nj = 0;
    g.stats_hook = nullptr;
}

void aerobulk_gpu_reset(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    Session *const mine = cur;
    for (int d = MAX_DEVICES - 1; d >= 0; --d) {   // session 0 last: its device stays the thread's current one
        cur = &sess[d];
        reset_session();
    }
    cur = mine;
    split_nd = 1;
}

// Warm-layer state of the session of `cur`.  which 0..3: dT_wl, Hz_wl, Qnt_ac, Tau_ac of the COARE scheme when a COARE
// session is open, else dT_wl (0) and the constant Hz_wl (1) of the ECMWF scheme; which 4 / 5 name the ECMWF pair
// explicitly (both schemes can hold a session at the same time, as the module arrays of the reference can).
static double *state_ptr(int which, long long *n, bool *const_hz)
{
    *const_hz = false;
    if (which >= 0 && which < 4 && g.n_coare) {
        *n = g.n_coare;
        return g.c_state[which];
    }
    if (g.n_ecmwf && (which == 0 || which == 1 || which == 4 || which == 5) && !(which < 4 && g.n_coare)) {
        *n = g.n_ecmwf;
        if (which == 1 || which == 5) {
            *const_hz = true;
            return nullptr;
        }
        return g.e_dT_wl;
    }
    *n = 0;
    return nullptr;
}

// get (dir 0) or set (dir 1) the state of every session that took part in the last (possibly split) call
static long state_io(int which, double *host, long n, int dir)
{
    if (!host) return 0;
    Session *const mine = cur;
    long long total = 0;
    for (int d = 0; d < split_nd; ++d) {
        cur = &sess[d];
        long long have = 0;
        bool chz = false;
        state_ptr(which, &have, &chz);
        total += have;
    }
    long done = 0;
    if (total == n && total > 0) {
        long long off = 0;
        for (int d = 0; d < split_nd; ++d) {
            cur = &sess[d];
            long long have = 0;
            bool chz = false;
            double *p = state_ptr(which, &have, &chz);
            if (have == 0) continue;
            cudaSetDevice(g.device);
            cudaStreamSynchronize(compute_stream());
            if (chz) {   // Hz_wl of the ECMWF scheme is the constant rd0 = 3 m (mod_skin_ecmwf.f90:57): nothing stored
                if (dir == 0)
                    for (long long i = 0; i < have; ++i) host[off + i] = 3.;
            } else if (!p) {
                off = -1;
                break;
            } else if (cudaMemcpy(dir == 0 ? (void *)(host + off) : (void *)p, dir == 0 ? (const void *)p : (const void *)(host + off),
                                  sizeof(double) * (size_t)have, dir == 0 ? cudaMemcpyDeviceToHost : cudaMemcpyHostToDevice) != cudaSuccess) {
                off = -1;
                break;
            }
            off += have;
        }
        done = (off == total) ? n : 0;
    }
    cur = mine;
    if (mine->device_ready) cudaSetDevice(mine->device);
    return done;
}

long aerobulk_gpu_get_state(int which, double *host_out, long n)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return state_io(which, host_out, n, 0);
}

long aerobulk_gpu_set_state(int which, const double *host_in, long n)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return state_io(which, const_cast<double *>(host_in), n, 1);
}

void aerobulk_gpu_new_session(void)
{
    // what a NEW PROCESS of the reference would start with: the SAVEd module variables of mod_const.f90:22-33 at their
    // initial values and no warm-layer arrays -- without giving the device buffers back (aerobulk_gpu_reset does that
    // too, at the price of a device synchronisation and re-allocation).  Settings of this library (device(s), stream,
    // error mode, verbosity, sort policy, rdt / gdept, async mode) are kept.  Deferred errors of earlier asynchronous
    // calls are NOT cleared: they still surface at the next synchronising call.
    std::lock_guard<std::mutex> lk(g_mu);
    for (int d = 0; d < MAX_DEVICES; ++d) {
        sess[d].nb_iter = 5;
        sess[d].nitend = 1;
        sess[d].l_use_skin_schemes = false;
        if (!sess[d].init_pending) sess[d].ihum = 0;
        sess[d].preinit_done = false;
        sess[d].n_coare = sess[d].n_ecmwf = 0;
    }
}

void aerobulk_gpu_set_async(int on)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.async_device = on != 0;
}

void aerobulk_gpu_set_kernel_timing(int on)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.time_kernels = on != 0;
    g.kt_used = 0;
}

int aerobulk_gpu_kernel_times(double *ms, int max)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g.device_ready || !ms) return 0;
    cudaSetDevice(g.device);
    cudaStreamSynchronize(compute_stream());
    int k = 0;
    for (size_t i = 0; i + 1 < g.kt_used && k < max; i += 2) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, g.kt_ev[i], g.kt_ev[i + 1]) != cudaSuccess) {
            cudaGetLastError();
            break;
        }
        ms[k++] = (double)t;
    }
    g.kt_used = 0;
    return k;
}

long aerobulk_gpu_launch_count(void)
{
    long t = 0;
    for (int d = 0; d < MAX_DEVICES; ++d) t += sess[d].launches;
    return t;
}
void aerobulk_gpu_reset_launch_count(void)
{
    for (int d = 0; d < MAX_DEVICES; ++d) sess[d].launches = 0;
}

double aerobulk_gpu_measure_fp64_peak(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (ensure_device()) return -1.;
    g.launches += 5;
    return abk::measure_fp64_peak(compute_stream());
}

// SURVEY.md 8d / BASELINE.md 3: fx + nb_iter*it FP64-pipe instruction equivalents per point
double aerobulk_gpu_work_per_point(const char *calgo, int skin, int nb_iter)
{
    const int a = calgo ? algo_id(calgo) : 0;
    double it = 0., fx = 0.;
    switch (a) {
    case abd::NCAR: it = 595.; fx = 1947.; break;
    case abd::ANDREAS: it = 2028.; fx = 1801.; break;
    case abd::COARE3P0: if (skin) { it = 4756.; fx = 4721.; } else { it = 1790.; fx = 4360.; } break;
    case abd::COARE3P6: if (skin) { it = 4733.; fx = 4698.; } else { it = 1767.; fx = 4337.; } break;
    case abd::ECMWF: if (skin) { it = 5006.; fx = 5389.; } else { it = 1378.; fx = 5028.; } break;
    default: return 0.;
    }
    return fx + nb_iter * it;
}

double aerobulk_gpu_bytes_per_point(const char *calgo, int skin)
{
    const int a = calgo ? algo_id(calgo) : 0;
    if (!a) return 0.;
    if (!skin || !has_skin_schemes(a)) return 88.;
    return a == abd::ECMWF ? 128. : 176.;
}

int aerobulk_gpu_kernel_info(const char *calgo, int skin, int zt_eq_zu, int *registers, int *local_bytes, int *blocks_per_sm)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.errcode = 0;
    g.errmsg[0] = 0;
    const int a = calgo ? algo_id(calgo) : 0;
    if (!a) return fail(AEROBULK_GPU_ERR_ALGO, "aerobulk_gpu_kernel_info: bulk algorithm %s is unknown!!!", calgo ? calgo : "(null)");
    int rc = ensure_device();
    if (rc) return rc;
    cudaFuncAttributes at;
    int blocks = 0;
    CUDA_TRY(abk::flux_kernel_attributes(a, skin && has_skin_schemes(a), zt_eq_zu != 0, &at, &blocks));
    if (registers) *registers = at.numRegs;
    if (local_bytes) *local_bytes = (int)at.localSizeBytes;
    if (blocks_per_sm) *blocks_per_sm = blocks;
    return 0;
}

const char *aerobulk_gpu_version(void) { return "aerobulk-b200 0.2 (sm_100a, FP64)"; }

int aerobulk_gpu_probe(int func, long long n, int nargs, const double *args, double *out)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g.errcode = 0;
    g.errmsg[0] = 0;
    if (n < 0 || nargs < 1 || nargs > 6 || !args || !out) return fail(AEROBULK_GPU_ERR_ARG, "aerobulk_gpu_probe: bad argument");
    int rc = ensure_device();
    if (rc) return rc;
    if (n == 0) return 0;
    rc = ensure_turb_slab(n * (nargs + 1));
    if (rc) return rc;
    cudaStream_t cs_ = compute_stream();
    CUDA_TRY(cudaMemcpyAsync(g.d_turb, args, sizeof(double) * (size_t)n * nargs, cudaMemcpyHostToDevice, cs_));
    double *d_out = g.d_turb + n * nargs;
    CUDA_TRY(abk::launch_probe(func, n, nargs, g.d_turb, d_out, cs_));
    g.launches += 1;
    CUDA_TRY(cudaMemcpyAsync(out, d_out, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, cs_));
    CUDA_TRY(cudaStreamSynchronize(cs_));
    return 0;
}

}  // extern "C"
