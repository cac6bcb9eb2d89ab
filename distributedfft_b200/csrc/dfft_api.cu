// dfft_api.cu -- C-ABI implementation: slab bookkeeping, communicator, plan, stage sequencing.
//
// Host-side counterpart of 3dmpifft_opt/include/fft_mpi_3d_api.cpp (plan :41-141, execute :181-214,
// stages :466-699) re-designed for B200: three batched pass launches per transform instead of two
// launches per plane, the pack folded into the Y-pass store, the all-to-all either fused into that
// store over NVLink peer mappings or handed to NCCL, CUDA events instead of host timers, explicit
// streams and no device-wide syncs on the production path.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/dfft.h"
#include "dfft_kernels.cuh"
#include "fft_tma.cuh"

using namespace dfft;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const char* fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    if (getenv("DFFT_VERBOSE")) fprintf(stderr, "[dfft] error %d: %s\n", code, buf);
    return code;
}
#define CU(x)                                                                                         \
    do {                                                                                              \
        cudaError_t e_ = (x);                                                                         \
        if (e_ != cudaSuccess) return fail(DFFT_ECUDA, "%s:%d CUDA call '%s' failed: %s", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
    } while (0)

extern "C" const char* dfft_last_error(void) { return g_err.c_str(); }
extern "C" int dfft_version(void) { return 100; }

extern "C" int dfft_length_kind(int n, int precision)
{
    if (n < 1 || n > (1 << 20) || (precision != DFFT_DOUBLE && precision != DFFT_FLOAT)) return 0;
    const SizeEntry* e = find_size_entry(n, precision);
    return !e ? 0 : (e->gen ? 1 : 2);
}

/* test hook: which multi-role kernels the entry of length n has (bit k: fused t0 kind k of FusedKind, bit 4: the kernel-chain
 * link fused_yx, bit 5: the single-kernel forward fused3); -1 if the length is unsupported */
extern "C" int dfft_debug_fused_kinds(int n, int precision)
{
    if (n < 1 || n > (1 << 20) || (precision != DFFT_DOUBLE && precision != DFFT_FLOAT)) return -1;
    const SizeEntry* e = find_size_entry(n, precision);
    if (!e) return -1;
    int m = 0;
    for (int k = 0; k < FK_COUNT; k++) m |= e->fused[k] ? 1 << k : 0;
    return m | (e->fused_yx ? 1 << 4 : 0) | (e->fused3 ? 1 << 5 : 0);
}

/* radix schedule the library uses for length n (contiguous-pass schedule for tuned lengths, the run-time schedule for
 * generic ones); returns the number of stages, 0 if unsupported */
extern "C" int dfft_length_schedule(int n, int precision, int* radices, int max_radices)
{
    if (n < 1 || n > (1 << 20) || (precision != DFFT_DOUBLE && precision != DFFT_FLOAT)) return 0;
    const SizeEntry* e = find_size_entry(n, precision);
    if (!e) return 0;
    if (radices)
        for (int i = 0; i < e->z_nstages && i < max_radices; i++) radices[i] = e->z_rad[i];
    return e->z_nstages;
}

/* test hook (host only, no device needed): ticket -> (role, part, plane, tile) of the single-kernel forward path;
 * ticket < 0 returns the number of tickets */
extern "C" long long dfft_debug_fused3_order(long long planes, long long rows, int GA, int GBk, int GXk, int K, int lag, long long ticket, long long out[4])
{
    Fused3Ctl F{};
    F.planes = planes; F.rows = rows; F.GA = GA; F.GBk = GBk; F.GB = GBk * K; F.GXk = GXk; F.GX = GXk * K; F.K = K; F.lag = lag;
    const Fused3Order o = fused3_prepare(F);
    const long long total = (long long)o.total;
    if (ticket < 0 || ticket >= total || !out) return total;
    int role, part, yfloor;
    unsigned plane, idx;
    fused3_decode(F, o, (unsigned)ticket, role, part, plane, idx, yfloor);
    out[0] = role; out[1] = part; out[2] = plane; out[3] = idx;
    return total;
}

extern "C" int dfft_supported_lengths(int precision, int* lengths, int max_lengths)
{
    std::vector<int> v;
    list_sizes(precision, v);
    std::sort(v.begin(), v.end());
    if (lengths)
        for (int i = 0; i < (int)v.size() && i < max_lengths; i++) lengths[i] = v[i];
    return (int)v.size();
}

// ------------------------------------------------------------------------------------------------
// slab geometry (fft_mpi_3d_api.cpp:56-66, 89-91, 232-316)
// ------------------------------------------------------------------------------------------------
static inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

struct Geom {
    long long n0, n1, n2;
    int P;
    long long xd() const { return cdiv(n0, P); }
    long long yd() const { return cdiv(n1, P); }
    long long last_n0() const { return n0 - (P - 1) * xd(); }
    long long last_n1() const { return n1 - (P - 1) * yd(); }
    long long n0l(int p) const { return p == P - 1 ? last_n0() : xd(); }
    long long n1l(int q) const { return q == P - 1 ? last_n1() : yd(); }
    long long in_count(int p) const { return n0l(p) * n1 * n2; }
    long long out_count(int q) const { return n0 * n1l(q) * n2; }
    long long max_count(int p) const { return std::max(in_count(p), out_count(p)); }
};

static int proper_device_num(long long n0, int wanted)
{
    if (wanted < 1) return 0;
    if (n0 % wanted == 0) return wanted;
    long long per = n0 / wanted + 1;
    int dev = (int)(n0 / per);
    if (n0 % per) dev += 1;
    return dev;
}

extern "C" int dfft_init(const long long N[3], int wanted, int* total, int* local, long long* counts)
{
    if (!N || wanted < 1 || N[0] < 1 || N[1] < 1 || N[2] < 1) return fail(DFFT_EINVAL, "dfft_init: bad arguments");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess) { cudaGetLastError(); ndev = 0; }
    if (ndev > 0 && wanted > ndev) wanted = ndev;   // api.cpp:236-239
    int dev = proper_device_num(N[0], wanted);
    if (dev < 1) return fail(DFFT_EUNSUPPORTED, "could not support this distribution of data");
    Geom g{N[0], N[1], N[2], dev};
    if (g.last_n1() < 1) return fail(DFFT_EUNSUPPORTED, "N1=%lld cannot be split over %d devices (empty last y-slab)", N[1], dev);
    if (counts)
        for (int i = 0; i < dev; i++) counts[i] = g.in_count(i);
    if (total) *total = dev;
    if (local) *local = dev;
    // peer access between the devices used (api.cpp:16-27)
    for (int i = 0; i < dev && i < ndev; i++) {
        int cur = 0;
        cudaGetDevice(&cur);
        if (cudaSetDevice(i) != cudaSuccess) { cudaGetLastError(); continue; }
        for (int j = 0; j < dev && j < ndev; j++) {
            if (i == j) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, i, j) == cudaSuccess && can) {
                cudaError_t pe = cudaDeviceEnablePeerAccess(j, 0);
                if (pe != cudaSuccess) cudaGetLastError();   // already enabled is fine
            }
        }
        cudaSetDevice(cur);
    }
    return 0;
}

extern "C" long long dfft_max_data_count(long long n0, long long n1, long long n2, int P, int is_last)
{
    if (P < 1) return -1;
    Geom g{n0, n1, n2, P};
    return g.max_count(is_last ? P - 1 : 0);
}

extern "C" long long dfft_local_size_3d(long long n0, long long n1, long long n2, int P, int dev, long long* ln0,
                                        long long* s0, long long* ln1, long long* s1)
{
    if (P < 1 || dev < 0 || dev >= P) return -1;
    Geom g{n0, n1, n2, P};
    if (ln0) *ln0 = g.n0l(dev);
    if (s0) *s0 = dev * g.xd();
    if (ln1) *ln1 = g.n1l(dev);
    if (s1) *s1 = dev * g.yd();
    return g.max_count(dev);
}

extern "C" void* dfft_alloc_local(long long count, int flag, int precision)
{
    if (count < 0) { fail(DFFT_EINVAL, "negative count"); return nullptr; }
    size_t bytes = (size_t)count * (precision == DFFT_FLOAT ? 8 : 16);
    if (bytes == 0) bytes = 16;
    void* p = nullptr;
    cudaError_t e;
    if (flag == DFFT_ALLOC_CPU) e = cudaMallocHost(&p, bytes);
    else if (flag == DFFT_ALLOC_DEV) e = cudaMalloc(&p, bytes);
    else { fail(DFFT_EINVAL, "Fail to allocate memory!"); return nullptr; }
    if (e != cudaSuccess) { fail(DFFT_ENOMEM, "allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e)); cudaGetLastError(); return nullptr; }
    return p;
}

extern "C" int dfft_free_local(void* p, int flag)
{
    if (!p) return 0;
    if (flag == DFFT_ALLOC_CPU) CU(cudaFreeHost(p));
    else CU(cudaFree(p));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// communicator
// ------------------------------------------------------------------------------------------------
struct dfft_comm_s {
    int nranks = 1;
    bool local = true;
    // local (threads of one process)
    std::mutex mu;
    std::condition_variable cv;
    int arrived = 0;
    long long gen = 0;
    std::vector<std::vector<unsigned char>> slots;
    // bootstrap (process per GPU)
    int rank = 0;
    dfft_allgather_fn ag = nullptr;
    void* ctx = nullptr;

    // A participant that fails in the middle of a collective sequence (plan creation) poisons the communicator: every
    // rank blocked in -- or later entering -- a barrier returns an error instead of waiting for a peer that will never come.
    bool failed = false;
    void poison()
    {
        std::lock_guard<std::mutex> lk(mu);
        failed = true;
        cv.notify_all();
    }
    int barrier()
    {
        std::unique_lock<std::mutex> lk(mu);
        if (failed) return -1;
        long long g = gen;
        if (++arrived == nranks) { arrived = 0; gen++; cv.notify_all(); }
        else cv.wait(lk, [&] { return gen != g || failed; });
        return failed ? -1 : 0;
    }
    int allgather(int r, const void* send, void* recv, size_t bytes)
    {
        if (nranks == 1) { memcpy(recv, send, bytes); return 0; }
        if (!local) return ag(ctx, send, recv, bytes);
        {
            std::lock_guard<std::mutex> lk(mu);
            slots[r].assign((const unsigned char*)send, (const unsigned char*)send + bytes);
        }
        if (barrier()) return -1;
        for (int i = 0; i < nranks; i++) memcpy((unsigned char*)recv + (size_t)i * bytes, slots[i].data(), bytes);
        if (barrier()) return -1;
        return 0;
    }
    int host_barrier(int r)
    {
        if (nranks == 1) return 0;
        if (local) return barrier();
        std::vector<unsigned char> tmp(nranks);
        unsigned char one = 1;
        return ag(ctx, &one, tmp.data(), 1);
    }
};

extern "C" int dfft_comm_create_local(int nranks, dfft_comm* comm)
{
    if (nranks < 1 || !comm) return fail(DFFT_EINVAL, "dfft_comm_create_local: bad arguments");
    dfft_comm c = new dfft_comm_s;
    c->nranks = nranks;
    c->local = true;
    c->slots.resize(nranks);
    *comm = c;
    return 0;
}

extern "C" int dfft_comm_create_bootstrap(int rank, int nranks, dfft_allgather_fn ag, void* ctx, dfft_comm* comm)
{
    if (nranks < 1 || rank < 0 || rank >= nranks || !comm || (nranks > 1 && !ag))
        return fail(DFFT_EINVAL, "dfft_comm_create_bootstrap: bad arguments");
    dfft_comm c = new dfft_comm_s;
    c->nranks = nranks;
    c->local = false;
    c->rank = rank;
    c->ag = ag;
    c->ctx = ctx;
    *comm = c;
    return 0;
}

/* host-side all-gather through the communicator (what plan creation uses to exchange IPC handles) */
extern "C" int dfft_comm_allgather(dfft_comm c, int rank, const void* send, void* recv, size_t bytes)
{
    if (!c || !send || !recv || rank < 0 || rank >= c->nranks) return fail(DFFT_EINVAL, "dfft_comm_allgather: bad arguments");
    if (c->allgather(rank, send, recv, bytes) != 0) return fail(DFFT_ECOMM, "bootstrap allgather failed");
    return 0;
}

extern "C" int dfft_comm_destroy(dfft_comm c)
{
    delete c;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// NCCL, loaded at run time (no link-time dependency; picks up the copy torch already loaded)
// ------------------------------------------------------------------------------------------------
struct NcclUid { char b[128]; };   // ncclUniqueId (NCCL_UNIQUE_ID_BYTES = 128), passed by value
struct NcclApi {
    void* h = nullptr;
    int (*GetUniqueId)(NcclUid*) = nullptr;
    int (*CommInitRank)(void**, int, NcclUid, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*AlltoAll)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;   // NCCL >= 2.28
    const char* (*GetErrorString)(int) = nullptr;
    int (*GetVersion)(int*) = nullptr;
    bool ok = false;
};

static NcclApi& nccl_api()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {getenv("DFFT_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (!n) continue;
            api.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (api.h) break;
        }
        if (!api.h) return;
#define LD(field, sym) *(void**)(&api.field) = dlsym(api.h, sym)
        LD(GetUniqueId, "ncclGetUniqueId");
        LD(CommInitRank, "ncclCommInitRank");
        LD(CommDestroy, "ncclCommDestroy");
        LD(GroupStart, "ncclGroupStart");
        LD(GroupEnd, "ncclGroupEnd");
        LD(Send, "ncclSend");
        LD(Recv, "ncclRecv");
        LD(AlltoAll, "ncclAlltoAll");
        LD(GetErrorString, "ncclGetErrorString");
        LD(GetVersion, "ncclGetVersion");
#undef LD
        api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.GroupStart && api.GroupEnd && api.Send && api.Recv;
    });
    return api;
}
#define NC(x)                                                                                          \
    do {                                                                                               \
        int r_ = (x);                                                                                  \
        if (r_ != 0) return fail(DFFT_ECOMM, "%s:%d NCCL call '%s' failed: %s", __FILE__, __LINE__, #x, \
                                 nccl_api().GetErrorString ? nccl_api().GetErrorString(r_) : "?");     \
    } while (0)

// ------------------------------------------------------------------------------------------------
// cross-device flags for the fused (P2P) exchange
// ------------------------------------------------------------------------------------------------
struct SyncBlock {
    unsigned long long arrive[DFFT_MAX_CHUNKS];  // arrive[s] = e : sender s finished writing my recv buffer for epoch e
    unsigned long long ready[DFFT_MAX_CHUNKS];   // ready[r] = e  : receiver r finished reading its recv buffer of epoch e
    unsigned long long part_arrive[DFFT_MAX_PARTS][DFFT_MAX_CHUNKS];   // overlapped mode: part k of sender s has arrived (epoch e)
};
struct FlagPtrs {
    unsigned long long* p[DFFT_MAX_CHUNKS];
};

__global__ void signal_flags_kernel(FlagPtrs dst, int n, unsigned long long value)
{
    const int q = threadIdx.x;
    if (q < n) {
        __threadfence_system();
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(dst.p[q]), "l"(value) : "memory");
    }
}
__global__ void wait_flags_kernel(const unsigned long long* flags, int n, unsigned long long value)
{
    const int q = threadIdx.x;
    if (q < n) {
        unsigned long long v;
        SpinGuard guard;   // a peer that never signals (it died) traps this kernel after DFFT_SPIN_TIMEOUT_NS instead of hanging the GPU
        do {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + q) : "memory");
            if (v < value) { __nanosleep(200); guard.tick(); }
        } while (v < value);
    }
    __threadfence_system();
}

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
struct dfft_plan_s {
    Geom g;
    int P = 1, me = 0, direction = DFFT_FORWARD, prec = 0, device = 0, sms = 148;
    unsigned flags = 0;
    int xmode = DFFT_EXCHANGE_P2P;
    size_t esz = 16;
    long long n0l = 0, n1l = 0, in_count = 0, out_count = 0, max_count = 0;
    void *in = nullptr, *out = nullptr, *buf1 = nullptr, *buf2 = nullptr;
    void* work = nullptr;   // plan-owned scratch / receive buffer: keeps bufferDev1 intact so execute is repeatable
    bool inplace = false;
    const SizeEntry *ez = nullptr, *ey = nullptr, *ex = nullptr;   // axes N2 (Z), N1 (Y), N0 (X)
    void *lut_z = nullptr, *lut_y = nullptr, *lut_x = nullptr;
    void* lut_xn = nullptr;   // X axis with the strided-local schedule (DFFT_NATURAL_SPECTRUM)
    // TMA-pipelined pass kernels (fft_tma.cuh) for the axes that have an instantiation: used for the passes whose load and
    // store are both local and un-chunked (Z, natural Y, X with the fused transpose); nullptr -> register-staged kernels
    const TmaEntry *tz = nullptr, *ty = nullptr, *tx = nullptr;
    void *lut_tz = nullptr, *lut_ty = nullptr, *lut_tx = nullptr;
    bool natural = false;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t pev[3][2] = {{nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}};   // per pass (Z, Y, X) brackets
    dfft_comm comm = nullptr;
    // p2p
    std::vector<void*> peer_work, peer_buf1;
    SyncBlock* sync = nullptr;
    std::vector<SyncBlock*> peer_sync;
    std::vector<void*> ipc_opened;
    unsigned long long epoch = 0;
    // nccl
    void* nccl = nullptr;
    int launches = 0;
    bool timed = false;
    // fused two-pass t0 (L2-resident intermediate): per-plane completion counters + ticket words
    bool fuse = false;
    int lag = 0;
    unsigned long long* plane_done = nullptr;
    unsigned int* ticket = nullptr;
    unsigned long long fuse_epoch = 0;
    // describe-only plans (DFFT_DRY_RUN): no CUDA call is made, buffers are symbolic addresses, execute records the
    // passes it would launch (dfft_debug_plan_ops) -- lets the CPU tests interpret the whole multi-device schedule
    bool dry = false;
    std::vector<std::string> ops;
    // overlapped forward (fft_fused3_kernel): own intermediate buffer, per-part counters
    bool overlap = false;
    int parts = 1;
    void* mid = nullptr;
    unsigned long long* part_done = nullptr;
    unsigned long long overlap_epoch = 0;
    // stream-pipelined forward (DFFT_PIPELINE): the z axis is cut into `parts`; the send side (stream: Z, then the Y pass of
    // part k with the pack / peer stores folded in, or + ncclAlltoAll of part k on the comm stream) runs ahead of the receive
    // side (stream2: X pass of part k as soon as part k has arrived from every sender) -- t2 and t3 overlap t0
    bool pipe = false;
    bool pipe_fyx = false;           // forward, cube, P2P: parts run as a chain of two-role kernels on ONE stream (fft_fused_yx_kernel:
                                     // Y pass of part k + X pass of part k-1 share every SM slot) instead of two streams
    bool in_pipe = false;            // inside fwd_pipelined: Pass::launch leaves the per-pass event brackets alone
    cudaStream_t stream2 = nullptr, stream3 = nullptr;   // receive side; NCCL part exchanges
    cudaEvent_t ev_join = nullptr, evb[2] = {nullptr, nullptr};
    cudaEvent_t ev_y[DFFT_MAX_PARTS] = {}, ev_a[DFFT_MAX_PARTS] = {};
    void* sendbuf = nullptr;         // NCCL: part-major packed send buffer
    unsigned long long* dbg = nullptr;   // DFFT_DEBUG_TIMELINE: device-side timeline of the single-kernel forward path
    unsigned int* done_ctr = nullptr; // [DFFT_MAX_PARTS] finished-CTA counters of the part kernels (arrival signal folded into the kernel)
};

// symbolic device address of a describe-only plan: device d (0-based), buffer id b: 1 bufferDev1, 2 bufferDev2 / user out,
// 3 work / receive buffer, 4 intermediate of the single-kernel path, 5 user in
static inline void* fake_addr(int d, int b) { return (void*)((((unsigned long long)(d + 1)) << 44) | (((unsigned long long)b) << 40)); }
static inline char* eoff(void* base, long long elems, size_t esz) { return (char*)base + (size_t)elems * esz; }
static inline cudaError_t ev_record(dfft_plan p, cudaEvent_t e) { return p->dry ? cudaSuccess : cudaEventRecord(e, p->stream); }
static inline cudaError_t ev_record_on(dfft_plan p, cudaEvent_t e, cudaStream_t st) { return p->dry ? cudaSuccess : cudaEventRecord(e, st); }
static inline cudaError_t stream_wait(dfft_plan p, cudaStream_t st, cudaEvent_t e) { return p->dry ? cudaSuccess : cudaStreamWaitEvent(st, e, 0); }

template <typename T>
static void record_op(dfft_plan p, const char* name, int phase, int N, int C, bool chunk_in, bool chunk_out, bool transposed_store, const TileArgs<T>& a)
{
    char buf[256];
    std::string o = "{";
    snprintf(buf, sizeof(buf), "\"op\": \"%s\", \"phase\": %d, \"N\": %d, \"C\": %d, \"G\": %d, \"W\": %d, \"ntiles\": %lld, \"inv\": %d, \"do_scale\": %d, \"scale\": %.17g, \"tw_n\": %lld, ",
             name, phase, N, C, a.G, a.W, a.ntiles, a.inv, a.do_scale, (double)a.scale, a.tw_n);
    o += buf;
    snprintf(buf, sizeof(buf), "\"in\": %llu, \"out\": %llu, \"ia\": [%lld, %lld, %lld, %lld], \"oa\": [%lld, %lld, %lld, %lld], \"tstore\": %d",
             (unsigned long long)(size_t)a.in, (unsigned long long)(size_t)a.out, a.ia.SA, a.ia.SB, a.ia.cs, a.ia.es, a.oa.SA, a.oa.SB, a.oa.cs, a.oa.es,
             transposed_store ? 1 : 0);
    o += buf;
    for (int side = 0; side < 2; side++) {
        const bool on = side == 0 ? chunk_in : chunk_out;
        if (!on) continue;
        const ChunkTab& ct = side == 0 ? a.ci : a.co;
        snprintf(buf, sizeof(buf), ", \"%s\": {\"ediv\": %d, \"nchunks\": %d, \"cptr\": [", side == 0 ? "ci" : "co", ct.ediv, ct.nchunks);
        o += buf;
        for (int q = 0; q < ct.nchunks; q++) { snprintf(buf, sizeof(buf), "%s%llu", q ? ", " : "", (unsigned long long)(size_t)ct.cptr[q]); o += buf; }
        o += "], \"SAq\": [";
        for (int q = 0; q < ct.nchunks; q++) { snprintf(buf, sizeof(buf), "%s%lld", q ? ", " : "", ct.SAq[q]); o += buf; }
        o += "]}";
    }
    o += "}";
    p->ops.push_back(o);
}

template <typename T> static cudaError_t upload_lut(void** dst, int nstages, const int* rad)
{
    std::vector<cx<T>> lut = build_lut<T>(nstages, rad);
    cudaError_t e = cudaMalloc(dst, lut.size() * sizeof(cx<T>));
    if (e != cudaSuccess) { *dst = nullptr; return e; }
    return cudaMemcpy(*dst, lut.data(), lut.size() * sizeof(cx<T>), cudaMemcpyHostToDevice);
}

static int share_pointer(dfft_plan p, void* mine, std::vector<void*>& peers)
{
    // make `mine` (a cudaMalloc allocation of this device) addressable by every rank
    const int P = p->P;
    peers.assign(P, nullptr);
    if (p->dry) return 0;   // describe-only plans compute peer addresses symbolically
    if (p->comm->local) {
        std::vector<void*> all(P);
        if (p->comm->allgather(p->me, &mine, all.data(), sizeof(void*)) != 0) return fail(DFFT_ECOMM, "a peer failed during plan creation");
        peers = all;
        return 0;
    }
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, mine));
    std::vector<cudaIpcMemHandle_t> all(P);
    if (p->comm->allgather(p->me, &h, all.data(), sizeof(h)) != 0) return fail(DFFT_ECOMM, "bootstrap allgather failed");
    for (int q = 0; q < P; q++) {
        if (q == p->me) { peers[q] = mine; continue; }
        void* ptr = nullptr;
        CU(cudaIpcOpenMemHandle(&ptr, all[q], cudaIpcMemLazyEnablePeerAccess));
        peers[q] = ptr;
        p->ipc_opened.push_back(ptr);
    }
    return 0;
}

static int plan_create(long long n0, long long n1, long long n2, void* in, void* out, dfft_comm comm, int dev_idx,
                       int P, int direction, int precision, unsigned flags, dfft_plan* plan_out);

extern "C" int dfft_plan_c2c_3d(long long n0, long long n1, long long n2, void* in, void* out, dfft_comm comm, int dev_idx,
                                int P, int direction, int precision, unsigned flags, dfft_plan* plan_out)
{
    const int rc = plan_create(n0, n1, n2, in, out, comm, dev_idx, P, direction, precision, flags, plan_out);
    // a participant that fails (bad argument, allocation, peer mapping ...) must not leave the others waiting for it
    // in the collective part of plan creation: the local communicator is poisoned and their barriers return an error
    if (rc != 0 && P > 1 && comm && comm->local && !(flags & DFFT_DRY_RUN)) comm->poison();
    return rc;
}

static int plan_create(long long n0, long long n1, long long n2, void* in, void* out, dfft_comm comm, int dev_idx,
                       int P, int direction, int precision, unsigned flags, dfft_plan* plan_out)
{
    if (!plan_out) return fail(DFFT_EINVAL, "null plan pointer");
    *plan_out = nullptr;
    if (n0 < 1 || n1 < 1 || n2 < 1 || P < 1 || dev_idx < 0 || dev_idx >= P || !in)
        return fail(DFFT_EINVAL, "dfft_plan_c2c_3d: bad arguments");
    if (direction != DFFT_FORWARD && direction != DFFT_BACKWARD) return fail(DFFT_EINVAL, "direction must be +1 or -1");
    if (precision != DFFT_DOUBLE && precision != DFFT_FLOAT) return fail(DFFT_EINVAL, "bad precision");
    if (P > DFFT_MAX_CHUNKS) return fail(DFFT_EUNSUPPORTED, "at most %d devices", DFFT_MAX_CHUNKS);
    const bool dry = (flags & DFFT_DRY_RUN) != 0;
    if (!dry && P > 1 && (!comm || comm->nranks != P)) return fail(DFFT_EINVAL, "a communicator of %d ranks is required", P);
    Geom g{n0, n1, n2, P};
    if (g.last_n0() < 1 || g.last_n1() < 1)
        return fail(DFFT_EUNSUPPORTED, "%lldx%lldx%lld cannot be split over %d devices (empty last slab); use dfft_init", n0, n1, n2, P);
    const SizeEntry* ez = find_size_entry((int)n2, precision);
    const SizeEntry* ey = find_size_entry((int)n1, precision);
    const SizeEntry* ex = find_size_entry((int)n0, precision);
    if (n0 > 1 << 20 || n1 > 1 << 20 || n2 > 1 << 20 || !ez || !ey || !ex)
        return fail(DFFT_EUNSUPPORTED, "unsupported transform length in %lldx%lldx%lld (see dfft_supported_lengths)", n0, n1, n2);

    dfft_plan p = new dfft_plan_s;
    p->g = g; p->P = P; p->me = dev_idx; p->direction = direction; p->prec = precision; p->flags = flags;
    p->esz = precision == DFFT_FLOAT ? 8 : 16;
    p->n0l = g.n0l(dev_idx); p->n1l = g.n1l(dev_idx);
    p->in_count = direction == DFFT_FORWARD ? g.in_count(dev_idx) : g.out_count(dev_idx);
    p->out_count = direction == DFFT_FORWARD ? g.out_count(dev_idx) : g.in_count(dev_idx);
    p->max_count = g.max_count(dev_idx);
    p->ez = ez; p->ey = ey; p->ex = ex; p->comm = comm;
    p->in = in; p->out = out;
    p->dry = dry;
    int rc = 0;
    // a rank that fails after the collective part has begun must not leave its peers waiting for it
    auto bail = [&](int code) { if (!dry && P > 1 && comm && comm->local) comm->poison(); dfft_destroy(p); return code; };   // poison BEFORE destroy's barrier
#define CUP(x)                                                                                        \
    do {                                                                                              \
        cudaError_t e_ = (x);                                                                         \
        if (e_ != cudaSuccess) return bail(fail(DFFT_ECUDA, "%s:%d CUDA call '%s' failed: %s", __FILE__, __LINE__, #x, cudaGetErrorString(e_))); \
    } while (0)
    if (!dry) {
        CUP(cudaGetDevice(&p->device));
        CUP(cudaDeviceGetAttribute(&p->sms, cudaDevAttrMultiProcessorCount, p->device));
    }
    // buffers (api.cpp:66-77)
    if (!out || out == in) { p->inplace = true; p->buf2 = in; }
    else p->buf2 = out;
    if (dry) p->buf1 = fake_addr(dev_idx, 1);
    else {
        CUP(cudaMalloc(&p->buf1, (size_t)p->max_count * p->esz));
        CUP(cudaMemcpy(p->buf1, in, (size_t)p->max_count * p->esz, cudaMemcpyDeviceToDevice));
        CUP(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
        for (auto& e : p->ev) CUP(cudaEventCreate(&e));
        for (auto& pe : p->pev) for (auto& e : pe) CUP(cudaEventCreate(&e));
    }
    if (dry) {
        // no twiddle tables: the interpreter of the recorded passes does its own transforms
    } else if (precision == DFFT_DOUBLE) {
        CUP(upload_lut<double>(&p->lut_z, ez->z_nstages, ez->z_rad));
        CUP(upload_lut<double>(&p->lut_y, ey->s_nstages, ey->s_rad));
        CUP(upload_lut<double>(&p->lut_x, ex->x_nstages, ex->x_rad));
    } else {
        CUP(upload_lut<float>(&p->lut_z, ez->z_nstages, ez->z_rad));
        CUP(upload_lut<float>(&p->lut_y, ey->s_nstages, ey->s_rad));
        CUP(upload_lut<float>(&p->lut_x, ex->x_nstages, ex->x_rad));
    }
    if (!dry) CUP(cudaGetLastError());
    if (!dry && !(flags & DFFT_NO_TMA)) {
        p->tz = find_tma_entry((int)n2, precision);
        p->ty = find_tma_entry((int)n1, precision);
        p->tx = find_tma_entry((int)n0, precision);
        const TmaEntry* te[3] = {p->tz, p->ty, p->tx};
        void** tl[3] = {&p->lut_tz, &p->lut_ty, &p->lut_tx};
        for (int i = 0; i < 3; i++) {
            if (!te[i]) continue;
            if (precision == DFFT_DOUBLE) CUP(upload_lut<double>(tl[i], te[i]->nstages, te[i]->rad));
            else CUP(upload_lut<float>(tl[i], te[i]->nstages, te[i]->rad));
        }
    }
    if (flags & DFFT_NATURAL_SPECTRUM) {
        // spectrum kept in natural [x][y][z] order: one device only (with P > 1 it would need a second all-to-all)
        if (P != 1) return bail(fail(DFFT_EUNSUPPORTED, "DFFT_NATURAL_SPECTRUM needs a single device (a distributed natural-order spectrum would take a second exchange)"));
        if ((flags & DFFT_EXCHANGE_MASK) == DFFT_EXCHANGE_STAGED) return bail(fail(DFFT_EINVAL, "DFFT_NATURAL_SPECTRUM cannot be combined with the staged mode"));
        p->natural = true;
        if (!dry) {
            if (precision == DFFT_DOUBLE) CUP(upload_lut<double>(&p->lut_xn, ex->s_nstages, ex->s_rad));
            else CUP(upload_lut<float>(&p->lut_xn, ex->s_nstages, ex->s_rad));
        }
    }
    // exchange mode
    int xmode = (int)(flags & DFFT_EXCHANGE_MASK);
    if (P == 1) xmode = xmode == DFFT_EXCHANGE_STAGED ? DFFT_EXCHANGE_STAGED : DFFT_EXCHANGE_P2P;
    else if (xmode == DFFT_EXCHANGE_AUTO) {
        const char* env = getenv("DFFT_EXCHANGE");
        if (env && !strcmp(env, "nccl")) xmode = DFFT_EXCHANGE_NCCL;
        else if (env && !strcmp(env, "staged")) xmode = DFFT_EXCHANGE_STAGED;
        else xmode = DFFT_EXCHANGE_P2P;
    }
    if (P > 1 && !dry) {
        // peer reachability (api.cpp:16-27 enables peer access in fft_mpi_init; done here so a plan does not
        // depend on dfft_init having run).  Threads of one process map peers directly and need
        // cudaDeviceEnablePeerAccess; separate processes get it from cudaIpcOpenMemHandle.
        std::vector<int> devs(P);
        if (comm->allgather(p->me, &p->device, devs.data(), sizeof(int)) != 0) return bail(fail(DFFT_ECOMM, "bootstrap allgather failed"));
        int reach = 1;
        if (comm->local) {
            for (int q = 0; q < P; q++) {
                if (q == p->me || devs[q] == p->device) continue;
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, p->device, devs[q]) != cudaSuccess || !can) { cudaGetLastError(); reach = 0; continue; }
                cudaError_t pe = cudaDeviceEnablePeerAccess(devs[q], 0);
                if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) reach = 0;
                cudaGetLastError();
            }
        }
        std::vector<int> all(P);
        if (comm->allgather(p->me, &reach, all.data(), sizeof(int)) != 0) return bail(fail(DFFT_ECOMM, "bootstrap allgather failed"));
        for (int q = 0; q < P; q++) reach &= all[q];
        if (!reach) {
            if ((flags & DFFT_EXCHANGE_MASK) == DFFT_EXCHANGE_AUTO && !getenv("DFFT_EXCHANGE")) xmode = DFFT_EXCHANGE_NCCL;
            else if (xmode != DFFT_EXCHANGE_NCCL) return bail(fail(DFFT_ECOMM, "peer access between the devices is not available; use DFFT_EXCHANGE_NCCL"));
        }
    }
    p->xmode = xmode;
    // the fused kernels pair the contiguous and the strided role of one table entry: square planes only
    {
        // policy: the fused kernel wins when the strided role's stores are NVLink-bound (P2P exchange: the
        // contiguous role then hides entirely under the link time); on one GPU / NCCL the two HBM-bound sweeps
        // are currently faster (profiles/: SM-side time of both roles adds up), so it is opt-in there.
        const char* env = getenv("DFFT_FUSE");
        // the fused kernel this plan would launch: the chunked kinds carry the exchange (P > 1); an entry has no launcher for a
        // kind whose roles do not fit one CTA's shared memory (make_entry), and such a plan runs the two passes separately
        const int kind = P > 1 ? (direction == DFFT_FORWARD ? FK_ZY_CO : FK_YZ_CI) : (direction == DFFT_FORWARD ? FK_ZY : FK_YZ);
        const bool can = n1 == n2 && ez->fused[kind] != nullptr;
        bool want = P > 1 && xmode == DFFT_EXCHANGE_P2P;
        if (env) want = strcmp(env, "0") != 0;
        if (flags & DFFT_FORCE_FUSE) want = true;
        if (flags & DFFT_NO_FUSE) want = false;
        p->fuse = can && want;
        if (getenv("DFFT_LAG")) p->lag = atoi(getenv("DFFT_LAG"));
        if (p->fuse && !dry) {
            CUP(cudaMalloc((void**)&p->plane_done, (size_t)p->n0l * sizeof(unsigned long long)));
            CUP(cudaMemset(p->plane_done, 0, (size_t)p->n0l * sizeof(unsigned long long)));
            CUP(cudaMalloc((void**)&p->ticket, 4 * sizeof(unsigned int)));
            CUP(cudaMemset(p->ticket, 0, 4 * sizeof(unsigned int)));
        }
    }

    if (dry && xmode == DFFT_EXCHANGE_STAGED) return bail(fail(DFFT_EINVAL, "DFFT_DRY_RUN cannot describe the staged mode"));
    if (dry) p->work = fake_addr(dev_idx, 3);
    else if (xmode != DFFT_EXCHANGE_STAGED) CUP(cudaMalloc(&p->work, (size_t)p->max_count * p->esz));
    {
        // opt-in: the whole forward transform of a device as one kernel with t3 overlapped behind per-part arrivals
        const char* env = getenv("DFFT_OVERLAP");
        const bool want = (flags & DFFT_OVERLAP_X) || (env && strcmp(env, "0") != 0);
        if (want && P > 1 && xmode == DFFT_EXCHANGE_P2P && direction == DFFT_FORWARD && p->fuse && ez->fused3 && ex == ez) {
            const int cy = ez->p_C, cx_ = ez->x_C;
            int lcm = cy > cx_ ? cy : cx_;   // both are powers of two in the tuned tables
            if (lcm % cy == 0 && lcm % cx_ == 0) {
                int K = 1;
                for (int k : {4, 2})
                    if (n2 % ((long long)k * lcm) == 0) { K = k; break; }
                if (getenv("DFFT_PARTS")) {
                    const int k = atoi(getenv("DFFT_PARTS"));
                    if (k >= 1 && k <= DFFT_MAX_PARTS && n2 % ((long long)k * lcm) == 0) K = k;
                }
                p->parts = K;
                p->overlap = true;
                if (dry) p->mid = fake_addr(dev_idx, 4);
                else {
                    CUP(cudaMalloc(&p->mid, (size_t)p->max_count * p->esz));
                    CUP(cudaMalloc((void**)&p->part_done, DFFT_MAX_PARTS * sizeof(unsigned long long)));
                    CUP(cudaMemset(p->part_done, 0, DFFT_MAX_PARTS * sizeof(unsigned long long)));
                }
            }
        }
    }
    {
        // stream-pipelined forward (z-parts): send side and receive side on two streams, see fwd_pipelined
        const char* env = getenv("DFFT_PIPELINE");
        // Policy, from the sweeps under profiles/ (r2_sweep_pipeline_{2,4}gpu.log, r2_sweep_kernel_chain*_{2,4}gpu.log):
        //  * 2 devices: the transform is HBM / L2-fabric bound and already at ~95 % of its (6+2) E M roofline without overlap
        //    (512^3: 1.38 ms plain, 1.43-1.57 ms in parts): never pipelined by default.
        //  * two streams (any exchange): a Y-part kernel and an X-part kernel each want both CTA slots of an SM, so they
        //    serialise or halve each other; NCCL's kernels compete for the same slots (4 devices, 512^3: 0.86 ms plain, 0.97-1.10 ms
        //    two-stream, NCCL 1.47 vs 1.50-1.62): opt-in only.
        //  * kernel chain (cubes, P2P): [Z + Y0] [Y1 + X0] ... [X last] with the two roles pinned to the two CTA slots of every SM.
        //    4 devices: 1024^3 8.79 -> 7.47 ms (-15 %), 512^3 0.87 -> 0.86 ms (a tie), 768^3 fp32 and 256^3 slightly slower.
        //    Default from 4 devices on for axes >= 1024 points, where the X pass that it hides is long enough to pay for the
        //    extra launches and the second read of the intermediate.
        // DFFT_FORCE_PIPELINE / DFFT_PIPELINE=1 pipeline wherever it is possible, DFFT_NO_PIPELINE / DFFT_PIPELINE=0 never.
        const bool possible = P > 1 && !p->overlap && (xmode == DFFT_EXCHANGE_P2P || xmode == DFFT_EXCHANGE_NCCL);
        const bool chain_ok = direction == DFFT_FORWARD && xmode == DFFT_EXCHANGE_P2P && p->fuse && ey == ex && ey->fused_yx != nullptr;
        bool want = possible && chain_ok && P >= 4 && n2 >= 1024;
        if (env) want = possible && strcmp(env, "0") != 0;
        if (flags & DFFT_FORCE_PIPELINE) want = possible;
        if (direction == DFFT_BACKWARD && getenv("DFFT_PIPELINE_BWD") && !strcmp(getenv("DFFT_PIPELINE_BWD"), "0")) want = false;
        if (flags & DFFT_NO_PIPELINE) want = false;
        if (xmode == DFFT_EXCHANGE_NCCL && (n0 % P || n1 % P)) want = false;   // ncclAlltoAll parts need equal chunks
        if (want) {
            const int cy = direction == DFFT_FORWARD ? ey->p_C : ey->s_C, cx_ = ex->x_C;
            const int m = cy > cx_ ? cy : cx_;
            int K = 0;
            if (m % cy == 0 && m % cx_ == 0) {
                for (int k : {4, 2})
                    if (n2 % ((long long)k * m) == 0 && n2 / k >= 32) { K = k; break; }
                if (getenv("DFFT_PARTS")) {
                    const int k = atoi(getenv("DFFT_PARTS"));
                    if (k >= 1 && k <= DFFT_MAX_PARTS && n2 % ((long long)k * m) == 0) K = k;
                }
            }
            if (K >= 1 && (K > 1 || getenv("DFFT_PARTS"))) {
                p->parts = K;
                p->pipe = true;
                {
                    const char* pm = getenv("DFFT_PIPE_MODE");   // "streams": the two-stream schedule even where the kernel chain is possible
                    p->pipe_fyx = direction == DFFT_FORWARD && xmode == DFFT_EXCHANGE_P2P && p->fuse && ey == ex && ey->fused_yx != nullptr &&
                                  !(pm && !strcmp(pm, "streams"));
                }
                if (dry) { p->mid = fake_addr(dev_idx, 4); p->sendbuf = fake_addr(dev_idx, 6); }
                else {
                    if (!p->mid && direction == DFFT_FORWARD) CUP(cudaMalloc(&p->mid, (size_t)p->max_count * p->esz));
                    if (xmode == DFFT_EXCHANGE_NCCL) {
                        CUP(cudaMalloc(&p->sendbuf, (size_t)p->max_count * p->esz));
                        CUP(cudaStreamCreateWithFlags(&p->stream3, cudaStreamNonBlocking));
                    }
                    if (xmode == DFFT_EXCHANGE_P2P && !getenv("DFFT_SIGNAL_KERNELS")) {
                        CUP(cudaMalloc((void**)&p->done_ctr, DFFT_MAX_PARTS * sizeof(unsigned int)));
                        CUP(cudaMemset(p->done_ctr, 0, DFFT_MAX_PARTS * sizeof(unsigned int)));
                    }
                    CUP(cudaStreamCreateWithFlags(&p->stream2, cudaStreamNonBlocking));
                    CUP(cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming));
                    for (auto& e : p->evb) CUP(cudaEventCreate(&e));
                    for (int k = 0; k < K; k++) {
                        CUP(cudaEventCreateWithFlags(&p->ev_y[k], cudaEventDisableTiming));
                        CUP(cudaEventCreateWithFlags(&p->ev_a[k], cudaEventDisableTiming));
                    }
                }
            }
        }
    }
    if (P > 1 && dry) {
        p->peer_work.resize(P);
        for (int q = 0; q < P; q++) p->peer_work[q] = fake_addr(q, 3);
    } else if (P > 1) {
        if (xmode == DFFT_EXCHANGE_P2P || xmode == DFFT_EXCHANGE_STAGED) {
            if (xmode == DFFT_EXCHANGE_P2P) {
                if ((rc = share_pointer(p, p->work, p->peer_work)) != 0) return bail(rc);
            } else {
                if ((rc = share_pointer(p, p->buf1, p->peer_buf1)) != 0) return bail(rc);
            }
            CUP(cudaMalloc((void**)&p->sync, sizeof(SyncBlock)));
            CUP(cudaMemset(p->sync, 0, sizeof(SyncBlock)));
            if (xmode == DFFT_EXCHANGE_P2P && !p->done_ctr && !getenv("DFFT_SIGNAL_KERNELS")) {
                CUP(cudaMalloc((void**)&p->done_ctr, DFFT_MAX_PARTS * sizeof(unsigned int)));
                CUP(cudaMemset(p->done_ctr, 0, DFFT_MAX_PARTS * sizeof(unsigned int)));
            }
            std::vector<void*> ps;
            if ((rc = share_pointer(p, p->sync, ps)) != 0) return bail(rc);
            p->peer_sync.resize(P);
            for (int q = 0; q < P; q++) p->peer_sync[q] = (SyncBlock*)ps[q];
        } else {
            NcclApi& api = nccl_api();
            if (!api.ok) return bail(fail(DFFT_ECOMM, "libnccl.so.2 could not be loaded (set DFFT_NCCL_LIB)"));
            NcclUid uid;
            memset(&uid, 0, sizeof(uid));
            if (p->me == 0) {
                int r = api.GetUniqueId(&uid);
                if (r != 0) return bail(fail(DFFT_ECOMM, "ncclGetUniqueId failed"));
            }
            std::vector<NcclUid> all(P);
            if (comm->allgather(p->me, &uid, all.data(), sizeof(uid)) != 0) return bail(fail(DFFT_ECOMM, "bootstrap allgather failed"));
            int r = api.CommInitRank(&p->nccl, P, all[0], p->me);
            if (r != 0) return bail(fail(DFFT_ECOMM, "ncclCommInitRank failed: %s", api.GetErrorString ? api.GetErrorString(r) : "?"));
        }
        if (comm->host_barrier(p->me) != 0) return bail(fail(DFFT_ECOMM, "a peer failed during plan creation"));
    }
    if (!dry) CUP(cudaDeviceSynchronize());
#undef CUP
    *plan_out = p;
    return 0;
}

extern "C" int dfft_destroy(dfft_plan p)
{
    if (!p) return 0;
    if (p->dry) { delete p; return 0; }   // nothing was allocated
    cudaSetDevice(p->device);
    if (p->stream) cudaStreamSynchronize(p->stream);
    if (p->P > 1 && p->comm && (p->sync || p->nccl)) p->comm->host_barrier(p->me);   // nobody still writes into my buffers
    if (p->nccl) nccl_api().CommDestroy(p->nccl);
    for (void* q : p->ipc_opened) cudaIpcCloseMemHandle(q);
    if (p->P > 1 && p->comm && !p->comm->local && !p->ipc_opened.empty()) p->comm->host_barrier(p->me);
    if (p->buf1) cudaFree(p->buf1);
    if (p->work) cudaFree(p->work);
    if (p->sync) cudaFree(p->sync);
    if (p->stream2) cudaStreamSynchronize(p->stream2);
    if (p->stream3) cudaStreamSynchronize(p->stream3);
    if (p->mid) cudaFree(p->mid);
    if (p->sendbuf) cudaFree(p->sendbuf);
    if (p->done_ctr) cudaFree(p->done_ctr);
    if (p->dbg) cudaFree(p->dbg);
    if (p->ev_join) cudaEventDestroy(p->ev_join);
    for (auto& e : p->evb) if (e) cudaEventDestroy(e);
    for (auto& e : p->ev_y) if (e) cudaEventDestroy(e);
    for (auto& e : p->ev_a) if (e) cudaEventDestroy(e);
    if (p->stream2) cudaStreamDestroy(p->stream2);
    if (p->stream3) cudaStreamDestroy(p->stream3);
    if (p->part_done) cudaFree(p->part_done);
    if (p->plane_done) cudaFree(p->plane_done);
    if (p->ticket) cudaFree(p->ticket);
    if (p->lut_z) cudaFree(p->lut_z);
    if (p->lut_y) cudaFree(p->lut_y);
    if (p->lut_x) cudaFree(p->lut_x);
    if (p->lut_xn) cudaFree(p->lut_xn);
    if (p->lut_tz) cudaFree(p->lut_tz);
    if (p->lut_ty) cudaFree(p->lut_ty);
    if (p->lut_tx) cudaFree(p->lut_tx);
    for (auto& e : p->ev) if (e) cudaEventDestroy(e);
    for (auto& pe : p->pev) for (auto& e : pe) if (e) cudaEventDestroy(e);
    if (p->stream) cudaStreamDestroy(p->stream);
    cudaGetLastError();
    delete p;
    return 0;
}

extern "C" int dfft_cleanup(void) { return 0; }

extern "C" int dfft_memcpy(void* dst, const void* src, size_t bytes, int kind)
{
    CU(cudaMemcpy(dst, src, bytes, kind == 1 ? cudaMemcpyHostToDevice : (kind == 2 ? cudaMemcpyDeviceToHost : cudaMemcpyDefault)));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// pass launches
// ------------------------------------------------------------------------------------------------
// start gate / completion signal folded into a pass kernel (TileArgs::wait_flags, TileArgs::sig) instead of separate
// one-CTA launches: `which` 0 = ready[], 1 = arrive[], 2 + k = part_arrive[k]
struct Fold {
    int wait_which = -1; unsigned long long wait_val = 0;
    int sig_which = -1; unsigned long long sig_val = 0;
    int ctr = 0;     // which done_ctr word counts the finished CTAs of this launch
};
template <typename T> static void apply_fold(dfft_plan p, TileArgs<T>& a, const Fold* f)
{
    if (!f || p->dry || !p->sync) return;
    auto mine = [&](int w) -> const unsigned long long* { return w == 0 ? p->sync->ready : (w == 1 ? p->sync->arrive : p->sync->part_arrive[w - 2]); };
    if (f->wait_which >= 0 && f->wait_val > 0) { a.wait_flags = mine(f->wait_which); a.wait_val = f->wait_val; a.wait_n = p->P; }
    if (f->sig_which >= 0) {
        a.sig_n = p->P; a.sig_val = f->sig_val; a.done_ctr = p->done_ctr + f->ctr;
        for (int q = 0; q < p->P; q++) {
            SyncBlock* sb = p->peer_sync[q];
            a.sig[q] = f->sig_which == 0 ? &sb->ready[p->me] : (f->sig_which == 1 ? &sb->arrive[p->me] : &sb->part_arrive[f->sig_which - 2][p->me]);
        }
    }
}

template <typename T> struct Pass {
    static int launch(dfft_plan p, const SizeEntry* e, int kind, TileArgs<T>& a, int axis_override = -1, cudaStream_t st = nullptr)
    {
        if (!st) st = p->stream;
        a.inv = p->direction == DFFT_BACKWARD ? 1 : 0;
        a.gen = e->gen;
        const int axis = axis_override >= 0 ? axis_override : (kind == PK_Z ? 0 : (kind == PK_Y || kind == PK_Y_CO || kind == PK_Y_CI ? 1 : 2));
        if (p->dry) {
            static const char* names[PK_COUNT] = {"Z", "Y", "Y_CO", "Y_CI", "XF", "XB", "XB_CO", "XF_TW"};
            const int C = kind == PK_Z ? e->z_C : (kind == PK_Y || kind == PK_Y_CI ? e->s_C : (kind == PK_Y_CO ? e->p_C : e->x_C));
            // phase 1 = runs after the exchange has delivered this device's receive buffer
            const bool fwd = p->direction == DFFT_FORWARD;
            const int phase = fwd ? (axis == 2 ? 1 : 0) : (axis == 2 ? 0 : 1);
            record_op<T>(p, names[kind], phase, e->N, C, kind == PK_Y_CI, kind == PK_Y_CO || kind == PK_XB_CO, kind == PK_XF || kind == PK_XF_TW, a);
            p->launches++;
            return 0;
        }
        if (!p->in_pipe) ev_record(p, p->pev[axis][0]);
        cudaError_t err = e->launch[kind](&a, p->sms, st);
        if (!p->in_pipe) ev_record(p, p->pev[axis][1]);
        if (err != cudaSuccess) return fail(DFFT_ECUDA, "pass launch (kind %d, N=%d) failed: %s", kind, e->N, cudaGetErrorString(err));
        p->launches++;
        return 0;
    }
    // one TMA-pipelined pass (fft_tma.cuh).  Tensor sides are described as (base, d1, d2, s1, s2, axis): a 3-D tensor of
    // complex elements, row length `d0`, dim1/dim2 extents and element strides, transform axis = tensor dim `axis` (1 or 2)
    struct TmaTensor { void* base; long long d0, d1, d2, s1, s2; };
    static int launch_tma(dfft_plan p, const TmaEntry* e, int mode, TmaArgs<T>& a, const TmaTensor* tin, const TmaTensor* tout, int axis,
                          cudaStream_t st = nullptr)
    {
        if (!st) st = p->stream;
        alignas(64) unsigned char mi[128], mo[128];
        const int rows = e->rows;
        const TmaTensor* ts[2] = {tin, tout};
        unsigned char* ms[2] = {mi, mo};
        for (int k = 0; k < 2; k++) {
            if (!ts[k]) continue;
            const int b1 = mode == TMA_Y ? rows : 1, b2 = mode == TMA_Y ? 1 : rows;
            const int rc = tma_encode_3d(ms[k], ts[k]->base, p->prec, ts[k]->d0, ts[k]->d1, ts[k]->d2, ts[k]->s1, ts[k]->s2, e->C, b1, b2);
            if (rc != 0) return fail(DFFT_ECUDA, "cuTensorMapEncodeTiled failed (%d) for a %lldx%lldx%lld tensor", rc, ts[k]->d0, ts[k]->d1, ts[k]->d2);
        }
        a.inv = p->direction == DFFT_BACKWARD ? 1 : 0;
        if (!p->in_pipe) ev_record(p, p->pev[axis][0]);
        cudaError_t err = e->launch(mode, &a, tin ? mi : nullptr, tout ? mo : nullptr, p->sms, st);
        if (!p->in_pipe) ev_record(p, p->pev[axis][1]);
        if (err != cudaSuccess) return fail(DFFT_ECUDA, "TMA pass launch (mode %d, N=%d) failed: %s", mode, e->N, cudaGetErrorString(err));
        p->launches++;
        return 0;
    }
    // contiguous lines of length N2 (n0l*N1 lines), src -> dst (in place when equal)
    static int z_pass(dfft_plan p, const void* src, void* dst, bool scale)
    {
        const Geom& g = p->g;
        if (p->tz && (p->tz->use & (1u << TMA_Z)) && !p->dry && (p->n0l * g.n1) % p->tz->C == 0) {
            TmaArgs<T> t{};
            t.in = (const cx<T>*)src; t.out = (cx<T>*)dst; t.lut = (const cx<T>*)p->lut_tz;
            t.ntiles = p->n0l * g.n1 / p->tz->C; t.G = (int)std::min<long long>(t.ntiles, 0x7fffffff);
            t.in_SA = t.out_SA = (long long)t.G * p->tz->C * g.n2;   // a = tile / G: only needed beyond 2^31 tiles
            t.do_scale = scale ? 1 : 0; t.scale = (T)(1.0 / ((double)g.n0 * (double)g.n1 * (double)g.n2));
            return launch_tma(p, p->tz, TMA_Z, t, nullptr, nullptr, 0);
        }
        TileArgs<T> a{};
        const int C = p->ez->z_C;
        const long long nlines = p->n0l * g.n1;
        a.in = (const cx<T>*)src; a.out = (cx<T>*)dst; a.lut = (const cx<T>*)p->lut_z;
        a.G = (int)cdiv(nlines, C); a.W = (int)std::min<long long>(nlines, 0x7fffffff); a.ntiles = a.G;
        a.ia = Affine{0, (long long)C * g.n2, g.n2, 1}; a.oa = a.ia;
        a.do_scale = scale ? 1 : 0; a.scale = (T)(1.0 / ((double)g.n0 * (double)g.n1 * (double)g.n2));
        return launch(p, p->ez, PK_Z, a);
    }
    // columns of length N1 (stride N2) of every local plane.  mode 0: src -> dst natural (in place when equal)
    // mode 1: chunked (packed / peer) store, mode 2: chunked (unpack) load
    static int y_pass(dfft_plan p, const void* src, void* dst, int mode, void* const* chunk_base, const Fold* fold = nullptr)
    {
        const Geom& g = p->g;
        if (mode == 0 && p->ty && (p->ty->use & (1u << TMA_Y)) && !p->dry && g.n2 % p->ty->C == 0) {
            TmaArgs<T> t{};
            t.lut = (const cx<T>*)p->lut_ty;
            t.G = (int)(g.n2 / p->ty->C); t.ntiles = p->n0l * t.G;
            TmaTensor ti{(void*)src, g.n2, g.n1, p->n0l, g.n2, g.n1 * g.n2}, to{dst, g.n2, g.n1, p->n0l, g.n2, g.n1 * g.n2};
            return launch_tma(p, p->ty, TMA_Y, t, &ti, &to, 1);
        }
        TileArgs<T> a{};
        const int C = mode == 1 ? p->ey->p_C : p->ey->s_C;
        a.in = (const cx<T>*)src; a.out = (cx<T>*)dst; a.lut = (const cx<T>*)p->lut_y;
        a.G = (int)cdiv(g.n2, C); a.W = (int)g.n2; a.ntiles = p->n0l * a.G;
        a.ia = Affine{g.n1 * g.n2, C, 1, g.n2}; a.oa = a.ia;
        if (mode != 0) {
            ChunkTab& ct = mode == 1 ? a.co : a.ci;
            ct.ediv = (int)g.yd(); ct.nchunks = p->P;
            for (int q = 0; q < p->P; q++) { ct.cptr[q] = chunk_base[q]; ct.SAq[q] = g.n1l(q) * g.n2; }
        }
        apply_fold<T>(p, a, fold);
        return launch(p, p->ey, mode == 0 ? PK_Y : (mode == 1 ? PK_Y_CO : PK_Y_CI), a);
    }
    // t0 in one persistent kernel (square planes): forward Z (zsrc -> mid) then Y (mid -> ydst, or chunked);
    // backward Y (ysrc or chunked -> mid) then Z (mid -> mid).  ymode as in y_pass.
    static int zy_fused(dfft_plan p, const void* src, void* mid, void* dst, int ymode, void* const* chunk_base, bool scale, const Fold* fold = nullptr)
    {
        const Geom& g = p->g;
        const SizeEntry* e = p->ez;
        const bool fwd = p->direction == DFFT_FORWARD;
        TileArgs<T> z{}, y{};
        const int CZ = (fwd && ymode == 1) ? e->f_zCp : e->f_zC, CY = (fwd && ymode == 1) ? e->p_C : e->s_C;
        z.lut = (const cx<T>*)p->lut_z; y.lut = (const cx<T>*)p->lut_y;
        z.inv = y.inv = fwd ? 0 : 1;
        // contiguous role, tiled per plane: tile (plane, b) = CZ lines starting at line b*CZ of the plane
        z.G = (int)cdiv(g.n1, CZ); z.W = (int)g.n1; z.ntiles = p->n0l * z.G;
        z.ia = Affine{g.n1 * g.n2, (long long)CZ * g.n2, g.n2, 1}; z.oa = z.ia;
        z.do_scale = scale ? 1 : 0; z.scale = (T)(1.0 / ((double)g.n0 * (double)g.n1 * (double)g.n2));
        y.G = (int)cdiv(g.n2, CY); y.W = (int)g.n2; y.ntiles = p->n0l * y.G;
        y.ia = Affine{g.n1 * g.n2, CY, 1, g.n2}; y.oa = y.ia;
        if (ymode != 0) {
            ChunkTab& ct = ymode == 1 ? y.co : y.ci;
            ct.ediv = (int)g.yd(); ct.nchunks = p->P;
            for (int q = 0; q < p->P; q++) { ct.cptr[q] = chunk_base[q]; ct.SAq[q] = g.n1l(q) * g.n2; }
        }
        if (fwd) { z.in = (const cx<T>*)src; z.out = (cx<T>*)mid; y.in = (const cx<T>*)mid; y.out = (cx<T>*)dst; }
        else { y.in = (const cx<T>*)src; y.out = (cx<T>*)mid; z.in = (const cx<T>*)mid; z.out = (cx<T>*)mid; }
        FusedCtl c{};
        c.plane_done = p->plane_done; c.ticket = p->ticket; c.planes = p->n0l;
        c.GA = fwd ? z.G : y.G; c.GB = fwd ? y.G : z.G;
        c.target = ++p->fuse_epoch * (unsigned long long)c.GA;
        c.lag = p->lag;
        const int kind = fwd ? (ymode == 1 ? FK_ZY_CO : FK_ZY) : (ymode == 2 ? FK_YZ_CI : FK_YZ);
        apply_fold<T>(p, fwd ? y : z, fold);   // fft_fused2_kernel gates on / signals through its second role's arguments
        if (p->dry) {
            z.gen = y.gen = nullptr;
            if (fwd) { record_op<T>(p, "fusedZ", 0, e->N, CZ, false, false, false, z); record_op<T>(p, "fusedY", 0, e->N, CY, false, ymode == 1, false, y); }
            else { record_op<T>(p, "fusedY", 1, e->N, CY, ymode == 2, false, false, y); record_op<T>(p, "fusedZ", 1, e->N, CZ, false, false, false, z); }
            p->launches++;
            return 0;
        }
        ev_record(p, p->pev[0][0]);
        cudaError_t err = fwd ? e->fused[kind](&z, &y, &c, p->sms, p->stream) : e->fused[kind](&y, &z, &c, p->sms, p->stream);
        ev_record(p, p->pev[0][1]);
        ev_record(p, p->pev[1][0]);
        ev_record(p, p->pev[1][1]);
        if (err != cudaSuccess) return fail(DFFT_ECUDA, "fused t0 launch (kind %d, N=%d) failed: %s", kind, e->N, cudaGetErrorString(err));
        p->launches++;
        return 0;
    }
    // forward t0 + t1 + t2 + t3 in one kernel (P2P, square planes): Z: buf1 -> mid, Y: mid -> peers' work, X: work -> buf2
    static int fwd_overlapped(dfft_plan p, void* const* peer_base)
    {
        const Geom& g = p->g;
        const SizeEntry* e = p->ez;
        TileArgs<T> z{}, y{}, x{};
        const int CZ = e->f_zCp, CY = e->p_C, CX = e->x_C;
        z.lut = (const cx<T>*)p->lut_z; y.lut = (const cx<T>*)p->lut_y; x.lut = (const cx<T>*)p->lut_x;
        z.G = (int)cdiv(g.n1, CZ); z.W = (int)g.n1; z.ntiles = p->n0l * z.G;
        z.ia = Affine{g.n1 * g.n2, (long long)CZ * g.n2, g.n2, 1}; z.oa = z.ia;
        z.in = (const cx<T>*)p->buf1; z.out = (cx<T>*)p->mid;
        y.G = (int)cdiv(g.n2, CY); y.W = (int)g.n2; y.ntiles = p->n0l * y.G;
        y.ia = Affine{g.n1 * g.n2, CY, 1, g.n2}; y.oa = y.ia;
        y.in = (const cx<T>*)p->mid; y.out = nullptr;
        y.co.ediv = (int)g.yd(); y.co.nchunks = p->P;
        for (int q = 0; q < p->P; q++) { y.co.cptr[q] = peer_base[q]; y.co.SAq[q] = g.n1l(q) * g.n2; }
        x.G = (int)cdiv(g.n2, CX); x.W = (int)g.n2; x.ntiles = p->n1l * x.G;
        x.ia = Affine{g.n2, CX, 1, p->n1l * g.n2};
        x.oa = Affine{g.n2 * g.n0, (long long)CX * g.n0, g.n0, 1};
        x.in = (const cx<T>*)p->work; x.out = (cx<T>*)p->buf2;
        Fused3Ctl c{};
        c.plane_done = p->plane_done; c.ticket = p->ticket; c.part_done = p->part_done;
        c.planes = p->n0l; c.rows = p->n1l; c.P = p->P; c.me = p->me;
        c.K = p->parts;
        c.GA = z.G; c.GB = y.G; c.GBk = y.G / c.K; c.GX = x.G; c.GXk = x.G / c.K;
        c.target = ++p->fuse_epoch * (unsigned long long)c.GA;
        c.epoch = ++p->overlap_epoch;
        c.part_target = c.epoch * (unsigned long long)(p->n0l * c.GBk);
        if (!p->dry) {
            c.my_arrive = &p->sync->part_arrive[0][0];
            for (int q = 0; q < p->P; q++) c.peer_arrive[q] = &p->peer_sync[q]->part_arrive[0][0];
        }
        c.lag = p->lag;
        c.dbg = nullptr;
        if (!p->dry && getenv("DFFT_DEBUG_TIMELINE")) {
            if (!p->dbg) cudaMalloc((void**)&p->dbg, 16 * sizeof(unsigned long long));
            cudaMemsetAsync(p->dbg, 0xff, 4 * sizeof(unsigned long long), p->stream);
            cudaMemsetAsync(p->dbg + 4, 0, 12 * sizeof(unsigned long long), p->stream);
            c.dbg = p->dbg;
        }
        if (p->dry) {
            record_op<T>(p, "ovlZ", 0, e->N, CZ, false, false, false, z);
            record_op<T>(p, "ovlY", 0, e->N, CY, false, true, false, y);
            record_op<T>(p, "ovlX", 1, e->N, CX, false, false, true, x);
            p->launches++;
            return 0;
        }
        ev_record(p, p->pev[0][0]);
        cudaError_t err = e->fused3(&z, &y, &x, &c, p->sms, p->stream);
        ev_record(p, p->pev[0][1]);
        for (int a = 1; a < 3; a++) { ev_record(p, p->pev[a][0]); ev_record(p, p->pev[a][1]); }
        if (err != cudaSuccess) return fail(DFFT_ECUDA, "overlapped forward launch (N=%d) failed: %s", e->N, cudaGetErrorString(err));
        p->launches++;
        return 0;
    }
    // X transform that keeps the natural [x][y][z] layout (single device): columns along x, stride N1*N2, src -> dst
    static int x_natural(dfft_plan p, const void* src, void* dst)
    {
        const Geom& g = p->g;
        TileArgs<T> a{};
        const int C = p->ex->s_C;
        a.in = (const cx<T>*)src; a.out = (cx<T>*)dst; a.lut = (const cx<T>*)p->lut_xn;
        a.G = (int)cdiv(g.n2, C); a.W = (int)g.n2; a.ntiles = g.n1 * a.G;
        a.ia = Affine{g.n2, C, 1, g.n1 * g.n2}; a.oa = a.ia;
        return launch(p, p->ex, PK_Y, a, 2);   // a strided-local kernel, timed as the X pass
    }
    // forward X: src = [x][y_l][z] -> dst = [y_l][z][x]
    static bool x_fwd_folds(dfft_plan p) { return !(p->tx && (p->tx->use & (1u << TMA_XF)) && !p->dry && p->g.n2 % p->tx->C == 0); }
    static int x_fwd(dfft_plan p, const void* src, void* dst, const Fold* fold = nullptr)
    {
        const Geom& g = p->g;
        if (p->tx && (p->tx->use & (1u << TMA_XF)) && !p->dry && g.n2 % p->tx->C == 0) {
            TmaArgs<T> t{};
            t.lut = (const cx<T>*)p->lut_tx; t.out = (cx<T>*)dst;
            t.G = (int)(g.n2 / p->tx->C); t.ntiles = p->n1l * t.G; t.out_SA = g.n2 * g.n0;
            TmaTensor ti{(void*)src, g.n2, p->n1l, g.n0, g.n2, p->n1l * g.n2};
            return launch_tma(p, p->tx, TMA_XF, t, &ti, nullptr, 2);
        }
        TileArgs<T> a{};
        const int C = p->ex->x_C;
        a.in = (const cx<T>*)src; a.out = (cx<T>*)dst; a.lut = (const cx<T>*)p->lut_x;
        a.G = (int)cdiv(g.n2, C); a.W = (int)g.n2; a.ntiles = p->n1l * a.G;
        a.ia = Affine{g.n2, C, 1, p->n1l * g.n2};
        a.oa = Affine{g.n2 * g.n0, (long long)C * g.n0, g.n0, 1};
        apply_fold<T>(p, a, fold);
        return launch(p, p->ex, PK_XF, a);
    }
    // ---- z-part variants (stream-pipelined forward): part k of K covers the columns z in [k*zk, (k+1)*zk) ----------
    // Y pass of one z-part: mid[x_l][y][z in part] -> chunk q (the rows of destination device q) at chunk_base[q], laid out
    // [x_l][y_l(q)][z'] with row length zk: the part-major receive (P2P) / send (NCCL) layout
    static void y_part_args(dfft_plan p, TileArgs<T>& a, const void* src, long long zk, int k, void* const* chunk_base, int C)
    {
        const Geom& g = p->g;
        a.in = (const cx<T>*)src + k * zk; a.out = nullptr; a.lut = (const cx<T>*)p->lut_y;
        a.G = (int)cdiv(zk, C); a.W = (int)zk; a.ntiles = p->n0l * a.G;
        a.ia = Affine{g.n1 * g.n2, C, 1, g.n2};
        a.oa = Affine{0, C, 1, zk};
        a.co.ediv = (int)g.yd(); a.co.nchunks = p->P;
        for (int q = 0; q < p->P; q++) { a.co.cptr[q] = chunk_base[q]; a.co.SAq[q] = g.n1l(q) * zk; }
        if (p->xmode == DFFT_EXCHANGE_P2P && !p->dry && p->done_ctr) {
            // the kernel's last CTA publishes "part k of sender me has arrived" (epoch) on every receiving device
            a.sig_n = p->P; a.sig_val = p->epoch; a.done_ctr = p->done_ctr + k;
            for (int q = 0; q < p->P; q++) a.sig[q] = &p->peer_sync[q]->part_arrive[k][p->me];
        }
    }
    static int y_part(dfft_plan p, const void* src, long long zk, int k, void* const* chunk_base, int cap)
    {
        TileArgs<T> a{};
        y_part_args(p, a, src, zk, k, chunk_base, p->ey->p_C);
        a.max_ctas_per_sm = cap;
        return launch(p, p->ey, PK_Y_CO, a);
    }
    // part 0 together with the Z pass of every plane in one persistent kernel (fft_fused2_kernel): Z: src -> mid (L2),
    // Y part 0: mid -> chunks
    static int zy_fused_part0(dfft_plan p, const void* src, void* mid, long long zk, void* const* chunk_base)
    {
        const Geom& g = p->g;
        const SizeEntry* e = p->ez;
        TileArgs<T> z{}, y{};
        const int CZ = e->f_zCp, CY = e->p_C;
        z.lut = (const cx<T>*)p->lut_z;
        z.G = (int)cdiv(g.n1, CZ); z.W = (int)g.n1; z.ntiles = p->n0l * z.G;
        z.ia = Affine{g.n1 * g.n2, (long long)CZ * g.n2, g.n2, 1}; z.oa = z.ia;
        z.in = (const cx<T>*)src; z.out = (cx<T>*)mid;
        y_part_args(p, y, mid, zk, 0, chunk_base, CY);
        FusedCtl c{};
        c.plane_done = p->plane_done; c.ticket = p->ticket; c.planes = p->n0l;
        c.GA = z.G; c.GB = y.G;
        c.target = ++p->fuse_epoch * (unsigned long long)c.GA;
        c.lag = p->lag;
        if (p->dry) {
            record_op<T>(p, "fusedZ", 0, e->N, CZ, false, false, false, z);
            record_op<T>(p, "fusedY", 0, e->N, CY, false, true, false, y);
            p->launches++;
            return 0;
        }
        cudaError_t err = e->fused[FK_ZY_CO](&z, &y, &c, p->sms, p->stream);
        if (err != cudaSuccess) return fail(DFFT_ECUDA, "fused t0 (part 0) launch (N=%d) failed: %s", e->N, cudaGetErrorString(err));
        p->launches++;
        return 0;
    }
    // X pass of one z-part on the receive side: rpart = [x (all N0)][y_l][z'] (row length zk) -> dst[y_l][z in part][x]
    static void x_part_args(dfft_plan p, TileArgs<T>& a, const void* rpart, void* dst, long long zk, int k)
    {
        const Geom& g = p->g;
        const int C = p->ex->x_C;
        a.in = (const cx<T>*)rpart; a.out = (cx<T>*)dst + k * zk * g.n0; a.lut = (const cx<T>*)p->lut_x;
        a.G = (int)cdiv(zk, C); a.W = (int)zk; a.ntiles = p->n1l * a.G;
        a.ia = Affine{zk, C, 1, p->n1l * zk};
        a.oa = Affine{g.n2 * g.n0, (long long)C * g.n0, g.n0, 1};
    }
    // Y pass of part k (stores to the peers) and X pass of part k-1 (already arrived) in one two-role kernel
    static int yx_fused(dfft_plan p, const void* mid, long long zk, int k, void* const* chunk_base, const void* rpart_prev, void* dst)
    {
        const SizeEntry* e = p->ey;
        TileArgs<T> y{}, x{};
        y_part_args(p, y, mid, zk, k, chunk_base, e->p_C);
        x_part_args(p, x, rpart_prev, dst, zk, k - 1);
        YxCtl c{};
        c.ticket = p->ticket;
        c.TA = (unsigned)y.ntiles; c.TB = (unsigned)x.ntiles;
        if (p->dry) {
            record_op<T>(p, "Y_CO", 0, e->N, e->p_C, false, true, false, y);
            record_op<T>(p, "XF", 1, e->N, e->x_C, false, false, true, x);
            p->launches++;
            return 0;
        }
        cudaError_t err = e->fused_yx(&y, &x, &c, p->sms, p->stream);
        if (err != cudaSuccess) return fail(DFFT_ECUDA, "fused Y+X part launch (N=%d, part %d) failed: %s", e->N, k, cudaGetErrorString(err));
        p->launches++;
        return 0;
    }
    static int x_part(dfft_plan p, const void* rpart, void* dst, long long zk, int k, int cap, cudaStream_t st)
    {
        const Geom& g = p->g;
        // the TMA kernel takes the whole SM (one CTA, 3-slot ring): only for a part that overlaps nothing (the last one)
        if (cap == 0 && p->tx && (p->tx->use & (1u << TMA_XF)) && !p->dry && zk % p->tx->C == 0) {
            TmaArgs<T> t{};
            t.lut = (const cx<T>*)p->lut_tx; t.out = (cx<T>*)dst + k * zk * g.n0;
            t.G = (int)(zk / p->tx->C); t.ntiles = p->n1l * t.G; t.out_SA = g.n2 * g.n0;
            TmaTensor ti{(void*)rpart, zk, p->n1l, g.n0, zk, p->n1l * zk};
            return launch_tma(p, p->tx, TMA_XF, t, &ti, nullptr, 2, st);
        }
        TileArgs<T> a{};
        const int C = p->ex->x_C;
        a.in = (const cx<T>*)rpart; a.out = (cx<T>*)dst + k * zk * g.n0; a.lut = (const cx<T>*)p->lut_x;
        a.G = (int)cdiv(zk, C); a.W = (int)zk; a.ntiles = p->n1l * a.G;
        a.ia = Affine{zk, C, 1, p->n1l * zk};
        a.oa = Affine{g.n2 * g.n0, (long long)C * g.n0, g.n0, 1};
        a.max_ctas_per_sm = cap;
        return launch(p, p->ex, PK_XF, a, -1, st);
    }
    // ---- z-part variants of the BACKWARD passes (stream-pipelined backward) --------------------------------------------------
    // inverse X pass of one z-part: src[y_l][z in part][x] -> chunk p (= the x-planes of destination device p) at chunk_base[p],
    // laid out [x_l][y_l][z'] with row length zk
    static int xb_part(dfft_plan p, const void* src, long long zk, int k, void* const* chunk_base, int cap)
    {
        const Geom& g = p->g;
        TileArgs<T> a{};
        const int C = p->ex->x_C;
        a.in = (const cx<T>*)src + k * zk * g.n0; a.out = nullptr; a.lut = (const cx<T>*)p->lut_x;
        a.G = (int)cdiv(zk, C); a.W = (int)zk; a.ntiles = p->n1l * a.G;
        a.ia = Affine{g.n2 * g.n0, (long long)C * g.n0, g.n0, 1};
        a.oa = Affine{0, C, 1, p->n1l * zk};
        a.co.ediv = (int)g.xd(); a.co.nchunks = p->P;
        for (int q = 0; q < p->P; q++) { a.co.cptr[q] = chunk_base[q]; a.co.SAq[q] = zk; }
        if (p->xmode == DFFT_EXCHANGE_P2P && !p->dry && p->done_ctr) {
            a.sig_n = p->P; a.sig_val = p->epoch; a.done_ctr = p->done_ctr + k;
            for (int q = 0; q < p->P; q++) a.sig[q] = &p->peer_sync[q]->part_arrive[k][p->me];
        }
        a.max_ctas_per_sm = cap;
        return launch(p, p->ex, PK_XB_CO, a);
    }
    // inverse Y pass of one z-part on the receive side: rpart = [sender q][x_l][y_l(q)][z'] -> dst[x_l][y][z in part]
    static void yinv_part_args(dfft_plan p, TileArgs<T>& a, const void* rpart, void* dst, long long zk, int k, int C)
    {
        const Geom& g = p->g;
        a.in = nullptr; a.out = (cx<T>*)dst + k * zk; a.lut = (const cx<T>*)p->lut_y;
        a.G = (int)cdiv(zk, C); a.W = (int)zk; a.ntiles = p->n0l * a.G;
        a.ia = Affine{0, C, 1, zk};
        a.oa = Affine{g.n1 * g.n2, C, 1, g.n2};
        a.ci.ediv = (int)g.yd(); a.ci.nchunks = p->P;
        for (int q = 0; q < p->P; q++) { a.ci.cptr[q] = eoff((void*)rpart, (long long)q * p->n0l * g.yd() * zk, p->esz); a.ci.SAq[q] = g.n1l(q) * zk; }
    }
    static int yinv_part(dfft_plan p, const void* rpart, void* dst, long long zk, int k, int cap, cudaStream_t st)
    {
        TileArgs<T> a{};
        yinv_part_args(p, a, rpart, dst, zk, k, p->ey->s_C);
        a.max_ctas_per_sm = cap;
        return launch(p, p->ey, PK_Y_CI, a, -1, st);
    }
    // the LAST part's inverse Y pass completes every plane: it runs fused with the inverse Z pass (fft_fused2_kernel, Y then Z)
    static int yz_fused_last_part(dfft_plan p, const void* rpart, void* dst, long long zk, int k, bool scale, cudaStream_t st)
    {
        const Geom& g = p->g;
        const SizeEntry* e = p->ez;
        TileArgs<T> z{}, y{};
        const int CZ = e->f_zC, CY = e->s_C;
        yinv_part_args(p, y, rpart, dst, zk, k, CY);
        y.inv = 1;
        z.lut = (const cx<T>*)p->lut_z; z.inv = 1;
        z.G = (int)cdiv(g.n1, CZ); z.W = (int)g.n1; z.ntiles = p->n0l * z.G;
        z.ia = Affine{g.n1 * g.n2, (long long)CZ * g.n2, g.n2, 1}; z.oa = z.ia;
        z.in = (const cx<T>*)dst; z.out = (cx<T>*)dst;
        z.do_scale = scale ? 1 : 0; z.scale = (T)(1.0 / ((double)g.n0 * (double)g.n1 * (double)g.n2));
        FusedCtl c{};
        c.plane_done = p->plane_done; c.ticket = p->ticket; c.planes = p->n0l;
        c.GA = y.G; c.GB = z.G;
        c.target = ++p->fuse_epoch * (unsigned long long)c.GA;
        c.lag = p->lag;
        if (p->dry) {
            record_op<T>(p, "fusedY", 1, e->N, CY, true, false, false, y);
            record_op<T>(p, "fusedZ", 1, e->N, CZ, false, false, false, z);
            p->launches++;
            return 0;
        }
        cudaError_t err = e->fused[FK_YZ_CI](&y, &z, &c, p->sms, st);
        if (err != cudaSuccess) return fail(DFFT_ECUDA, "fused inverse t0 (last part) launch (N=%d) failed: %s", e->N, cudaGetErrorString(err));
        p->launches++;
        return 0;
    }
    // backward X: src = [y_l][z][x] -> dst = [x][y_l][z] (chunked by destination device when chunk_base)
    static int x_bwd(dfft_plan p, const void* src, void* dst, void* const* chunk_base, const Fold* fold = nullptr)
    {
        const Geom& g = p->g;
        if (!chunk_base && p->tx && (p->tx->use & (1u << TMA_XB)) && !p->dry && g.n2 % p->tx->C == 0) {
            TmaArgs<T> t{};
            t.lut = (const cx<T>*)p->lut_tx; t.in = (const cx<T>*)src;
            t.G = (int)(g.n2 / p->tx->C); t.ntiles = p->n1l * t.G; t.in_SA = g.n2 * g.n0;
            TmaTensor to{dst, g.n2, p->n1l, g.n0, g.n2, p->n1l * g.n2};
            return launch_tma(p, p->tx, TMA_XB, t, nullptr, &to, 2);
        }
        TileArgs<T> a{};
        const int C = p->ex->x_C;
        a.in = (const cx<T>*)src; a.out = (cx<T>*)dst; a.lut = (const cx<T>*)p->lut_x;
        a.G = (int)cdiv(g.n2, C); a.W = (int)g.n2; a.ntiles = p->n1l * a.G;
        a.ia = Affine{g.n2 * g.n0, (long long)C * g.n0, g.n0, 1};
        a.oa = Affine{g.n2, C, 1, p->n1l * g.n2};
        if (chunk_base) {
            a.co.ediv = (int)g.xd(); a.co.nchunks = p->P;
            for (int q = 0; q < p->P; q++) { a.co.cptr[q] = chunk_base[q]; a.co.SAq[q] = g.n2; }
        }
        if (chunk_base) apply_fold<T>(p, a, fold);
        return launch(p, p->ex, chunk_base ? PK_XB_CO : PK_XB, a);
    }
};


// exchange offsets (api.cpp:84-133, 613-627): where chunk (sender s -> receiver r) starts
static long long send_off(const Geom& g, int s, int r, int dir)
{
    return dir == DFFT_FORWARD ? (long long)r * g.n0l(s) * g.yd() * g.n2 : (long long)r * g.xd() * g.n1l(s) * g.n2;
}
static long long recv_off(const Geom& g, int s, int r, int dir)
{
    return dir == DFFT_FORWARD ? (long long)s * g.xd() * g.n1l(r) * g.n2 : (long long)s * g.n0l(r) * g.yd() * g.n2;
}
static long long xchg_count(const Geom& g, int s, int r, int dir)
{
    return dir == DFFT_FORWARD ? g.n0l(s) * g.n1l(r) * g.n2 : g.n0l(r) * g.n1l(s) * g.n2;
}

/* the reference's TransInfo table (fft_mpi_common.h:24-29, filled at api.cpp:84-133) */
extern "C" int dfft_exchange_table(long long n0, long long n1, long long n2, int P, int dev, int direction, long long* scount,
                                   long long* soffset, long long* rcount, long long* roffset)
{
    if (P < 1 || dev < 0 || dev >= P || (direction != DFFT_FORWARD && direction != DFFT_BACKWARD)) return fail(DFFT_EINVAL, "bad arguments");
    Geom g{n0, n1, n2, P};
    if (g.last_n0() < 1 || g.last_n1() < 1) return fail(DFFT_EUNSUPPORTED, "empty last slab");
    for (int i = 0; i < P; i++) {
        if (scount) scount[i] = xchg_count(g, dev, i, direction);
        if (soffset) soffset[i] = send_off(g, dev, i, direction);
        if (rcount) rcount[i] = xchg_count(g, i, dev, direction);
        if (roffset) roffset[i] = recv_off(g, i, dev, direction);
    }
    return 0;
}

// which: 0 = ready[], 1 = arrive[], 2 + k = part_arrive[k][]
static int flags_signal(dfft_plan p, int which, unsigned long long value, cudaStream_t st = nullptr)
{
    if (p->dry) return 0;
    FlagPtrs fp{};
    for (int q = 0; q < p->P; q++) {
        SyncBlock* sb = p->peer_sync[q];
        fp.p[q] = which == 1 ? &sb->arrive[p->me] : (which == 0 ? &sb->ready[p->me] : &sb->part_arrive[which - 2][p->me]);
    }
    signal_flags_kernel<<<1, DFFT_MAX_CHUNKS, 0, st ? st : p->stream>>>(fp, p->P, value);
    CU(cudaGetLastError());
    p->launches++;
    return 0;
}
static int flags_wait(dfft_plan p, int which, unsigned long long value, cudaStream_t st = nullptr)
{
    if (value == 0 || p->dry) return 0;
    const unsigned long long* f = which == 1 ? p->sync->arrive : (which == 0 ? p->sync->ready : p->sync->part_arrive[which - 2]);
    wait_flags_kernel<<<1, DFFT_MAX_CHUNKS, 0, st ? st : p->stream>>>(f, p->P, value);
    CU(cudaGetLastError());
    p->launches++;
    return 0;
}

static int nccl_exchange(dfft_plan p, const void* sendbuf, void* recvbuf)
{
    const Geom& g = p->g;
    const int dir = p->direction;
    if (p->dry) {   // describe the all-to-all: element offsets and counts of every chunk this device sends
        char buf[160];
        std::string o = "{\"op\": \"alltoall\", \"phase\": 0, ";
        snprintf(buf, sizeof(buf), "\"send\": %llu, \"recv\": %llu, \"esz\": %zu, \"chunks\": [", (unsigned long long)(size_t)sendbuf,
                 (unsigned long long)(size_t)recvbuf, p->esz);
        o += buf;
        for (int q = 0; q < p->P; q++) {
            snprintf(buf, sizeof(buf), "%s[%d, %lld, %lld, %lld]", q ? ", " : "", q, send_off(g, p->me, q, dir), recv_off(g, p->me, q, dir), xchg_count(g, p->me, q, dir));
            o += buf;
        }
        o += "]}";
        p->ops.push_back(o);
        p->launches++;
        return 0;
    }
    NcclApi& api = nccl_api();
    bool even = true;
    for (int q = 0; q < p->P; q++)
        if (xchg_count(g, p->me, q, dir) != xchg_count(g, 0, 0, dir) || xchg_count(g, q, p->me, dir) != xchg_count(g, 0, 0, dir)) even = false;
    if (even && api.AlltoAll && !getenv("DFFT_NCCL_SENDRECV")) {
        NC(api.AlltoAll(sendbuf, recvbuf, (size_t)xchg_count(g, 0, 0, dir) * p->esz, /*ncclInt8*/ 0, p->nccl, p->stream));
    } else {
        NC(api.GroupStart());
        for (int q = 0; q < p->P; q++) {
            NC(api.Send(eoff((void*)sendbuf, send_off(g, p->me, q, dir), p->esz), (size_t)xchg_count(g, p->me, q, dir) * p->esz, 0, q, p->nccl, p->stream));
            NC(api.Recv(eoff(recvbuf, recv_off(g, q, p->me, dir), p->esz), (size_t)xchg_count(g, q, p->me, dir) * p->esz, 0, q, p->nccl, p->stream));
        }
        NC(api.GroupEnd());
    }
    p->launches++;
    return 0;
}

// one z-part of the all-to-all in NCCL mode (even split): `count` elements to / from every device, chunk q of the send
// part at q*count, the chunk received from device s at s*count of the receive part
static int nccl_exchange_part(dfft_plan p, const void* sendpart, void* recvpart, long long count, cudaStream_t st)
{
    if (p->dry) {
        char buf[160];
        std::string o = "{\"op\": \"alltoall\", \"phase\": 0, ";
        snprintf(buf, sizeof(buf), "\"send\": %llu, \"recv\": %llu, \"esz\": %zu, \"chunks\": [", (unsigned long long)(size_t)sendpart,
                 (unsigned long long)(size_t)recvpart, p->esz);
        o += buf;
        for (int q = 0; q < p->P; q++) {
            snprintf(buf, sizeof(buf), "%s[%d, %lld, %lld, %lld]", q ? ", " : "", q, (long long)q * count, (long long)p->me * count, count);
            o += buf;
        }
        o += "]}";
        p->ops.push_back(o);
        p->launches++;
        return 0;
    }
    NcclApi& api = nccl_api();
    if (api.AlltoAll && !getenv("DFFT_NCCL_SENDRECV")) {
        NC(api.AlltoAll(sendpart, recvpart, (size_t)count * p->esz, /*ncclInt8*/ 0, p->nccl, st));
    } else {
        NC(api.GroupStart());
        for (int q = 0; q < p->P; q++) {
            NC(api.Send(eoff((void*)sendpart, (long long)q * count, p->esz), (size_t)count * p->esz, 0, q, p->nccl, st));
            NC(api.Recv(eoff(recvpart, (long long)q * count, p->esz), (size_t)count * p->esz, 0, q, p->nccl, st));
        }
        NC(api.GroupEnd());
    }
    p->launches++;
    return 0;
}

// Stream-pipelined forward transform (P > 1).  The reference runs t0, t1, t2, t3 back to back with a device-wide sync
// after each (fft_mpi_3d_api.cpp:181-201, 610-672: no overlap at all).  Here the z axis is cut into K parts:
//   send side, plan stream    : Z pass of the slab (fused with Y part 0 through L2 when the planes are square), then for
//                               every part k the Y pass of its columns, whose store IS the pack (t1) and -- P2P -- the
//                               all-to-all (t2): rows go straight into the peers' receive buffers over NVLink, followed by a
//                               per-part arrival flag.  NCCL: the packed part is handed to ncclAlltoAll on the comm stream.
//   receive side, second stream: as soon as part k has arrived from every sender, the X pass of the (y_l, z in part k)
//                               lines (t3, unpack + transpose folded into its load / store), while later parts are still
//                               being computed and sent.
// Both sides cap their resident CTAs per SM while they overlap so that they co-reside on every SM.
// Receive / send buffers are part-major: part k of device q = [x (all N0)][y_l][z'] with z' < zk at k * N0 * n1_l(q) * zk.
template <typename T> static int fwd_pipelined(dfft_plan p)
{
    const Geom& g = p->g;
    const int P = p->P, me = p->me, K = p->parts;
    const long long zk = g.n2 / K;
    const bool p2p = p->xmode == DFFT_EXCHANGE_P2P;
    cudaStream_t A = p->stream, B = p->stream2, Cs = p->stream3;
    int rc = 0;
    struct Guard { dfft_plan p; ~Guard() { p->in_pipe = false; } } guard{p};
    p->in_pipe = true;
    int cap = 1;
    if (getenv("DFFT_PIPE_CAP")) cap = atoi(getenv("DFFT_PIPE_CAP"));
    if (p2p) {
        p->epoch++;
        if ((rc = flags_wait(p, 0, p->epoch - 1))) return rc;   // every receiver has consumed the previous epoch
    }
    CU(ev_record(p, p->pev[0][0]));
    if (p->pipe_fyx) {
        // chain of two-role kernels on the plan stream: [Z + Y part 0] [Y part 1 + X part 0] ... [Y part K-1 + X part K-2] [X part K-1]
        for (int k = 0; k < K; k++) {
            void* base[DFFT_MAX_CHUNKS];
            for (int q = 0; q < P; q++) base[q] = eoff(p->peer_work[q], ((long long)k * g.n0 + (long long)me * g.xd()) * g.n1l(q) * zk, p->esz);
            if (k == 0) rc = Pass<T>::zy_fused_part0(p, p->buf1, p->mid, zk, base);
            else {
                // part k-1 must have arrived from every sender before the kernel whose X role consumes it starts: a one-CTA gate
                // kernel, not a poll inside the full-grid kernel (which would hold every SM slot while it waits, see execute_fused)
                if ((rc = flags_wait(p, 2 + k - 1, p->epoch, A))) return rc;
                rc = Pass<T>::yx_fused(p, p->mid, zk, k, base, eoff(p->work, (long long)(k - 1) * g.n0 * p->n1l * zk, p->esz), p->buf2);
            }
            if (rc) return rc;
            if (!p->done_ctr && (rc = flags_signal(p, 2 + k, p->epoch, A))) return rc;   // else the kernel's last CTA publishes the flags
        }
        CU(ev_record(p, p->pev[0][1]));
        CU(ev_record(p, p->pev[1][0])); CU(ev_record(p, p->pev[1][1]));
        CU(ev_record(p, p->ev[1]));
        if ((rc = flags_wait(p, 2 + K - 1, p->epoch, A))) return rc;
        CU(ev_record(p, p->evb[0]));
        CU(ev_record(p, p->pev[2][0]));
        if ((rc = Pass<T>::x_part(p, eoff(p->work, (long long)(K - 1) * g.n0 * p->n1l * zk, p->esz), p->buf2, zk, K - 1, 0, A))) return rc;
        CU(ev_record(p, p->pev[2][1]));
        CU(ev_record(p, p->evb[1]));
        if ((rc = flags_signal(p, 0, p->epoch, A))) return rc;
        CU(ev_record(p, p->ev[2]));
        CU(ev_record(p, p->ev[3]));
        p->timed = true;
        return 0;
    }
    for (int k = 0; k < K; k++) {
        void* base[DFFT_MAX_CHUNKS];
        for (int q = 0; q < P; q++)
            base[q] = p2p ? eoff(p->peer_work[q], ((long long)k * g.n0 + (long long)me * g.xd()) * g.n1l(q) * zk, p->esz)
                          : eoff(p->sendbuf, ((long long)k * P + q) * p->n0l * g.yd() * zk, p->esz);
        if (k == 0 && p->fuse) rc = Pass<T>::zy_fused_part0(p, p->buf1, p->mid, zk, base);
        else {
            if (k == 0 && (rc = Pass<T>::z_pass(p, p->buf1, p->mid, false))) return rc;
            rc = Pass<T>::y_part(p, p->mid, zk, k, base, k > 0 ? cap : 0);
        }
        if (rc) return rc;
        if (p2p) {
            if (!p->done_ctr && (rc = flags_signal(p, 2 + k, p->epoch, A))) return rc;   // else folded into the part kernel
        } else {
            const long long chunk = p->n0l * g.yd() * zk;
            CU(ev_record_on(p, p->ev_y[k], A));
            CU(stream_wait(p, Cs, p->ev_y[k]));
            if ((rc = nccl_exchange_part(p, eoff(p->sendbuf, (long long)k * P * chunk, p->esz), eoff(p->work, (long long)k * P * chunk, p->esz), chunk, Cs))) return rc;
            CU(ev_record_on(p, p->ev_a[k], Cs));
        }
    }
    CU(ev_record(p, p->pev[0][1]));
    CU(ev_record(p, p->pev[1][0]));
    CU(ev_record(p, p->pev[1][1]));
    CU(ev_record(p, p->ev[1]));
    for (int k = 0; k < K; k++) {
        if (p2p) { if ((rc = flags_wait(p, 2 + k, p->epoch, B))) return rc; }
        else CU(stream_wait(p, B, p->ev_a[k]));
        if (k == 0) CU(ev_record_on(p, p->pev[2][0], B));
        if (k == K - 1) CU(ev_record_on(p, p->evb[0], B));
        if ((rc = Pass<T>::x_part(p, eoff(p->work, (long long)k * g.n0 * p->n1l * zk, p->esz), p->buf2, zk, k, k < K - 1 ? cap : 0, B))) return rc;
    }
    CU(ev_record_on(p, p->pev[2][1], B));
    CU(ev_record_on(p, p->evb[1], B));
    if (p2p && (rc = flags_signal(p, 0, p->epoch, B))) return rc;
    CU(ev_record_on(p, p->ev_join, B));
    CU(stream_wait(p, A, p->ev_join));
    CU(ev_record(p, p->ev[2]));
    CU(ev_record(p, p->ev[3]));
    p->timed = true;
    return 0;
}

// Stream-pipelined backward transform (P > 1): the mirror image of fwd_pipelined.  Send side (plan stream): the inverse X
// pass of z-part k, whose chunked store drops the x-planes of every destination straight into its receive buffer (P2P) or
// into the part-major send buffer followed by ncclAlltoAll of the part (NCCL).  Receive side (second stream): as soon as part k
// has arrived from every sender, the inverse Y pass of its columns (unpack folded into the load); the last part's Y pass
// completes every plane and runs fused with the inverse Z pass.  Receive layout of device p, part k:
// [sender q][x_l][y_l(q)][z'] at k * n0_l(p) * N1 * zk + q * n0_l(p) * yd * zk.
template <typename T> static int bwd_pipelined(dfft_plan p)
{
    const Geom& g = p->g;
    const int P = p->P, me = p->me, K = p->parts;
    const long long zk = g.n2 / K;
    const bool p2p = p->xmode == DFFT_EXCHANGE_P2P;
    const bool scale = (p->flags & DFFT_SCALE_BACKWARD) != 0;
    cudaStream_t A = p->stream, B = p->stream2, Cs = p->stream3;
    int rc = 0;
    struct Guard { dfft_plan p; ~Guard() { p->in_pipe = false; } } guard{p};
    p->in_pipe = true;
    int cap = 1;
    if (getenv("DFFT_PIPE_CAP")) cap = atoi(getenv("DFFT_PIPE_CAP"));
    if (p2p) {
        p->epoch++;
        if ((rc = flags_wait(p, 0, p->epoch - 1))) return rc;
    }
    CU(ev_record(p, p->pev[2][0]));
    for (int k = 0; k < K; k++) {
        void* base[DFFT_MAX_CHUNKS];
        for (int q = 0; q < P; q++)
            base[q] = p2p ? eoff(p->peer_work[q], ((long long)k * g.n1 + (long long)me * g.yd()) * g.n0l(q) * zk, p->esz)
                          : eoff(p->sendbuf, ((long long)k * P + q) * g.xd() * p->n1l * zk, p->esz);
        if ((rc = Pass<T>::xb_part(p, p->buf1, zk, k, base, k > 0 ? cap : 0))) return rc;
        if (p2p) {
            if (!p->done_ctr && (rc = flags_signal(p, 2 + k, p->epoch, A))) return rc;
        } else {
            const long long chunk = g.xd() * p->n1l * zk;
            CU(ev_record_on(p, p->ev_y[k], A));
            CU(stream_wait(p, Cs, p->ev_y[k]));
            if ((rc = nccl_exchange_part(p, eoff(p->sendbuf, (long long)k * P * chunk, p->esz), eoff(p->work, (long long)k * P * chunk, p->esz), chunk, Cs))) return rc;
            CU(ev_record_on(p, p->ev_a[k], Cs));
        }
    }
    CU(ev_record(p, p->pev[2][1]));
    CU(ev_record(p, p->ev[1]));
    for (int k = 0; k < K; k++) {
        if (p2p) { if ((rc = flags_wait(p, 2 + k, p->epoch, B))) return rc; }
        else CU(stream_wait(p, B, p->ev_a[k]));
        if (k == 0) CU(ev_record_on(p, p->pev[1][0], B));
        if (k == K - 1) CU(ev_record_on(p, p->evb[0], B));
        const void* rpart = eoff(p->work, (long long)k * p->n0l * g.n1 * zk, p->esz);
        if (k == K - 1 && p->fuse) rc = Pass<T>::yz_fused_last_part(p, rpart, p->buf2, zk, k, scale, B);
        else rc = Pass<T>::yinv_part(p, rpart, p->buf2, zk, k, k < K - 1 ? cap : 0, B);
        if (rc) return rc;
    }
    CU(ev_record_on(p, p->pev[1][1], B));
    if (!p->fuse) {
        // inverse Z pass of the whole slab on the receive stream (Pass::z_pass launches on the plan stream: join first)
        CU(ev_record_on(p, p->ev_join, B));
        CU(stream_wait(p, A, p->ev_join));
        if ((rc = Pass<T>::z_pass(p, p->buf2, p->buf2, scale))) return rc;
        CU(ev_record(p, p->evb[1]));
        CU(ev_record(p, p->pev[0][0])); CU(ev_record(p, p->pev[0][1]));
        if (p2p && (rc = flags_signal(p, 0, p->epoch, A))) return rc;
    } else {
        CU(ev_record_on(p, p->pev[0][0], B)); CU(ev_record_on(p, p->pev[0][1], B));
        CU(ev_record_on(p, p->evb[1], B));
        if (p2p && (rc = flags_signal(p, 0, p->epoch, B))) return rc;
        CU(ev_record_on(p, p->ev_join, B));
        CU(stream_wait(p, A, p->ev_join));
    }
    CU(ev_record(p, p->ev[2]));
    CU(ev_record(p, p->ev[3]));
    p->timed = true;
    return 0;
}

template <typename T> static int execute_fused(dfft_plan p)
{
    const Geom& g = p->g;
    const int P = p->P, me = p->me;
    int rc;
    p->launches = 0;
    CU(ev_record(p, p->ev[0]));
    if (p->pipe) return p->direction == DFFT_FORWARD ? fwd_pipelined<T>(p) : bwd_pipelined<T>(p);
    if (p->direction == DFFT_FORWARD) {
        // t0 (+t1): Z pass out of place (bufferDev1 survives), Y pass with the pack (and, P2P, the
        // all-to-all) folded into its store
        if (P == 1) {
            if (p->fuse) {
                if ((rc = Pass<T>::zy_fused(p, p->buf1, p->work, p->work, 0, nullptr, false))) return rc;
            } else {
                if ((rc = Pass<T>::z_pass(p, p->buf1, p->work, false))) return rc;
                if ((rc = Pass<T>::y_pass(p, p->work, p->work, 0, nullptr))) return rc;
            }
            CU(ev_record(p, p->ev[1]));
            CU(ev_record(p, p->ev[2]));
            if (p->natural) { if ((rc = Pass<T>::x_natural(p, p->work, p->buf2))) return rc; }
            else if ((rc = Pass<T>::x_fwd(p, p->work, p->buf2))) return rc;
        } else if (p->xmode == DFFT_EXCHANGE_P2P) {
            void* base[DFFT_MAX_CHUNKS];
            for (int q = 0; q < P; q++) base[q] = eoff(p->peer_work[q], recv_off(g, me, q, DFFT_FORWARD), p->esz);
            p->epoch++;
            if (p->overlap) {
                if ((rc = flags_wait(p, 0, p->epoch - 1))) return rc;   // every receiver has consumed the previous epoch
                if ((rc = Pass<T>::fwd_overlapped(p, base))) return rc;
                CU(ev_record(p, p->ev[1]));
                CU(ev_record(p, p->ev[2]));
                if ((rc = flags_signal(p, 0, p->epoch))) return rc;
                CU(ev_record(p, p->ev[3]));
                p->timed = true;
                return 0;
            }
            // The completion SIGNALS ride inside the pass kernels (their last CTA publishes the flags: 4 launches per transform
            // instead of 6, DFFT_SIGNAL_KERNELS=1 restores the separate launches).  The GATES stay one-CTA kernels on purpose: a
            // full-grid kernel that spins on a peer's flag holds every SM slot, and with two plans in flight per device (bench.py's
            // e2e leg) device A can then wait for a kernel of device B that cannot start because B's SMs are held by a kernel waiting for A.
            const bool fold = p->done_ctr != nullptr && !p->dry;
            Fold fy; fy.sig_which = 1; fy.sig_val = p->epoch; fy.ctr = 0;
            Fold fx; fx.sig_which = 0; fx.sig_val = p->epoch; fx.ctr = 1;
            const bool foldx = fold && Pass<T>::x_fwd_folds(p);
            if (p->fuse) {
                if ((rc = flags_wait(p, 0, p->epoch - 1))) return rc;   // every receiver has consumed the previous epoch
                if ((rc = Pass<T>::zy_fused(p, p->buf1, p->buf2, nullptr, 1, base, false, fold ? &fy : nullptr))) return rc;
            } else {
                if ((rc = Pass<T>::z_pass(p, p->buf1, p->buf2, false))) return rc;
                if ((rc = flags_wait(p, 0, p->epoch - 1))) return rc;
                if ((rc = Pass<T>::y_pass(p, p->buf2, nullptr, 1, base, fold ? &fy : nullptr))) return rc;
            }
            if (!fold && (rc = flags_signal(p, 1, p->epoch))) return rc;
            CU(ev_record(p, p->ev[1]));
            if ((rc = flags_wait(p, 1, p->epoch))) return rc;        // t2: exposed wait for the slowest sender
            CU(ev_record(p, p->ev[2]));
            if ((rc = Pass<T>::x_fwd(p, p->work, p->buf2, foldx ? &fx : nullptr))) return rc;
            if (!foldx && (rc = flags_signal(p, 0, p->epoch))) return rc;
        } else {
            void* base[DFFT_MAX_CHUNKS];
            for (int q = 0; q < P; q++) base[q] = eoff(p->buf2, send_off(g, me, q, DFFT_FORWARD), p->esz);
            if (p->fuse) {
                if ((rc = Pass<T>::zy_fused(p, p->buf1, p->work, nullptr, 1, base, false))) return rc;
            } else {
                if ((rc = Pass<T>::z_pass(p, p->buf1, p->work, false))) return rc;
                if ((rc = Pass<T>::y_pass(p, p->work, nullptr, 1, base))) return rc;
            }
            CU(ev_record(p, p->ev[1]));
            if ((rc = nccl_exchange(p, p->buf2, p->work))) return rc;
            CU(ev_record(p, p->ev[2]));
            if ((rc = Pass<T>::x_fwd(p, p->work, p->buf2))) return rc;
        }
        CU(ev_record(p, p->ev[3]));
    } else {
        const bool scale = (p->flags & DFFT_SCALE_BACKWARD) != 0;
        if (P == 1) {
            if (p->natural) { if ((rc = Pass<T>::x_natural(p, p->buf1, p->buf2))) return rc; }
            else if ((rc = Pass<T>::x_bwd(p, p->buf1, p->buf2, nullptr))) return rc;
            CU(ev_record(p, p->ev[1]));
            CU(ev_record(p, p->ev[2]));
            if (p->fuse) { if ((rc = Pass<T>::zy_fused(p, p->buf2, p->buf2, nullptr, 0, nullptr, scale))) return rc; }
            else if ((rc = Pass<T>::y_pass(p, p->buf2, p->buf2, 0, nullptr))) return rc;
        } else if (p->xmode == DFFT_EXCHANGE_P2P) {
            p->epoch++;
            const bool fold = p->done_ctr != nullptr && !p->dry;
            Fold fxb; fxb.sig_which = 1; fxb.sig_val = p->epoch; fxb.ctr = 0;      // signals folded, gates separate (see the forward branch)
            Fold fyz; fyz.ctr = 1;
            if (p->fuse) { fyz.sig_which = 0; fyz.sig_val = p->epoch; }   // the fused kernel is the last one: it also signals "consumed"
            if ((rc = flags_wait(p, 0, p->epoch - 1))) return rc;
            void* base[DFFT_MAX_CHUNKS];
            for (int q = 0; q < P; q++) base[q] = eoff(p->peer_work[q], recv_off(g, me, q, DFFT_BACKWARD), p->esz);
            if ((rc = Pass<T>::x_bwd(p, p->buf1, nullptr, base, fold ? &fxb : nullptr))) return rc;
            if (!fold && (rc = flags_signal(p, 1, p->epoch))) return rc;
            CU(ev_record(p, p->ev[1]));
            if ((rc = flags_wait(p, 1, p->epoch))) return rc;
            CU(ev_record(p, p->ev[2]));
            void* cb[DFFT_MAX_CHUNKS];
            for (int q = 0; q < P; q++) cb[q] = eoff(p->work, (long long)q * p->n0l * g.yd() * g.n2, p->esz);
            if (p->fuse) { if ((rc = Pass<T>::zy_fused(p, nullptr, p->buf2, nullptr, 2, cb, scale, fold ? &fyz : nullptr))) return rc; }
            else if ((rc = Pass<T>::y_pass(p, nullptr, p->buf2, 2, cb, fold ? &fyz : nullptr))) return rc;
            if (!(fold && p->fuse) && (rc = flags_signal(p, 0, p->epoch))) return rc;
        } else {
            if ((rc = Pass<T>::x_bwd(p, p->buf1, p->buf2, nullptr))) return rc;
            CU(ev_record(p, p->ev[1]));
            if ((rc = nccl_exchange(p, p->buf2, p->work))) return rc;
            CU(ev_record(p, p->ev[2]));
            void* cb[DFFT_MAX_CHUNKS];
            for (int q = 0; q < P; q++) cb[q] = eoff(p->work, (long long)q * p->n0l * g.yd() * g.n2, p->esz);
            if (p->fuse) { if ((rc = Pass<T>::zy_fused(p, nullptr, p->buf2, nullptr, 2, cb, scale))) return rc; }
            else if ((rc = Pass<T>::y_pass(p, nullptr, p->buf2, 2, cb))) return rc;
        }
        if (!p->fuse && (rc = Pass<T>::z_pass(p, p->buf2, p->buf2, scale))) return rc;
        CU(ev_record(p, p->ev[3]));
    }
    p->timed = true;
    return 0;
}

// reference-like stage-by-stage execution (api.cpp:181-214 with its device-wide syncs)
template <typename T> static int execute_stage(dfft_plan p, int stage)
{
    const Geom& g = p->g;
    const int P = p->P, me = p->me, dir = p->direction;
    int rc = 0;
    // map "k-th executed stage" to the reference stage id
    const int sid = dir == DFFT_FORWARD ? stage : 3 - stage;
    if (sid == 0) {          // fftZY
        void* buf = dir == DFFT_FORWARD ? p->buf1 : p->buf2;
        if (dir == DFFT_FORWARD) {
            if ((rc = Pass<T>::z_pass(p, buf, buf, false))) return rc;
            if ((rc = Pass<T>::y_pass(p, buf, buf, 0, nullptr))) return rc;
        } else {
            if ((rc = Pass<T>::y_pass(p, buf, buf, 0, nullptr))) return rc;
            if ((rc = Pass<T>::z_pass(p, buf, buf, (p->flags & DFFT_SCALE_BACKWARD) != 0))) return rc;
        }
    } else if (sid == 1) {   // localTransposeUneven
        cudaError_t e = launch_pack_rows(p->buf1, p->buf2, (int)p->esz, p->n0l, g.n1, g.n2, P, dir == DFFT_FORWARD, p->sms, p->stream);
        if (e != cudaSuccess) return fail(DFFT_ECUDA, "pack launch failed: %s", cudaGetErrorString(e));
        p->launches++;
    } else if (sid == 2) {   // slabAlltoall
        if (P > 1) {
            CU(cudaStreamSynchronize(p->stream));
            p->comm->host_barrier(me);   // every sender's buf2 is packed, every receiver's buf1 is free
            for (int q = 0; q < P; q++) {
                CU(cudaMemcpyAsync(eoff(p->peer_buf1[q], recv_off(g, me, q, dir), p->esz), eoff(p->buf2, send_off(g, me, q, dir), p->esz),
                                   (size_t)xchg_count(g, me, q, dir) * p->esz, cudaMemcpyDefault, p->stream));
                p->launches++;
            }
            CU(cudaStreamSynchronize(p->stream));
            p->comm->host_barrier(me);
        } else {
            CU(cudaMemcpyAsync(p->buf1, p->buf2, (size_t)p->in_count * p->esz, cudaMemcpyDeviceToDevice, p->stream));
            p->launches++;
        }
    } else {                 // fftX
        if (dir == DFFT_FORWARD) rc = Pass<T>::x_fwd(p, p->buf1, p->buf2);
        else rc = Pass<T>::x_bwd(p, p->buf1, p->buf2, nullptr);
        if (rc) return rc;
    }
    CU(cudaStreamSynchronize(p->stream));
    return 0;
}

extern "C" int dfft_execute_stage(dfft_plan p, int stage)
{
    if (!p || stage < 0 || stage > 3 || p->dry) return fail(DFFT_EINVAL, "dfft_execute_stage: bad arguments");
    if (p->xmode != DFFT_EXCHANGE_STAGED) return fail(DFFT_EINVAL, "dfft_execute_stage needs a plan created with DFFT_EXCHANGE_STAGED");
    CU(cudaSetDevice(p->device));
    return p->prec == DFFT_DOUBLE ? execute_stage<double>(p, stage) : execute_stage<float>(p, stage);
}

extern "C" int dfft_execute(dfft_plan p)
{
    if (!p) return fail(DFFT_EINVAL, "null plan");
    if (p->dry) p->ops.clear();
    else CU(cudaSetDevice(p->device));
    if (p->xmode == DFFT_EXCHANGE_STAGED) {
        p->launches = 0;
        for (int s = 0; s < 4; s++) {
            CU(ev_record(p, p->ev[s]));
            int rc = p->prec == DFFT_DOUBLE ? execute_stage<double>(p, s) : execute_stage<float>(p, s);
            if (rc) return rc;
        }
        CU(ev_record(p, p->ev[4]));
        p->timed = true;
        return 0;
    }
    return p->prec == DFFT_DOUBLE ? execute_fused<double>(p) : execute_fused<float>(p);
}

extern "C" int dfft_synchronize(dfft_plan p)
{
    if (!p) return fail(DFFT_EINVAL, "null plan");
    if (p->dry) return 0;
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->stream));
    return 0;
}

extern "C" int dfft_get_timings(dfft_plan p, double t[5])
{
    if (!p || !t) return fail(DFFT_EINVAL, "bad arguments");
    if (!p->timed || p->dry) return fail(DFFT_EINVAL, "no execute to time yet");
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->stream));
    float ms[4] = {0, 0, 0, 0};
    if (p->xmode == DFFT_EXCHANGE_STAGED) {
        for (int s = 0; s < 4; s++) CU(cudaEventElapsedTime(&ms[s], p->ev[s], p->ev[s + 1]));
        if (p->direction == DFFT_BACKWARD) { std::swap(ms[0], ms[3]); std::swap(ms[1], ms[2]); }
        for (int s = 0; s < 4; s++) t[s] = ms[s];
    } else if (p->pipe) {
        // send side [start, last part issued] = t0 (+t1, + the sends); exposed exchange = from there until the last part has
        // arrived from every sender; t3 = the X pass of the last part (the earlier parts ran under t0)
        float a, b, c;
        CU(cudaEventElapsedTime(&a, p->ev[0], p->ev[1]));
        CU(cudaEventElapsedTime(&b, p->ev[1], p->evb[0]));
        CU(cudaEventElapsedTime(&c, p->evb[0], p->evb[1]));
        if (b < 0) { c += b; b = 0; }
        if (p->direction == DFFT_FORWARD) { t[0] = a; t[1] = 0; t[2] = b; t[3] = c; }
        else { t[3] = a; t[2] = b; t[1] = 0; t[0] = c; }   // backward: the send side is t3 (inverse X), the receive tail t0
    } else {
        float a, b, c;
        CU(cudaEventElapsedTime(&a, p->ev[0], p->ev[1]));
        CU(cudaEventElapsedTime(&b, p->ev[1], p->ev[2]));
        CU(cudaEventElapsedTime(&c, p->ev[2], p->ev[3]));
        if (p->direction == DFFT_FORWARD) { t[0] = a; t[1] = 0; t[2] = b; t[3] = c; }
        else { t[3] = a; t[2] = b; t[1] = 0; t[0] = c; }
    }
    t[4] = t[0] + t[1] + t[2] + t[3];
    return 0;
}

extern "C" int dfft_get_pass_timings(dfft_plan p, double t[3])
{
    if (!p || !t) return fail(DFFT_EINVAL, "bad arguments");
    if (!p->timed || p->dry) return fail(DFFT_EINVAL, "no execute to time yet");
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->stream));
    for (int a = 0; a < 3; a++) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, p->pev[a][0], p->pev[a][1]));
        t[a] = ms;
    }
    return 0;
}

extern "C" int dfft_execute_host_async(dfft_plan p, const void* host_in, void* host_out)
{
    if (!p || !host_in || !host_out || p->dry) return fail(DFFT_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    CU(cudaMemcpyAsync(p->buf1, host_in, (size_t)p->in_count * p->esz, cudaMemcpyHostToDevice, p->stream));
    int rc = dfft_execute(p);
    if (rc) return rc;
    CU(cudaMemcpyAsync(host_out, p->buf2, (size_t)p->out_count * p->esz, cudaMemcpyDeviceToHost, p->stream));
    return 0;
}

extern "C" int dfft_execute_host(dfft_plan p, const void* host_in, void* host_out)
{
    int rc = dfft_execute_host_async(p, host_in, host_out);
    if (rc) return rc;
    CU(cudaStreamSynchronize(p->stream));
    return 0;
}

extern "C" int dfft_plan_buffers(dfft_plan p, void** b1, void** b2)
{
    if (!p) return fail(DFFT_EINVAL, "null plan");
    if (b1) *b1 = p->buf1;
    if (b2) *b2 = p->buf2;
    return 0;
}
extern "C" int dfft_plan_counts(dfft_plan p, long long* ic, long long* oc, long long* mc)
{
    if (!p) return fail(DFFT_EINVAL, "null plan");
    if (ic) *ic = p->in_count;
    if (oc) *oc = p->out_count;
    if (mc) *mc = p->max_count;
    return 0;
}
/* test hook: JSON array of the passes the last dfft_execute of a DFFT_DRY_RUN plan recorded; returns the length needed */
extern "C" long long dfft_debug_plan_ops(dfft_plan p, char* buf, long long cap)
{
    if (!p) return -1;
    std::string o = "[";
    for (size_t i = 0; i < p->ops.size(); i++) { if (i) o += ", "; o += p->ops[i]; }
    o += "]";
    if (buf && cap > (long long)o.size()) memcpy(buf, o.c_str(), o.size() + 1);
    return (long long)o.size() + 1;
}

extern "C" int dfft_plan_launches(dfft_plan p) { return p ? p->launches : 0; }
extern "C" int dfft_plan_exchange(dfft_plan p) { return p ? p->xmode : 0; }
/* bit 0 / 1 / 2: the un-chunked Z / Y / X pass of this plan runs on the TMA-pipelined kernel (fft_tma.cuh) */
extern "C" int dfft_plan_tma_mask(dfft_plan p)
{
    if (!p || p->dry) return 0;
    const Geom& g = p->g;
    int m = 0;
    if (p->tz && (p->tz->use & (1u << TMA_Z)) && (p->n0l * g.n1) % p->tz->C == 0) m |= 1;
    if (p->ty && (p->ty->use & (1u << TMA_Y)) && g.n2 % p->ty->C == 0) m |= 2;
    if (p->tx && (p->tx->use & (1u << (p->direction == DFFT_FORWARD ? TMA_XF : TMA_XB))) && g.n2 % p->tx->C == 0) m |= 4;
    return m;
}
/* developer hook (DFFT_DEBUG_TIMELINE=1, single-kernel forward path): device-side timeline of the last execute, microseconds
 * relative to the kernel's start: [0] end of phase 0, [1] first X tile, [2] kernel end, [3..5] mean us per Z / Y / X tile,
 * [6..8] tile counts, [9] mean X-side wait per CTA, [10] max wait */
extern "C" int dfft_debug_timeline(dfft_plan p, double out[11])
{
    if (!p || !p->dbg || !out) return fail(DFFT_EINVAL, "no timeline recorded (set DFFT_DEBUG_TIMELINE=1 and use DFFT_OVERLAP_X)");
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->stream));
    unsigned long long h[16];
    CU(cudaMemcpy(h, p->dbg, sizeof(h), cudaMemcpyDeviceToHost));
    const double t0 = (double)h[0];
    out[0] = ((double)h[4] - t0) * 1e-3; out[1] = ((double)h[1] - t0) * 1e-3; out[2] = ((double)h[5] - t0) * 1e-3;
    for (int r = 0; r < 3; r++) { out[3 + r] = h[9 + r] ? (double)h[6 + r] / (double)h[9 + r] * 1e-3 : 0; out[6 + r] = (double)h[9 + r]; }
    const double ctas = (double)p->sms * 2;
    out[9] = (double)h[12] / ctas * 1e-3; out[10] = (double)h[13] * 1e-3;
    return 0;
}
extern "C" int dfft_plan_pipeline_parts(dfft_plan p) { return p && p->pipe ? p->parts : 0; }
/* 1: the parts run as a chain of two-role kernels on one stream (fft_fused_yx_kernel), 0: two streams / not pipelined */
extern "C" int dfft_plan_pipeline_chain(dfft_plan p) { return p && p->pipe && p->pipe_fyx ? 1 : 0; }
extern "C" int dfft_plan_fused(dfft_plan p) { return p && p->fuse && p->xmode != DFFT_EXCHANGE_STAGED ? (p->overlap ? 2 : 1) : 0; }
extern "C" void* dfft_plan_stream(dfft_plan p) { return p ? (void*)p->stream : nullptr; }

// ------------------------------------------------------------------------------------------------
// batched local transforms: plan / launch / delete, the templateFFT engine surface
// (3dmpifft_opt/include/templateFFT.h:361-365 initializeFFT / launchFFTKernel / deleteFFT)
// ------------------------------------------------------------------------------------------------
struct LinePass {
    const SizeEntry* e = nullptr;
    int kind = PK_Z;
    void* lut = nullptr;
    Affine ia{}, oa{};
    int G = 0, W = 0;
    long long ntiles = 0;
    long long tw_n = 0;          // four-step twiddle modulus (PK_XF_TW)
    int src = 0, dst = 0;        // 0 = the caller's data, 1 = the plan's temporary
};
struct dfft_lines_plan_s {
    int prec = 0, device = 0, sms = 148, npass = 0;
    bool ordered = false;        // passes run in the same order for both directions (four-step)
    void* temp = nullptr;
    LinePass pass[2];
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    bool timed = false;
};

template <typename T> static void upload_lut_e(void** dst, const SizeEntry* e, bool contiguous)
{
    if (contiguous) upload_lut<T>(dst, e->z_nstages, e->z_rad);
    else upload_lut<T>(dst, e->s_nstages, e->s_rad);
}

static int make_line_pass(LinePass& lp, int n, long long stride, long long nlines, long long inner, long long inner_dist, long long outer_dist,
                          int precision, bool dry = false)
{
    const SizeEntry* e = find_size_entry(n, precision);
    if (!e) return fail(DFFT_EUNSUPPORTED, "unsupported length %d", n);
    lp.e = e;
    if (stride == 1) {
        if (inner_dist != n || (inner != nlines && outer_dist != inner * n)) return fail(DFFT_EUNSUPPORTED, "contiguous lines must be densely packed");
        const int C = e->z_C;
        lp.G = (int)cdiv(nlines, C); lp.W = (int)std::min<long long>(nlines, 0x7fffffff); lp.ntiles = lp.G;
        lp.ia = Affine{0, (long long)C * n, n, 1};
        lp.oa = lp.ia;
        lp.kind = PK_Z;
    } else {
        if (inner_dist != 1 || inner < 1 || nlines % inner) return fail(DFFT_EUNSUPPORTED, "strided lines must be columns (inner_dist == 1)");
        const int C = e->s_C;
        lp.G = (int)cdiv(inner, C); lp.W = (int)inner; lp.ntiles = (nlines / inner) * lp.G;
        lp.ia = Affine{outer_dist, C, 1, stride};
        lp.oa = lp.ia;
        lp.kind = PK_Y;
    }
    if (dry) return 0;
    if (precision == DFFT_DOUBLE) upload_lut_e<double>(&lp.lut, e, stride == 1);
    else upload_lut_e<float>(&lp.lut, e, stride == 1);
    if (cudaGetLastError() != cudaSuccess || !lp.lut) return fail(DFFT_ECUDA, "twiddle table upload failed");
    return 0;
}

static int lines_plan_common(dfft_lines_plan p, int precision)
{
    p->prec = precision;
    CU(cudaGetDevice(&p->device));
    CU(cudaDeviceGetAttribute(&p->sms, cudaDevAttrMultiProcessorCount, p->device));
    CU(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    for (auto& e : p->ev) CU(cudaEventCreate(&e));
    return 0;
}

extern "C" int dfft_lines_destroy(dfft_lines_plan p)
{
    if (!p) return 0;
    cudaSetDevice(p->device);
    if (p->stream) cudaStreamSynchronize(p->stream);
    for (int i = 0; i < 2; i++) if (p->pass[i].lut) cudaFree(p->pass[i].lut);
    if (p->temp) cudaFree(p->temp);
    for (auto& e : p->ev) if (e) cudaEventDestroy(e);
    if (p->stream) cudaStreamDestroy(p->stream);
    cudaGetLastError();
    delete p;
    return 0;
}

// Long contiguous lines (beyond one shared-memory line): four-step decomposition n = n1 * n2 in two passes,
//   A: view the line as [n1][n2]; FFT along n1 (stride n2), multiply by W_n^(n2*k1), store transposed -> temp [n2][k1]
//   B: FFT along n2 (stride n1) of temp, stored to the caller's buffer at [k2][k1] = natural order X[k1 + n1*k2]
// -- what the reference does with its multi-upload axes and reorderFourStep = 1 (templateFFT.cpp:4007-4106, 5951).
// Validated against numpy on B200 (tests/test_gpu_parity.py::test_four_step_long_lines, profiles/r2_pytest_gpu_1xB200.log);
// DFFT_NO_LONG_LINES=1 restores the "unsupported length" answer.
static int make_four_step(dfft_lines_plan p, int n, long long nlines, int precision, bool dry = false)
{
    long long best1 = 0;
    int best_score = -1;
    for (long long d = 2; d * d <= (long long)n * 4 && d < n; d++) {
        if (n % d) continue;
        const SizeEntry *e1 = find_size_entry((int)d, precision), *e2 = find_size_entry((int)(n / d), precision);
        if (!e1 || !e2) continue;
        const long long q = n / d;
        const double ratio = d > q ? (double)d / q : (double)q / d;
        int score = (e1->gen ? 0 : 1000) + (e2->gen ? 0 : 1000) + (int)(500.0 / ratio);
        if (score > best_score) { best_score = score; best1 = d; }
    }
    if (!best1) return fail(DFFT_EUNSUPPORTED, "length %d cannot be split into two supported factors", n);
    const int n1 = (int)best1, n2 = n / n1;
    const size_t esz = precision == DFFT_FLOAT ? 8 : 16;
    if (dry) p->temp = fake_addr(0, 4);
    else CU(cudaMalloc(&p->temp, (size_t)nlines * n * esz));
    // pass A: columns of the [n1][n2] matrix of every line, transposed store + twiddle
    LinePass& a = p->pass[0];
    a.e = find_size_entry(n1, precision);
    {
        const int C = a.e->x_C;
        a.G = (int)cdiv(n2, C); a.W = n2; a.ntiles = nlines * a.G;
        a.ia = Affine{(long long)n, C, 1, n2};
        a.oa = Affine{(long long)n, (long long)C * n1, n1, 1};
        a.kind = PK_XF_TW; a.tw_n = n; a.src = 0; a.dst = 1;
        if (dry) {}
        else if (precision == DFFT_DOUBLE) upload_lut<double>(&a.lut, a.e->x_nstages, a.e->x_rad);
        else upload_lut<float>(&a.lut, a.e->x_nstages, a.e->x_rad);
    }
    // pass B: columns of the [n2][n1] matrix in temp, natural-order result in the caller's buffer
    LinePass& b = p->pass[1];
    b.e = find_size_entry(n2, precision);
    {
        const int C = b.e->s_C;
        b.G = (int)cdiv(n1, C); b.W = n1; b.ntiles = nlines * b.G;
        b.ia = Affine{(long long)n, C, 1, n1};
        b.oa = b.ia;
        b.kind = PK_Y; b.src = 1; b.dst = 0;
        if (dry) {}
        else if (precision == DFFT_DOUBLE) upload_lut<double>(&b.lut, b.e->s_nstages, b.e->s_rad);
        else upload_lut<float>(&b.lut, b.e->s_nstages, b.e->s_rad);
    }
    if (!dry && (cudaGetLastError() != cudaSuccess || !a.lut || !b.lut)) return fail(DFFT_ECUDA, "twiddle table upload failed");
    p->npass = 2;
    p->ordered = true;
    return 0;
}

extern "C" int dfft_lines_plan_create(int n, long long stride, long long nlines, long long inner, long long inner_dist, long long outer_dist,
                                      int precision, dfft_lines_plan* out)
{
    if (!out) return fail(DFFT_EINVAL, "null plan pointer");
    *out = nullptr;
    if (n < 1 || nlines < 0 || stride < 1 || (precision != DFFT_DOUBLE && precision != DFFT_FLOAT)) return fail(DFFT_EINVAL, "bad arguments");
    dfft_lines_plan p = new dfft_lines_plan_s;
    int rc = lines_plan_common(p, precision);
    const char* nolong = getenv("DFFT_NO_LONG_LINES");
    if (!rc && !find_size_entry(n, precision) && stride == 1 && inner_dist == n && !(nolong && atoi(nolong) != 0)) {
        rc = make_four_step(p, n, nlines, precision);
    } else {
        if (!rc) rc = make_line_pass(p->pass[0], n, stride, nlines, inner, inner_dist, outer_dist, precision);
        p->npass = 1;
    }
    if (rc) { dfft_lines_destroy(p); return rc; }
    *out = p;
    return 0;
}

/* batch of 2-D transforms, nx fastest: the reference's FFTdim = 2 application (Test_2D.cpp: size = {X, Y, Z}) */
extern "C" int dfft_lines_plan_create_2d(int nx, int ny, long long batch, int precision, dfft_lines_plan* out)
{
    if (!out) return fail(DFFT_EINVAL, "null plan pointer");
    *out = nullptr;
    if (nx < 1 || ny < 1 || batch < 0 || (precision != DFFT_DOUBLE && precision != DFFT_FLOAT)) return fail(DFFT_EINVAL, "bad arguments");
    dfft_lines_plan p = new dfft_lines_plan_s;
    int rc = lines_plan_common(p, precision);
    if (!rc) rc = make_line_pass(p->pass[0], nx, 1, (long long)ny * batch, (long long)ny * batch, nx, 0, precision);
    if (!rc) rc = make_line_pass(p->pass[1], ny, nx, (long long)nx * batch, nx, 1, (long long)nx * ny, precision);
    if (rc) { dfft_lines_destroy(p); return rc; }
    p->npass = 2;
    *out = p;
    return 0;
}

template <typename T> static int lines_execute_impl(dfft_lines_plan p, void* data, int direction)
{
    CU(cudaEventRecord(p->ev[0], p->stream));
    for (int k = 0; k < p->npass; k++) {
        const LinePass& lp = p->pass[(direction == DFFT_BACKWARD && !p->ordered) ? p->npass - 1 - k : k];
        if (lp.ntiles <= 0) continue;
        TileArgs<T> a{};
        a.in = (const cx<T>*)(lp.src ? p->temp : data); a.out = (cx<T>*)(lp.dst ? p->temp : data); a.lut = (const cx<T>*)lp.lut;
        a.ia = lp.ia; a.oa = lp.oa; a.G = lp.G; a.W = lp.W; a.ntiles = lp.ntiles;
        a.inv = direction == DFFT_BACKWARD; a.gen = lp.e->gen; a.tw_n = lp.tw_n;
        cudaError_t err = lp.e->launch[lp.kind](&a, p->sms, p->stream);
        if (err != cudaSuccess) return fail(DFFT_ECUDA, "line pass launch failed: %s", cudaGetErrorString(err));
    }
    CU(cudaEventRecord(p->ev[1], p->stream));
    p->timed = true;
    return 0;
}

extern "C" int dfft_lines_execute(dfft_lines_plan p, void* data, int direction)
{
    if (!p || !data || (direction != DFFT_FORWARD && direction != DFFT_BACKWARD)) return fail(DFFT_EINVAL, "bad arguments");
    CU(cudaSetDevice(p->device));
    return p->prec == DFFT_DOUBLE ? lines_execute_impl<double>(p, data, direction) : lines_execute_impl<float>(p, data, direction);
}

extern "C" int dfft_lines_synchronize(dfft_lines_plan p)
{
    if (!p) return fail(DFFT_EINVAL, "null plan");
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->stream));
    return 0;
}

extern "C" void* dfft_lines_stream(dfft_lines_plan p) { return p ? (void*)p->stream : nullptr; }

/* test hook (host only): the passes a lines plan would launch for `direction`, as JSON (same format as dfft_debug_plan_ops;
 * the caller's data is buffer 1 of device 0, the plan's temporary buffer 4); two_d != 0: 2-D plan (n = nx, stride = ny,
 * nlines = batch).  Long lines always use the four-step plan here.  Returns the bytes needed, < 0 on error. */
extern "C" long long dfft_debug_lines_ops(int n, long long stride, long long nlines, long long inner, long long inner_dist, long long outer_dist,
                                          int precision, int direction, int two_d, char* buf, long long cap)
{
    dfft_lines_plan_s lp;
    dfft_plan_s rec;   // only its `ops` vector is used
    rec.dry = true;
    lp.prec = precision;
    int rc = 0;
    if (two_d) {
        const int nx = n, ny = (int)stride;
        const long long batch = nlines;
        rc = make_line_pass(lp.pass[0], nx, 1, (long long)ny * batch, (long long)ny * batch, nx, 0, precision, true);
        if (!rc) rc = make_line_pass(lp.pass[1], ny, nx, (long long)nx * batch, nx, 1, (long long)nx * ny, precision, true);
        lp.npass = 2;
    } else if (!find_size_entry(n, precision) && stride == 1 && inner_dist == n) {
        rc = make_four_step(&lp, n, nlines, precision, true);
    } else {
        rc = make_line_pass(lp.pass[0], n, stride, nlines, inner, inner_dist, outer_dist, precision, true);
        lp.npass = 1;
    }
    if (rc) return rc;
    static const char* names[PK_COUNT] = {"Z", "Y", "Y_CO", "Y_CI", "XF", "XB", "XB_CO", "XF_TW"};
    for (int k = 0; k < lp.npass; k++) {
        const LinePass& ps = lp.pass[(direction == DFFT_BACKWARD && !lp.ordered) ? lp.npass - 1 - k : k];
        TileArgs<double> a{};
        a.in = (const double2*)(ps.src ? lp.temp : fake_addr(0, 1)); a.out = (double2*)(ps.dst ? lp.temp : fake_addr(0, 1));
        a.ia = ps.ia; a.oa = ps.oa; a.G = ps.G; a.W = ps.W; a.ntiles = ps.ntiles;
        a.inv = direction == DFFT_BACKWARD; a.tw_n = ps.tw_n;
        const int C = ps.kind == PK_Z ? ps.e->z_C : (ps.kind == PK_Y ? ps.e->s_C : ps.e->x_C);
        record_op<double>(&rec, names[ps.kind], k, ps.e->N, C, false, false, ps.kind == PK_XF_TW, a);
    }
    lp.temp = nullptr;
    std::string o = "[";
    for (size_t i = 0; i < rec.ops.size(); i++) { if (i) o += ", "; o += rec.ops[i]; }
    o += "]";
    if (buf && cap > (long long)o.size()) memcpy(buf, o.c_str(), o.size() + 1);
    return (long long)o.size() + 1;
}

extern "C" int dfft_fft_lines(void* data, int n, long long stride, long long nlines, long long inner, long long inner_dist,
                              long long outer_dist, int direction, int precision)
{
    if (!data || n < 1 || nlines < 0 || stride < 1) return fail(DFFT_EINVAL, "bad arguments");
    if (direction != DFFT_FORWARD && direction != DFFT_BACKWARD) return fail(DFFT_EINVAL, "direction must be +1 or -1");
    if (nlines == 0) return 0;
    dfft_lines_plan p = nullptr;
    int rc = dfft_lines_plan_create(n, stride, nlines, inner, inner_dist, outer_dist, precision, &p);
    if (rc) return rc;
    rc = dfft_lines_execute(p, data, direction);
    if (!rc) rc = dfft_lines_synchronize(p);
    dfft_lines_destroy(p);
    return rc;
}
