/*
 * dfft.h -- C ABI of the B200-native slab-decomposed 3-D complex-to-complex FFT (libdfft.so).
 *
 * This is the drop-in boundary for the hot path of lueelu/DistributedFFT's `3dmpifft_opt`:
 * every entry point below names the reference interface it replaces (paths relative to the
 * reference tree).  Plain pointers and sizes only; all functions return 0 on success and a
 * negative DFFT_E* code on failure (dfft_last_error() gives the message).  The reference aborts
 * with exit(EXIT_FAILURE) on every error (3dmpifft_opt/include/fft_mpi_common.h:31-102); the C++
 * shim include/fft_mpi_3d_api.h keeps that behaviour on top of this ABI.
 *
 * Data model (identical to the reference, SURVEY.md Appendix A):
 *   global array A[x][y][z], z fastest, N0 = X slowest; P devices; device p owns the x-slab
 *   [p*xd, p*xd + n0_l), xd = ceil(N0/P), the last device the remainder.
 *   forward : in = natural x-slab [x_l][y][z]  ->  out = y-slab, TRANSPOSED [y_l][z][x] (x fastest)
 *   backward: in = [y_l][z][x]                 ->  out = natural [x_l][y][z], unnormalised.
 *   complex = interleaved (re, im) doubles (precision 0) or floats (precision 1).
 *
 * Threading: a plan belongs to one device; one host thread per device may create/execute plans
 * concurrently (the reference's `#pragma omp parallel for num_threads(devices)` loop,
 * 3dmpifft_opt/fftSpeed3d_c2c.cpp:49), or one process per device (torchrun) with a bootstrap
 * callback.  Collective calls (plan creation with P > 1, execute with P > 1, destroy) must be made
 * by all P participants.
 */
#ifndef DFFT_H
#define DFFT_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DFFT_FORWARD 1      /* fft_mpi_common.h:18 FORWARD  */
#define DFFT_BACKWARD (-1)  /* fft_mpi_common.h:19 BACKWARD */
#define DFFT_ALLOC_CPU 1    /* fft_mpi_common.h:15 ALLOC_CPU (pinned host memory here) */
#define DFFT_ALLOC_DEV (-1) /* fft_mpi_common.h:16 ALLOC_DEV */

#define DFFT_DOUBLE 0
#define DFFT_FLOAT 1

/* plan flags */
#define DFFT_EXCHANGE_AUTO 0u    /* P2P when every peer is reachable, else NCCL */
#define DFFT_EXCHANGE_P2P 1u     /* t1+t2 fused: the Y pass stores straight into the peers' receive buffers over NVLink */
#define DFFT_EXCHANGE_NCCL 2u    /* Y pass packs locally, grouped ncclSend/ncclRecv (ncclAlltoAll when the library has it) */
#define DFFT_EXCHANGE_STAGED 3u  /* reference-like: separate pack kernel + peer copies, device sync after every stage */
#define DFFT_EXCHANGE_MASK 3u
#define DFFT_SCALE_BACKWARD 4u   /* divide by N0*N1*N2 in the last backward pass (the `roc` variant's scale_element,
                                    3dmpifft_roc/include/fft_mpi_3d_api.cpp:208-210); default off like 3dmpifft_opt */

#define DFFT_NO_FUSE 8u          /* t0 as two HBM sweeps (Z pass, Y pass) */
#define DFFT_FORCE_FUSE 16u      /* t0 as ONE persistent kernel whose Z->Y intermediate stays in L2 (square planes only).
                                    Default: fused when the exchange is P2P (the Y stores are NVLink-bound and hide the
                                    Z role), two sweeps otherwise */

#define DFFT_NATURAL_SPECTRUM 64u /* single device: the spectrum (forward output / backward input) is kept in natural
                                    [x][y][z] order instead of the reference's transposed [y][z][x] (SURVEY 8f rank 1) */
#define DFFT_DRY_RUN 128u         /* describe-only plan (tests): no CUDA call, `in`/`out` are symbolic addresses, dfft_execute records
                                    the passes it would launch; read them with dfft_debug_plan_ops.  `comm` may be NULL */
#define DFFT_OVERLAP_X 32u       /* EXPERIMENTAL (forward, P2P, square planes): the whole transform of a device as one kernel;
                                    the z axis is sent in parts and the X lines of a part start as soon as it has arrived
                                    from every sender, overlapping t3 with the NVLink-bound sends (env DFFT_OVERLAP=1) */

#define DFFT_NO_PIPELINE 256u     /* P > 1: do NOT cut the z axis into parts.  Pipelined plans overlap t2 / t3 with t0 -- the reference has no
                                    overlap at all (fft_mpi_3d_api.cpp:610-672).  Two schedules exist: a CHAIN of two-role kernels on
                                    the plan stream, [Z + Y part 0] [Y part 1 + X part 0] ... [X last part] (forward, cubes, P2P
                                    exchange), and a TWO-STREAM schedule (send side / receive side, any direction, P2P or NCCL).
                                    Default (measured, DESIGN.md 5.1): the chain, from 4 devices on, for axes >= 1024 points.
                                    env DFFT_PIPELINE=0 / 1 overrides, DFFT_PARTS=k picks the number of parts,
                                    DFFT_PIPE_MODE=streams prefers the two-stream schedule */
#define DFFT_FORCE_PIPELINE 1024u /* pipelined plan wherever one is possible (also 2 devices, short axes, backward, NCCL with equal chunks) */

#define DFFT_NO_TMA 512u          /* use the register-staged pass kernels everywhere.  Default: passes whose load and store are both
                                    local and un-chunked (Z, natural Y, X) run on the TMA-pipelined kernels (fft_tma.cuh: 3-slot
                                    shared-memory ring fed and drained by cp.async.bulk / cp.async.bulk.tensor) for the lengths
                                    that have an instantiation; env DFFT_TMA=0 has the same effect */

#define DFFT_EINVAL (-1)
#define DFFT_ECUDA (-2)
#define DFFT_EUNSUPPORTED (-3)
#define DFFT_ECOMM (-4)
#define DFFT_ENOMEM (-5)

typedef struct dfft_plan_s* dfft_plan;
typedef struct dfft_comm_s* dfft_comm;

/* Bootstrap all-gather supplied by the host program in process-per-GPU mode: every rank
 * contributes `bytes` bytes from `send`; on return `recv` holds nranks*bytes in rank order.
 * Plays the role MPI_Comm plays in the reference (fft_mpi_3d_api.h:68,70). */
typedef int (*dfft_allgather_fn)(void* ctx, const void* send, void* recv, size_t bytes);

/* -- library ------------------------------------------------------------------------------- */
const char* dfft_last_error(void);
int dfft_version(void);
/* 2: `n` has a tuned kernel; 1: handled by the run-time-scheduled kernel (any length whose prime factors are
 * in {2,3,5,7,11,13} -- the set templateFFT accepts, templateFFT.cpp:3956-3964 -- up to 6400 points in double and
 * 12800 in float, i.e. while two copies of a line fit in shared memory); 0: unsupported (other primes, or longer:
 * the reference switches to multi-upload passes there, templateFFT.cpp:4007-4106, which this library does not have) */
int dfft_length_kind(int n, int precision);
/* test hook (host only): the multi-role kernels the table entry of length n has -- bit k: fused t0 kind k (0 Z+Y, 1 Z+Y with
 * the chunked store, 2 Y+Z, 3 Y+Z with the chunked load), bit 4: the kernel-chain link, bit 5: the single-kernel forward.  A
 * kind whose roles need more shared memory than one CTA may have is absent; -1: unsupported length */
int dfft_debug_fused_kinds(int n, int precision);
/* radix schedule used for length n (stage order as executed); returns the number of stages, 0 if unsupported */
int dfft_length_schedule(int n, int precision, int* radices, int max_radices);
/* test hook (host only): ticket order of the single-kernel forward path (fft_fused3_kernel); out = role (0 Z, 1 Y, 2 X),
 * part, plane, tile; returns the number of tickets (ticket < 0: only that) */
long long dfft_debug_fused3_order(long long planes, long long rows, int GA, int GBk, int GXk, int K, int lag, long long ticket,
                                  long long out[4]);
/* test hook: JSON description of the passes recorded by the last dfft_execute of a DFFT_DRY_RUN plan (affine maps, chunk
 * tables, symbolic buffer addresses: device d, buffer b at ((d+1) << 44) | (b << 40), b = 1 bufferDev1, 2 out, 3 receive/work,
 * 4 intermediate, 5 in).  Returns the number of bytes needed (including the terminator). */
long long dfft_debug_plan_ops(dfft_plan plan, char* buf, long long cap);
/* test hook (host only): the passes a lines plan (1-D, 2-D when two_d != 0: n = nx, stride = ny, nlines = batch, or the
 * four-step plan of a long line) would launch, same JSON as dfft_debug_plan_ops: data = buffer 1, temporary = buffer 4 */
long long dfft_debug_lines_ops(int n, long long stride, long long nlines, long long inner, long long inner_dist, long long outer_dist,
                               int precision, int direction, int two_d, char* buf, long long cap);
/* number of TUNED transform lengths for a precision; fills `lengths` (may be NULL) */
int dfft_supported_lengths(int precision, int* lengths, int max_lengths);

/* -- slab bookkeeping ---------------------------------------------------------------------- */
/* fft_mpi_init, fft_mpi_3d_api.cpp:3-39 (+ getProperDeviceNum :232-272, getDataCountForNode :274-287):
 * shrink `wanted_devices` (clamped to the visible device count unless that is 0) so that ceil-blocks
 * of N[0] leave no device empty, return per-device input element counts, enable peer access
 * between the devices used.  `counts` must have room for `wanted_devices` entries. */
int dfft_init(const long long N[3], int wanted_devices, int* total_devices, int* local_devices, long long* counts);
/* getMaxDataCount, fft_mpi_3d_api.cpp:289-316: elements each of in/out must hold on a device */
long long dfft_max_data_count(long long n0, long long n1, long long n2, int total_devices, int is_last_device);
/* fft_mpi_local_size_3d (declared fft_mpi_3d_api.h:73, never defined in the reference): returns the
 * allocation count and the slab owned by `dev_idx` before (x) and after (y) the exchange */
long long dfft_local_size_3d(long long n0, long long n1, long long n2, int total_devices, int dev_idx,
                             long long* local_n0, long long* local_0_start, long long* local_n1,
                             long long* local_1_start);
/* fft_mpi_alloc_local_memory, fft_mpi_3d_api.cpp:216-230 (64-bit count; ALLOC_CPU is pinned) */
void* dfft_alloc_local(long long count, int flag, int precision);
int dfft_free_local(void* ptr, int flag);

/* -- communicator -------------------------------------------------------------------------- */
/* P device-threads inside one process (the reference's multi-GPU-per-rank mode). Returns one shared
 * handle; every participating thread passes it to dfft_plan_c2c_3d with its own dev_idx. */
int dfft_comm_create_local(int nranks, dfft_comm* comm);
/* One process per GPU; `allgather` is used during plan creation / teardown only. */
int dfft_comm_create_bootstrap(int rank, int nranks, dfft_allgather_fn allgather, void* ctx, dfft_comm* comm);
int dfft_comm_destroy(dfft_comm comm);
/* host-side all-gather through a communicator (what plan creation uses to swap IPC handles / the NCCL id) */
int dfft_comm_allgather(dfft_comm comm, int rank, const void* send, void* recv, size_t bytes);
/* the reference's TransInfo exchange table of one device (fft_mpi_common.h:24-29, fft_mpi_3d_api.cpp:84-133):
 * element counts and offsets of the chunk sent to / received from every device i */
int dfft_exchange_table(long long n0, long long n1, long long n2, int total_devices, int dev_idx, int direction,
                        long long* scount, long long* soffset, long long* rcount, long long* roffset);

/* -- plan / execute ------------------------------------------------------------------------ */
/* fft_mpi_plan_dft_c2c_3d, fft_mpi_3d_api.cpp:41-141.  Same ownership rules: `in`/`out` are the
 * caller's device buffers of dfft_max_data_count() elements; out == NULL or out == in means in
 * place; the plan owns bufferDev1 and copies `in` into it at creation (api.cpp:76-77); bufferDev2
 * aliases `out`.  Execute never re-reads `in`: refill bufferDev1 (dfft_plan_buffers) to transform new
 * data, exactly like the reference driver does (fftSpeed3d_c2c.cpp:78).
 * `comm` may be NULL when total_devices == 1.  `dev_idx` is this device's global index (= rank).
 * The CUDA device current at the call is the plan's device. */
int dfft_plan_c2c_3d(long long n0, long long n1, long long n2, void* in, void* out, dfft_comm comm, int dev_idx,
                     int total_devices, int direction, int precision, unsigned flags, dfft_plan* plan);
/* fft_mpi_execute_dft_3d_c2c, fft_mpi_3d_api.cpp:181-214.  Asynchronous on the plan's stream;
 * dfft_synchronize() or dfft_get_timings() waits.  Result in bufferDev2 (= out). */
int dfft_execute(dfft_plan plan);
int dfft_synchronize(dfft_plan plan);
/* One reference stage at a time (0: t0 fftZY, 1: t1 pack, 2: t2 all-to-all, 3: t3 fftX, in the
 * order the plan's direction executes them), leaving bufferDev1/bufferDev2 exactly as the reference
 * leaves them after that stage.  Requires a plan created with DFFT_EXCHANGE_STAGED.  Synchronous. */
int dfft_execute_stage(dfft_plan plan, int stage);
/* Host-buffer entry: copies `host_in` (input-slab elements) to bufferDev1, executes, copies the
 * result slab to `host_out`; copies are on the plan's stream (pinned buffers overlap). Synchronous. */
int dfft_execute_host(dfft_plan plan, const void* host_in, void* host_out);
/* Same, but returns once the three operations are enqueued on the plan's stream (dfft_synchronize waits).
 * Two plans driven alternately keep PCIe busy in both directions: plan A's D2H overlaps plan B's H2D. */
int dfft_execute_host_async(dfft_plan plan, const void* host_in, void* host_out);
/* milliseconds of the last execute: t[0..3] = t0,t1,t2,t3 as the reference prints them
 * (api.cpp:201; fused stages report 0 for t1 and the *exposed* wait for t2), t[4] = total. */
int dfft_get_timings(dfft_plan plan, double t_ms[5]);
/* milliseconds of the Z, Y and X pass kernels of the last execute (CUDA events around each launch) */
int dfft_get_pass_timings(dfft_plan plan, double t_ms[3]);
/* bufferDev1 / bufferDev2 of the plan (fft_mpi_3d_api.h:24; the driver writes into bufferDev1) */
int dfft_plan_buffers(dfft_plan plan, void** buffer1, void** buffer2);
/* element counts of this device's input slab and output slab */
int dfft_plan_counts(dfft_plan plan, long long* in_count, long long* out_count, long long* max_count);
/* kernels launched by the last execute (for bench.py's gpu_launches) */
int dfft_plan_launches(dfft_plan plan);
/* 2: forward transform runs as the single overlapped kernel (DFFT_OVERLAP_X); 1: t0 runs as the fused two-pass
 * kernel (square planes, N1 == N2); 0: separate passes */
int dfft_plan_fused(dfft_plan plan);
/* bit 0 / 1 / 2 set: the plan's un-chunked Z / Y / X pass runs on the TMA-pipelined kernel (fft_tma.cuh) */
int dfft_plan_tma_mask(dfft_plan plan);
/* developer hook: device-side timeline of the last execute of a DFFT_OVERLAP_X plan created under DFFT_DEBUG_TIMELINE=1 (microseconds
 * from kernel start: end of phase 0, first X tile, kernel end; mean us per Z / Y / X tile; tile counts; mean / max arrival wait) */
int dfft_debug_timeline(dfft_plan plan, double out[11]);
/* number of z-parts of the stream-pipelined forward / backward path, 0 when the plan does not use it */
int dfft_plan_pipeline_parts(dfft_plan plan);
/* 1: the z-parts of a pipelined forward plan run as a chain of two-role kernels on one stream (Y pass of part k + X pass of
 * part k-1 in one kernel: cubes with the P2P exchange), 0: as two streams, or not pipelined */
int dfft_plan_pipeline_chain(dfft_plan plan);
/* which exchange the plan resolved to (DFFT_EXCHANGE_*) */
int dfft_plan_exchange(dfft_plan plan);
/* the stream the plan launches on (a cudaStream_t), so callers can time with events on it */
void* dfft_plan_stream(dfft_plan plan);
/* fft_mpi_destroy_plan, fft_mpi_3d_api.cpp:143-179 (collective when P > 1) */
int dfft_destroy(dfft_plan plan);
/* fft_mpi_cleanup (declared fft_mpi_3d_api.h:69, never defined in the reference) */
int dfft_cleanup(void);

/* convenience for hosts without a CUDA runtime binding (tests): synchronous cudaMemcpy,
 * kind 1 = host->device, 2 = device->host, 0 = default (UVA) */
int dfft_memcpy(void* dst, const void* src, size_t bytes, int kind);

/* -- batched local transforms: the templateFFT engine surface (3dmpifft_opt/include/templateFFT.h:361-365) -----
 *    initializeFFT(app, config)   -> dfft_lines_plan_create / dfft_lines_plan_create_2d
 *    launchFFTKernel(app, inverse)-> dfft_lines_execute (asynchronous on the plan's stream, in place)
 *    deleteFFT(app)               -> dfft_lines_destroy
 *    Line l starts at data + (l / inner) * outer_dist + (l % inner) * inner_dist (in elements), points are
 *    `stride` elements apart.  Supported shapes: stride == 1 with densely packed lines (inner_dist == n), or
 *    stride > 1 with inner_dist == 1 (columns of row-major matrices: `inner` columns per matrix, matrices
 *    `outer_dist` apart).  The 2-D plan transforms `batch` row-major ny x nx matrices (nx fastest), the
 *    reference's FFTdim = 2 application (templateFFT/batchTest/Test_2D.cpp). */
typedef struct dfft_lines_plan_s* dfft_lines_plan;
int dfft_lines_plan_create(int n, long long stride, long long nlines, long long inner, long long inner_dist,
                           long long outer_dist, int precision, dfft_lines_plan* plan);
int dfft_lines_plan_create_2d(int nx, int ny, long long batch, int precision, dfft_lines_plan* plan);
int dfft_lines_execute(dfft_lines_plan plan, void* data, int direction);
int dfft_lines_synchronize(dfft_lines_plan plan);
void* dfft_lines_stream(dfft_lines_plan plan);
int dfft_lines_destroy(dfft_lines_plan plan);
/* one-shot convenience (plan + execute + synchronize + destroy), used by the per-axis parity tests */
int dfft_fft_lines(void* data, int n, long long stride, long long nlines, long long inner, long long inner_dist,
                   long long outer_dist, int direction, int precision);

#ifdef __cplusplus
}
#endif
#endif /* DFFT_H */
