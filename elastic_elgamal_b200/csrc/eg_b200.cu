// eg_b200.cu -- the C ABI (include/eg_b200.h) and kernel launches of the B200 batch engine.
//
// Host side: context / scratch management, per-election transcript prefixes (computed once with the same
// __host__ __device__ Merlin code the kernels use), slot tables that describe which equation of which
// proof each thread evaluates, chunked execution.  All group / field / hash arithmetic of a batch runs in
// the kernels below; there is no CPU path (eg_ctx_create fails without a device).
#ifdef EG_HOSTSIM
#include "hostsim_cuda.h"      // test-only stand-in for the CUDA runtime (tests/hostsim): malloc/memcpy, no device
// Kernels in the test harness: launch() runs a __global__ function once per (block, thread), one after the other, with the
// built-in indices set first.  The pretend device has one SM that holds one CTA of any kernel, so a persistent grid is a
// single CTA.
#define __global__
#define __launch_bounds__(...)
struct dim3 {
    unsigned x, y, z;
    dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
static thread_local dim3 blockIdx, threadIdx, blockDim, gridDim;
template <class K, class... A> static void hs_launch(K kernel, dim3 grid, dim3 block, const A &...args) {
    gridDim = grid; blockDim = block;
    for (unsigned b = 0; b < grid.x * grid.y * grid.z; b++) {
        blockIdx = dim3(b % grid.x, b / grid.x % grid.y, b / (grid.x * grid.y));
        for (unsigned t = 0; t < block.x * block.y * block.z; t++) {
            threadIdx = dim3(t % block.x, t / block.x % block.y, t / (block.x * block.y));
            kernel(args...);
        }
    }
}
enum cudaDeviceAttr { cudaDevAttrMultiProcessorCount = 16 };
static cudaError_t cudaDeviceGetAttribute(int *v, cudaDeviceAttr, int) { *v = 1; return cudaSuccess; }
template <class K> static cudaError_t cudaOccupancyMaxActiveBlocksPerMultiprocessor(int *n, K, int, size_t) { *n = 1; return cudaSuccess; }
#else
#include <cuda_runtime.h>
#endif

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <new>
#include <string>
#include <vector>

#include "../../include/eg_b200.h"
#include "kernels.cuh"
#include "weighted_sum.cuh"
#include "group_sum.cuh"

using namespace eg;

#include "device_kernels.inc"

// =================================================================== context

#define EG_STAT_KINDS 4          // timed kernel kinds (eg_last_kernel_stats): 0 = k_commit, 1 = k_ring, 2 = k_msm, 3 = k_ring_pair

struct dev_buf {
    void *p = nullptr;
    size_t cap = 0;
};

struct eg_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool has_receiver = false, has_blinding_base = false;
    uint8_t key[32];
    uint8_t blinding_base[32];
    uint32_t *d_table_g = nullptr, *d_table_k = nullptr, *d_table_h = nullptr, *d_status = nullptr;
    std::string err;
    uint64_t launches = 0;
    float timings[5] = {0, 0, 0, 0, 0};
    cudaEvent_t ev[8];
    std::vector<cudaEvent_t> commit_ev;     // pairs (start, stop) around every k_commit / k_ring launch of the current call
    std::vector<uint8_t> commit_ev_kind;    // per pair: 0 = k_commit, 1 = k_ring, 2 = k_msm, 3 = k_ring_pair
    size_t commit_ev_used = 0;
    uint64_t kind_tasks[EG_STAT_KINDS] = {0, 0, 0, 0}, kind_launches[EG_STAT_KINDS] = {0, 0, 0, 0};   // per kind, current call
    float kind_ms[EG_STAT_KINDS] = {0, 0, 0, 0};
    // grow-only scratch
    cudaStream_t copy_stream = nullptr;     // host -> device prefetch of the next chunk
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr};
    cudaEvent_t ev_pipe[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // pipeline_chunks: in / done / out per buffer set
    dev_buf pp[2][5];                       // double-buffered inputs / outputs of the pipelined provers
    dev_buf in2[3];
    dev_buf pts, enc, commit, chal, flags, res[3], in[4], verdicts, partial, running, adm, misc, slots, consts, res_big, term;
    terminal_params term_plan;   // deferred encodings of the slot table uploaded last (upload_slots); n_pts == 0: none
    size_t adm_used = 0;      // cached points in `adm` (32 words each); entries 0,1 = the [O, G] pair
    std::map<std::string, std::vector<uint64_t>> adm_cache_key;
    size_t chunk_items = 0;   // 0 = default
    int ring_mode = 0;        // 2: k_ring (one thread per ring, chunked tables); 1: k_commit / k_ring_hash launches per equation;
                              // 0: chosen per chunk (1 when the chunk cannot fill the persistent k_ring grid, run_ring_job)
    int prover_ct = 0;        // eg_ctx_set_prover_mode: constant-time fixed-base arithmetic for the provers' secret scalars
    std::map<const void *, int> resident;   // resident CTAs of each persistent-grid kernel (resident_ctas)
    dev_buf ring_scratch;
    // per-call narrow fixed-base tables of the participant keys of a key set (api_sharing.inc), cached by key bytes
    dev_buf xtab;
    uint8_t xtab_key[8][32];
    bool xtab_valid[8] = {false, false, false, false, false, false, false, false};
    size_t key_table_min = 32768;   // eg_ctx_set_key_table_min
    // multi-GPU (comm.inc): NCCL communicator of a per-rank context (eg_ctx_attach_comm) or of a child of a multi-device
    // context (eg_ctx_create_multi); `children` is non-empty only for the latter's parent, which owns no device state
    void *comm = nullptr;
    int rank = 0, world = 1;
    dev_buf gather;
    std::vector<eg_ctx *> children;
    eg_ctx *parent = nullptr;
    std::vector<uint8_t> host_tally;        // child of a multi context: its partial tally, host copy
    uint32_t comm_bad = 0;                  // host copy of the combine kernel's flag (comm_combine / comm_check)
    bool comm_pending = false;
    dev_buf ws[13];                         // scratch of eg_ciphertexts_weighted_sum and _group_sum (api_weighted_sum.inc,
                                            // api_group_sum.inc)
};

struct eg_dlog_table {
    eg_ctx *ctx;
    uint64_t lo, hi;      // the whole range [lo, hi)
    uint64_t m;           // baby steps: the device table holds [lo, lo + min(m, hi - lo))
    uint64_t giants;      // ceil((hi - lo) / m); 1: a range table, no giant-step walk
    uint32_t step[24];    // giants > 1: -[m/2]G in affine Niels form (dlog_walk_params::step)
    size_t cap;
    uint32_t *d_keys;     // cap * 8 words
    uint64_t *d_vals;     // cap
    std::vector<eg_dlog_table *> children;   // table of a multi-device context: one replica per device
};

static eg_status fail(eg_ctx *ctx, eg_status st, const char *what, cudaError_t ce = cudaSuccess) {
    if (ctx) {
        ctx->err = what;
        if (ce != cudaSuccess) { ctx->err += ": "; ctx->err += cudaGetErrorString(ce); }
    }
    return st;
}

#define CU(call)                                                            \
    do {                                                                    \
        cudaError_t ce_ = (call);                                           \
        if (ce_ != cudaSuccess) return fail(ctx, EG_ERR_CUDA, #call, ce_);  \
    } while (0)

static eg_status ensure(eg_ctx *ctx, dev_buf &b, size_t bytes) {
    if (b.cap >= bytes) return EG_SUCCESS;
    if (b.p) { cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8;
    cudaError_t ce = cudaMalloc(&b.p, want);
    if (ce != cudaSuccess) { cudaGetLastError(); return fail(ctx, EG_ERR_OUT_OF_MEMORY, "cudaMalloc scratch", ce); }
    b.cap = want;
    return EG_SUCCESS;
}

#define TRY(expr)                              \
    do {                                       \
        eg_status st_ = (expr);                \
        if (st_ != EG_SUCCESS) return st_;     \
    } while (0)

static inline unsigned grid_for(size_t threads, unsigned block) { return (unsigned)((threads + block - 1) / block); }

// Per-call statistics of the equation-evaluation kernels (eg_last_kernel_stats): stat_begin / stat_end put one CUDA event
// pair around a launch of kind `kind` (EG_STAT_KINDS) and count it, `tasks` = what the launch evaluates (equation sides for
// k_commit / k_ring / k_ring_pair, multi-scalar sums for k_msm).
static void reset_call_stats(eg_ctx *ctx) {
    ctx->commit_ev_used = 0;
    for (int q = 0; q < EG_STAT_KINDS; q++) { ctx->kind_tasks[q] = 0; ctx->kind_launches[q] = 0; ctx->kind_ms[q] = 0; }
    for (float &t : ctx->timings) t = 0;
}

// After a failure inside a chunk loop: copies of earlier chunks may still be in flight to / from the caller's buffers and
// the context's staging; drain both streams (ignoring their status) so that the caller may free its buffers and the next
// call on the context starts clean.
static eg_status drain_on_error(eg_ctx *ctx, eg_status st) {
    if (st != EG_SUCCESS) {
        if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
        if (ctx->stream) cudaStreamSynchronize(ctx->stream);
        cudaGetLastError();
    }
    return st;
}

static void stat_begin(eg_ctx *ctx, int kind, size_t tasks) {
    if (ctx->commit_ev_used + 2 > ctx->commit_ev.size()) {
        cudaEvent_t a = nullptr, b = nullptr;
        cudaEventCreate(&a); cudaEventCreate(&b);
        ctx->commit_ev.push_back(a); ctx->commit_ev.push_back(b);
    }
    if (ctx->commit_ev_kind.size() < ctx->commit_ev.size() / 2) ctx->commit_ev_kind.resize(ctx->commit_ev.size() / 2);
    ctx->commit_ev_kind[ctx->commit_ev_used / 2] = (uint8_t)kind;
    ctx->kind_tasks[kind] += tasks; ctx->kind_launches[kind]++;
    cudaEventRecord(ctx->commit_ev[ctx->commit_ev_used], ctx->stream);
    ctx->commit_ev_used += 2;
}

static void stat_end(eg_ctx *ctx) { cudaEventRecord(ctx->commit_ev[ctx->commit_ev_used - 1], ctx->stream); }

// ------------------------------------------------------------------- kernel launches

// The only kernel start site.  The test harness (EG_HOSTSIM) runs the same __global__ function on the CPU once per
// (block, thread), so that its tests cover the index mapping the GPU runs.
template <class... KP, class... A>
static void launch(eg_ctx *ctx, void (*kernel)(KP...), dim3 grid, unsigned block, const A &...args) {
#ifdef EG_HOSTSIM
    hs_launch(kernel, grid, dim3(block), args...);
#else
    kernel<<<grid, block, 0, ctx->stream>>>(args...);
#endif
    ctx->launches++;
}

// one thread per task: ceil(total / block) CTAs of `block` threads
template <class... KP, class... A>
static void launch_flat(eg_ctx *ctx, void (*kernel)(KP...), size_t total, unsigned block, const A &...args) {
    launch(ctx, kernel, grid_for(total, block), block, args...);
}

// CTAs of `kernel` (at `threads` per CTA) that the device holds at once, queried once per context
template <class K>
static eg_status resident_ctas(eg_ctx *ctx, K kernel, unsigned threads, size_t &ctas) {
    int &cached = ctx->resident[reinterpret_cast<const void *>(kernel)];
    if (cached == 0) {
        int per_sm = 0, sms = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, (int)threads, 0));
        CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
        if (per_sm < 1) return fail(ctx, EG_ERR_CUDA, "a persistent kernel does not fit on an SM");
        cached = per_sm * sms;
    }
    ctas = (size_t)cached;
    return EG_SUCCESS;
}

// Persistent grid: at most one wave of resident CTAs, whose threads stride over the `total` tasks.
template <class... KP, class... A>
static eg_status launch_persistent(eg_ctx *ctx, void (*kernel)(KP...), unsigned threads, size_t total, const A &...args) {
    size_t ctas = 0;
    TRY(resident_ctas(ctx, kernel, threads, ctas));
    launch(ctx, kernel, (unsigned)std::min<size_t>(ctas, (total + threads - 1) / threads), threads, args...);
    return EG_SUCCESS;
}

// k_ring's two shapes (device_kernels.inc): rings of <= 2 equations run one CTA of 512 threads per SM with 4-chunk
// tables, longer rings 2 CTAs of 256 threads
struct ring_shape {
    void (*kernel)(ring_params);
    unsigned threads;
};
static ring_shape ring_shape_for(bool short_rings) {
    if (short_rings) return {k_ring<EG_RING2_THREADS, EG_RING2_MINBLOCKS, EG_VCHUNKS_SHORT>, EG_RING2_THREADS};
    return {k_ring<EG_RING_THREADS, EG_RING_MINBLOCKS, EG_VCHUNKS_LONG>, EG_RING_THREADS};
}

// resident threads of the persistent k_ring grid of one shape
static eg_status ring_resident_threads(eg_ctx *ctx, bool short_rings, size_t &threads) {
    const ring_shape s = ring_shape_for(short_rings);
    size_t ctas = 0;
    TRY(resident_ctas(ctx, s.kernel, s.threads, ctas));
    threads = ctas * s.threads;
    return EG_SUCCESS;
}

// Chunk size rounded down to a whole number of waves of the persistent k_ring grid: a chunk of `chunk` items starts
// chunk x rings_per_item ring threads, and a last partial wave costs as much as a full one (47 662 range proofs x 8 rings
// are 5.03 waves of 75 776 threads).  Explicit chunk sizes (eg_ctx_set_chunk_items) are left alone.
static size_t wave_chunk(eg_ctx *ctx, size_t chunk, size_t rings_per_item, bool short_rings) {
#if !defined(EG_HOSTSIM) && !defined(EG_NO_WAVE_CHUNK)
    size_t resident = 0;
    if (ctx->chunk_items || rings_per_item == 0) return chunk;
    if (ring_resident_threads(ctx, short_rings, resident) != EG_SUCCESS) return chunk;
    const size_t waves = chunk * rings_per_item / resident;
    if (waves >= 2) chunk = waves * resident / rings_per_item;
#else
    (void)ctx; (void)rings_per_item; (void)short_rings;
#endif
    return chunk;
}

// Double-buffered chunk pipeline for entry points whose host traffic is comparable to their kernel time (the provers:
// 64 B of randomness in per draw, whole proofs out).  stage_in(c, b) enqueues the host -> device copies of chunk c into
// buffer set b on `cs`; compute(c, b) enqueues its kernels on ctx->stream; stage_out(c, b) enqueues the device -> host
// copies of its results on `cs`.  While the host is blocked in the (pageable) copies of chunks c + 1 and c - 1, the GPU
// runs chunk c.  Hazards: set b's inputs are rewritten only after chunk c - 2's kernels (ev done), its outputs only after
// they were copied out (ev out).
template <class In, class Run, class Out>
static eg_status pipeline_chunks_impl(eg_ctx *ctx, size_t n_chunks, In stage_in, Run compute, Out stage_out) {
    cudaStream_t cs = ctx->copy_stream;
    cudaEvent_t *ev_in = ctx->ev_pipe, *ev_done = ctx->ev_pipe + 2, *ev_out = ctx->ev_pipe + 4;
    if (n_chunks == 0) return EG_SUCCESS;
    TRY(stage_in(0, 0, cs));
    CU(cudaEventRecord(ev_in[0], cs));
    for (size_t c = 0; c < n_chunks; c++) {
        const int b = (int)(c & 1);
        CU(cudaStreamWaitEvent(ctx->stream, ev_in[b], 0));
        if (c >= 2) CU(cudaStreamWaitEvent(ctx->stream, ev_out[b], 0));
        TRY(compute(c, b));
        CU(cudaEventRecord(ev_done[b], ctx->stream));
        if (c + 1 < n_chunks) {
            if (c >= 1) CU(cudaStreamWaitEvent(cs, ev_done[b ^ 1], 0));
            TRY(stage_in(c + 1, b ^ 1, cs));
            CU(cudaEventRecord(ev_in[b ^ 1], cs));
        }
        if (c >= 1) {
            CU(cudaStreamWaitEvent(cs, ev_done[b ^ 1], 0));
            TRY(stage_out(c - 1, b ^ 1, cs));
            CU(cudaEventRecord(ev_out[b ^ 1], cs));
        }
    }
    const int lb = (int)((n_chunks - 1) & 1);
    CU(cudaStreamWaitEvent(cs, ev_done[lb], 0));
    TRY(stage_out(n_chunks - 1, lb, cs));
    CU(cudaStreamSynchronize(cs));
    CU(cudaStreamSynchronize(ctx->stream));
    return EG_SUCCESS;
}

template <class In, class Run, class Out>
static eg_status pipeline_chunks(eg_ctx *ctx, size_t n_chunks, In stage_in, Run compute, Out stage_out) {
    return drain_on_error(ctx, pipeline_chunks_impl(ctx, n_chunks, stage_in, compute, stage_out));
}

static void launch_decode(eg_ctx *ctx, const decode_params &P) { launch_flat(ctx, k_decode, P.n * (size_t)P.n_slots, 256, P); }

static void launch_scalars(eg_ctx *ctx, const scalars_params &P) { launch_flat(ctx, k_scalars, P.n, 256, P); }

static void launch_commit(eg_ctx *ctx, const commit_params &P) {
    const size_t total = P.n * (size_t)P.n_slots;
    stat_begin(ctx, 0, total);
    launch_flat(ctx, k_commit, total, EG_COMMIT_THREADS, P);
    stat_end(ctx);
}

static void launch_terminal(eg_ctx *ctx, const terminal_params &P) { launch_flat(ctx, k_terminal, P.n, 128, P); }

// equation sides of a ring job (tasks of k_ring / k_ring_pair), and whether all its rings have <= 2 equations
static size_t ring_sides(const ring_params &P, bool &short_rings) {
    size_t sides = 0;
    short_rings = true;
    for (uint32_t r = 0; r < P.n_rings; r++) { sides += 2 * (size_t)P.sizes[r]; short_rings = short_rings && P.sizes[r] <= 2; }
    return sides * P.n;
}

// One launch evaluates every equation of every ring of the chunk.  Accounted like k_commit: tasks = equation sides.
static eg_status launch_ring(eg_ctx *ctx, ring_params &P) {
    bool short_rings = true;
    const size_t sides = ring_sides(P, short_rings);
    const ring_shape s = ring_shape_for(short_rings);
    size_t resident = 0;
    TRY(ring_resident_threads(ctx, short_rings, resident));
    TRY(ensure(ctx, ctx->ring_scratch, resident * 2 * EG_VTAB_WORDS * 4));
    P.scratch = (uint32_t *)ctx->ring_scratch.p;
    stat_begin(ctx, 1, sides);
    TRY(launch_persistent(ctx, s.kernel, s.threads, P.n * (size_t)P.n_rings, P));
    stat_end(ctx);
    return EG_SUCCESS;
}

// Pair engine (ring mode 3): two lanes per ring, one launch for all equations of a small chunk; the job's extra single-use
// equation sides (X.n_slots > 0: the sum proof of an EncryptedChoice) ride along as further lanes of the same launch, so the
// longest chain of the launch stays the ring's.  Accounted like k_ring (tasks = equation sides), under its own kind (3).
static eg_status launch_ring_pair(eg_ctx *ctx, ring_params &P, const commit_params &X) {
    bool short_rings = true;
    const size_t sides = ring_sides(P, short_rings), lanes = 2 * P.n * (size_t)P.n_rings, extra = P.n * (size_t)X.n_slots;
    TRY(ensure(ctx, ctx->ring_scratch, lanes * EG_VTAB_WORDS * 4));
    P.scratch = (uint32_t *)ctx->ring_scratch.p;
    stat_begin(ctx, 3, sides + extra);
    launch_flat(ctx, short_rings ? k_ring_pair<EG_VCHUNKS_SHORT> : k_ring_pair<EG_VCHUNKS_LONG>, lanes + extra, EG_PAIR_THREADS, P, X);
    stat_end(ctx);
    return EG_SUCCESS;
}

// one phase of a prover (k_prove, k_rprove): persistent grid, 2 EG_VTAB_WORDS words of window-table scratch per thread
template <class Params>
static eg_status launch_prover_phase(eg_ctx *ctx, void (*kernel)(Params, uint32_t *), const Params &P, size_t total) {
    size_t ctas = 0;
    TRY(resident_ctas(ctx, kernel, EG_RING_THREADS, ctas));
    TRY(ensure(ctx, ctx->ring_scratch, ctas * EG_RING_THREADS * 2 * EG_VTAB_WORDS * 4));
    return launch_persistent(ctx, kernel, EG_RING_THREADS, total, P, (uint32_t *)ctx->ring_scratch.p);
}

static eg_status launch_prove(eg_ctx *ctx, const prove_params &P) {
    TRY(launch_prover_phase(ctx, k_prove<0>, P, P.n * (size_t)P.options));
    TRY(launch_prover_phase(ctx, k_prove<1>, P, P.n));
    return launch_prover_phase(ctx, k_prove<2>, P, P.n * (size_t)P.options);
}

static eg_status launch_rprove(eg_ctx *ctx, const rprove_params &P) {
    TRY(launch_prover_phase(ctx, k_rprove<0>, P, P.n * (size_t)(P.n_rings + 1)));
    TRY(launch_prover_phase(ctx, k_rprove<1>, P, P.n));
    return launch_prover_phase(ctx, k_rprove<2>, P, P.n * (size_t)P.n_rings);
}

static eg_status launch_encrypt(eg_ctx *ctx, const encrypt_params &P) { return launch_persistent(ctx, k_encrypt, EG_RING_THREADS, P.n, P); }

static eg_status launch_decrypt(eg_ctx *ctx, int op, const decrypt_params &P) {
    const bool ct = P.rnd.ct != 0;
    void (*kernel)(decrypt_params) = op == EG_DEC_PLAIN ? (ct ? k_decrypt<EG_DEC_PLAIN, true> : k_decrypt<EG_DEC_PLAIN, false>)
                                                        : (ct ? k_decrypt<EG_DEC_PROOF, true> : k_decrypt<EG_DEC_PROOF, false>);
    return launch_persistent(ctx, kernel, EG_DECRYPT_THREADS, P.n, P);
}

static eg_status launch_sumsq_prove(eg_ctx *ctx, const sumsq_prove_params &P) {
    return launch_persistent(ctx, k_sumsq_prove, EG_RING_THREADS, P.n, P);
}

static eg_status launch_sumsq_stage(eg_ctx *ctx, const sumsq_stage_params &P) {
    launch_flat(ctx, k_sumsq_stage, P.n, 256, P);
    return EG_SUCCESS;
}

static eg_status launch_ceq_prove(eg_ctx *ctx, const ceq_prove_params &P) {
    return launch_persistent(ctx, k_ceq_prove, EG_DECRYPT_THREADS, P.n, P);
}

static eg_status launch_pop_prove(eg_ctx *ctx, const pop_prove_params &P) {
    TRY(launch_persistent(ctx, k_pop_prove<0>, EG_DECRYPT_THREADS, P.n * (size_t)P.k, P));
    return launch_persistent(ctx, k_pop_prove<1>, EG_DECRYPT_THREADS, P.n, P);
}

static void launch_ring_hash(eg_ctx *ctx, const ring_hash_params &P) { launch_flat(ctx, k_ring_hash, P.n * (size_t)P.n_slots, 128, P); }

static void launch_ring_final(eg_ctx *ctx, const ring_final_params &P) { launch_flat(ctx, k_ring_final, P.n, 128, P); }

static void launch_logeq_final(eg_ctx *ctx, const logeq_final_params &P) { launch_flat(ctx, k_logeq_final, P.n, 128, P); }

static void launch_choice_sum(eg_ctx *ctx, const choice_sum_params &P) { launch_flat(ctx, k_choice_sum, 2 * P.n, 128, P); }

static void launch_range_last(eg_ctx *ctx, const range_last_params &P) { launch_flat(ctx, k_range_last, 2 * P.n, 128, P); }

static void launch_verdict(eg_ctx *ctx, const verdict_params &P) { launch_flat(ctx, k_verdict, P.n, 256, P); }

static void launch_qv_verdict(eg_ctx *ctx, const qv_verdict_params &P) { launch_flat(ctx, k_qv_verdict, P.n, 256, P); }

static void launch_share_verdict(eg_ctx *ctx, const share_verdict_params &P) {
    const size_t total = P.n * (size_t)P.n_shares;
    launch_flat(ctx, k_share_verdict, total, 256, P, total);
}

// wide fixed-base table of one base (ge.cuh): EG_WIDE_TABLE_WORDS words, followed by EG_WIDE_SCRATCH_WORDS of window bases
#define EG_TABLE_ALLOC_BYTES ((EG_WIDE_TABLE_WORDS + EG_WIDE_SCRATCH_WORDS) * 4)
template <int BITS>
static void launch_build_table_b(eg_ctx *ctx, const uint32_t *enc_words, int use_generator, uint32_t *table, uint32_t *status) {
    uint32_t *bases = table + EG_BITS_TABLE_WORDS(BITS);
    launch(ctx, k_wide_bases<BITS>, 1, 1, enc_words, use_generator, bases, status);
    launch_flat(ctx, k_wide_fill<BITS>, (size_t)EG_BITS_WINDOWS(BITS) * (EG_BITS_ENTRIES(BITS) / EG_WIDE_BLOCK), 64, bases, table);
}
static void launch_build_table(eg_ctx *ctx, const uint32_t *enc_words, int use_generator, uint32_t *table, uint32_t *status) {
    launch_build_table_b<EG_WIDE_BITS>(ctx, enc_words, use_generator, table, status);
}
// narrow (EG_NARROW_BITS) table of a per-call base: EG_NARROW_ALLOC_WORDS words at `table`
static void launch_build_narrow_table(eg_ctx *ctx, const uint32_t *enc_words, uint32_t *table, uint32_t *status) {
    launch_build_table_b<EG_NARROW_BITS>(ctx, enc_words, 0, table, status);
}

static void launch_admissible(eg_ctx *ctx, const uint64_t *values, int count, uint32_t *adm) {
    launch_flat(ctx, k_admissible, count, 64, values, count, adm);
}

// per-slot masked sums of planar points into `partial` (blocks per slot returned)
static int launch_tally_partial(eg_ctx *ctx, const uint32_t *pts, size_t n, int n_slots, const uint8_t *verdicts, uint32_t *partial) {
    const int blocks = (int)std::max<size_t>(1, std::min<size_t>(EG_TALLY_BLOCKS, (n + EG_TALLY_THREADS - 1) / EG_TALLY_THREADS));
    launch(ctx, k_tally_partial, dim3(blocks, n_slots), EG_TALLY_THREADS, pts, n, verdicts, partial);
    return blocks;
}

static void launch_tally_final(eg_ctx *ctx, const uint32_t *partial, int count, int n_slots, uint32_t *running, int accumulate,
                               uint8_t *encode_out) {
    launch(ctx, k_tally_final, n_slots, 32, partial, count, running, accumulate, encode_out);
}

static void launch_elements_validate(eg_ctx *ctx, const uint8_t *enc, size_t n, uint8_t *ok) {
    launch_flat(ctx, k_elements_validate, n, 128, enc, n, ok);
}

static void launch_scalars_validate(eg_ctx *ctx, const uint8_t *sc_in, size_t n, uint8_t *ok) {
    launch_flat(ctx, k_scalars_validate, n, 256, sc_in, n, ok);
}

static void launch_keyset_verdict(eg_ctx *ctx, const keyset_verdict_params &P) { launch_flat(ctx, k_keyset_verdict, P.n, 256, P); }

static void launch_unpack(eg_ctx *ctx, const unpack_params &P) { launch_flat(ctx, k_unpack, P.n, 256, P); }

static void launch_b64url(eg_ctx *ctx, const b64_params &P, bool encode) {
    launch_flat(ctx, encode ? k_b64url<1> : k_b64url<0>, P.n * (size_t)P.groups, 256, P);
}

static void launch_scalars_from_wide(eg_ctx *ctx, const uint8_t *wide, size_t n, uint8_t *out) {
    launch_flat(ctx, k_scalars_from_wide, n, 256, wide, n, out);
}

static void launch_double_mul(eg_ctx *ctx, const uint8_t *a, const uint8_t *A, const uint8_t *b, size_t n, int mode, uint8_t *out, uint8_t *okv) {
    launch_flat(ctx, k_double_mul, n, EG_COMMIT_THREADS, a, A, b, n, mode, ctx->d_table_g, out, okv);
}

static void launch_ciphertexts_sum(eg_ctx *ctx, const uint8_t *parts, size_t n_parts, size_t n_cts, uint8_t *out, uint32_t *bad) {
    launch_flat(ctx, k_ciphertexts_sum, 2 * n_cts, 64, parts, n_parts, n_cts, out, bad);
}

// k_msm over the slot table uploaded last; slots whose encoding was deferred by upload_slots are encoded together by
// k_terminal (one inversion per item) right after.
static eg_status launch_msm(eg_ctx *ctx, const msm_params &P0) {
    msm_params P = P0;
    const uint32_t n_term = ctx->term_plan.n_pts;
    if (n_term) {
        TRY(ensure(ctx, ctx->term, P.n * (size_t)n_term * 128));
        P.term_pts = (uint32_t *)ctx->term.p;
    }
    const size_t total = P.n * (size_t)P.n_slots;
    stat_begin(ctx, 2, total);
    launch_flat(ctx, k_msm, total, 128, P);
    stat_end(ctx);
    if (n_term) {
        terminal_params tp = ctx->term_plan;
        tp.n = P.n; tp.term_pts = P.term_pts; tp.commit = P.commit;
        launch_terminal(ctx, tp);
    }
    return EG_SUCCESS;
}

static void launch_sigma_final(eg_ctx *ctx, const sigma_final_params &P) { launch_flat(ctx, k_sigma_final, P.n, 128, P); }

static void launch_sumsq_final(eg_ctx *ctx, const sumsq_final_params &P) { launch_flat(ctx, k_sumsq_final, P.n, 128, P); }

// `P` lives in host memory; the device copy `d_P` is what the kernel reads (the struct exceeds the 4 KB launch limit)
static void launch_share_final(eg_ctx *ctx, const share_final_params &P, const share_final_params *d_P) {
    launch_flat(ctx, k_share_final, P.n * (size_t)P.n_shares, 128, d_P);
}

static void launch_dlog_build(eg_ctx *ctx, const dlog_build_params &P, size_t threads) {
    launch_flat(ctx, k_dlog_build, threads, 128, P, threads);
}

static void launch_dlog_lookup(eg_ctx *ctx, const dlog_lookup_params &P) { launch_flat(ctx, k_dlog_lookup, P.n, 128, P); }

static void launch_dlog_get(eg_ctx *ctx, const dlog_get_params &P) { launch_flat(ctx, k_dlog_get, P.n, 128, P); }

// Giant-step walk of a BSGS table (giants > 1) over the items that the probe of giant step 0 left at found 0.  Each item gets
// `segs` threads of seg_steps consecutive steps: enough threads in all to fill the GPU when the batch is small (one element
// spreads over the whole device), one per item when the batch alone fills it, and never fewer than EG_WALK_MIN_STEPS steps
// per thread, which keep the cost of a thread's start ([1/2]M and one fixed-base product, about 3 000 field operations)
// small against its walk.
#ifdef EG_HOSTSIM
#define EG_WALK_MIN_STEPS 16           // the CPU harness: short segments, so that small tables cross segment boundaries
#define EG_WALK_TARGET_THREADS 64
#else
#define EG_WALK_MIN_STEPS 2048
#define EG_WALK_TARGET_THREADS (1u << 18)
#endif
static void launch_dlog_walk(eg_ctx *ctx, const eg_dlog_table *t, size_t n, const uint8_t *enc, uint64_t *values, uint8_t *found) {
    if (t->giants <= 1 || n == 0) return;
    dlog_walk_params P;
    memset(&P, 0, sizeof P);
    const uint64_t steps = t->giants - 1;
    const uint64_t max_segs = (steps + EG_WALK_MIN_STEPS - 1) / EG_WALK_MIN_STEPS;
    const uint64_t want = std::max<uint64_t>(1, (EG_WALK_TARGET_THREADS + n - 1) / n);
    uint64_t segs = std::max<uint64_t>(1, std::min(max_segs, want));
    P.seg_steps = (steps + segs - 1) / segs;
    P.seg_steps = (P.seg_steps + EG_WALK_BLOCK - 1) / EG_WALK_BLOCK * EG_WALK_BLOCK;
    segs = (steps + P.seg_steps - 1) / P.seg_steps;
    P.n = n; P.enc = enc; P.found = found; P.values = (unsigned long long *)values;
    P.lo = t->lo; P.hi = t->hi; P.m = t->m; P.giants = t->giants; P.segs = (uint32_t)segs;
    P.cap = t->cap; P.keys = t->d_keys; P.vals = (const unsigned long long *)t->d_vals; P.table_g = ctx->d_table_g;
    for (int w = 0; w < 24; w++) P.step[w] = t->step[w];
    const size_t total = n * (size_t)segs;
    launch_flat(ctx, k_dlog_walk, total, EG_DECRYPT_THREADS, P, total);
}

#include "comm.inc"

#ifdef EG_HOSTSIM
extern "C" const char *eg_version(void) { return "eg_b200 0.1.0 HOSTSIM test harness (not a product build)"; }
#else
extern "C" const char *eg_version(void) { return "eg_b200 0.1.0 sm_100a"; }
#endif

extern "C" const char *eg_last_error(const eg_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

// on a multi-device context: the sum over its devices
extern "C" uint64_t eg_kernel_launch_count(const eg_ctx *ctx) {
    if (!ctx) return 0;
    uint64_t total = ctx->launches;
    for (const eg_ctx *c : ctx->children) total += c->launches;
    return total;
}

extern "C" void *eg_ctx_stream(const eg_ctx *ctx) { return ctx ? (void *)ctx_first(const_cast<eg_ctx *>(ctx))->stream : nullptr; }

// the ring-proof equation kernels: kinds 0 (k_commit), 1 (k_ring) and 3 (k_ring_pair) of eg_last_kernel_stats
extern "C" eg_status eg_last_commit_stats(const eg_ctx *ctx, uint64_t *launches, uint64_t *tasks, float *ms) {
    if (!ctx) return EG_ERR_INVALID_ARG;
    uint64_t l = 0, t = 0;
    for (int kind : {0, 1, 3}) {
        uint64_t kl = 0, kt = 0;
        eg_last_kernel_stats(ctx, kind, &kl, &kt, nullptr);
        l += kl; t += kt;
    }
    float m = ctx->timings[2];          // on a multi-device context: the slowest device
    if (ctx_is_multi(ctx)) { m = 0; for (const eg_ctx *c : ctx->children) m = std::max(m, c->timings[2]); }
    if (launches) *launches = l;
    if (tasks) *tasks = t;
    if (ms) *ms = m;
    return EG_SUCCESS;
}

// kind 0: k_commit launches of the last call, kind 1: k_ring launches (tasks = equation sides), kind 2: k_msm (tasks = sums),
// kind 3: k_ring_pair launches (tasks = equation sides)
extern "C" eg_status eg_last_kernel_stats(const eg_ctx *ctx, int kind, uint64_t *launches, uint64_t *tasks, float *ms) {
    if (!ctx || kind < 0 || kind >= EG_STAT_KINDS) return EG_ERR_INVALID_ARG;
    if (ctx_is_multi(ctx)) {
        uint64_t l = 0, t = 0; float m = 0;
        for (const eg_ctx *c : ctx->children) { l += c->kind_launches[kind]; t += c->kind_tasks[kind]; m = std::max(m, c->kind_ms[kind]); }
        if (launches) *launches = l;
        if (tasks) *tasks = t;
        if (ms) *ms = m;
        return EG_SUCCESS;
    }
    if (launches) *launches = ctx->kind_launches[kind];
    if (tasks) *tasks = ctx->kind_tasks[kind];
    if (ms) *ms = ctx->kind_ms[kind];
    return EG_SUCCESS;
}

extern "C" eg_status eg_last_timings(const eg_ctx *ctx, float out_ms[5]) {
    if (!ctx || !out_ms) return EG_ERR_INVALID_ARG;
    for (int i = 0; i < 5; i++) out_ms[i] = ctx->timings[i];
    for (const eg_ctx *c : ctx->children)
        for (int i = 0; i < 5; i++) out_ms[i] = std::max(out_ms[i], c->timings[i]);
    return EG_SUCCESS;
}


extern "C" eg_status eg_selftest_field(eg_ctx *ctx, size_t n, uint64_t seed, uint64_t *mismatches) {
    if (!ctx || !mismatches) return EG_ERR_INVALID_ARG;
    if (ctx_is_multi(ctx)) {
        *mismatches = 0;
        for (eg_ctx *c : ctx->children) {
            uint64_t m = 0;
            eg_status st = eg_selftest_field(c, n, seed, &m);
            if (st != EG_SUCCESS) { ctx->err = c->err; return st; }
            *mismatches += m;
        }
        return EG_SUCCESS;
    }
    CU(cudaSetDevice(ctx->device));
    *mismatches = 0;
#ifndef EG_HOSTSIM
    unsigned long long *d = (unsigned long long *)(ctx->d_status + 64);
    CU(cudaMemsetAsync(d, 0, 8, ctx->stream));
    launch_flat(ctx, k_selftest_field, n, 128, n, seed, d);
    unsigned long long h = 0;
    CU(cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    *mismatches = h;
#else
    (void)n; (void)seed;
#endif
    return EG_SUCCESS;
}

extern "C" eg_status eg_ctx_set_chunk_items(eg_ctx *ctx, size_t items) {
    if (!ctx) return EG_ERR_INVALID_ARG;
    ctx->chunk_items = items;
    for (eg_ctx *c : ctx->children) c->chunk_items = items;
    return EG_SUCCESS;
}

extern "C" eg_status eg_ctx_set_ring_mode(eg_ctx *ctx, int mode) {
    if (!ctx || mode < 0 || mode > 3) return EG_ERR_INVALID_ARG;
    ctx->ring_mode = mode;
    for (eg_ctx *c : ctx->children) c->ring_mode = mode;
    return EG_SUCCESS;
}

extern "C" eg_status eg_ctx_set_key_table_min(eg_ctx *ctx, size_t min_tallies) {
    if (!ctx) return EG_ERR_INVALID_ARG;
    ctx->key_table_min = min_tallies;
    for (eg_ctx *c : ctx->children) c->key_table_min = min_tallies;
    return EG_SUCCESS;
}

extern "C" eg_status eg_ctx_set_prover_mode(eg_ctx *ctx, int constant_time) {
    if (!ctx || constant_time < 0 || constant_time > 1) return EG_ERR_INVALID_ARG;
    ctx->prover_ct = constant_time;
    for (eg_ctx *c : ctx->children) c->prover_ct = constant_time;
    return EG_SUCCESS;
}

extern "C" eg_status eg_ctx_create(int device_id, eg_ctx **out) {
    if (!out) return EG_ERR_INVALID_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device_id < 0 || device_id >= count) {
        cudaGetLastError();
        return EG_ERR_NO_DEVICE;
    }
    eg_ctx *ctx = new (std::nothrow) eg_ctx();
    if (!ctx) return EG_ERR_OUT_OF_MEMORY;
    ctx->device = device_id;
    auto bail = [&](eg_status st) { eg_ctx_destroy(ctx); return st; };
    if (cudaSetDevice(device_id) != cudaSuccess) return bail(EG_ERR_NO_DEVICE);
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(EG_ERR_CUDA);
    for (auto &e : ctx->ev) if (cudaEventCreate(&e) != cudaSuccess) return bail(EG_ERR_CUDA);
    if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(EG_ERR_CUDA);
    for (auto &e : ctx->ev_h2d) if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return bail(EG_ERR_CUDA);
    for (auto &e : ctx->ev_pipe) if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return bail(EG_ERR_CUDA);
    if (cudaMalloc(&ctx->d_table_g, EG_TABLE_ALLOC_BYTES) != cudaSuccess) return bail(EG_ERR_OUT_OF_MEMORY);
    if (cudaMalloc(&ctx->d_table_k, EG_TABLE_ALLOC_BYTES) != cudaSuccess) return bail(EG_ERR_OUT_OF_MEMORY);
    if (cudaMalloc(&ctx->d_status, 1024) != cudaSuccess) return bail(EG_ERR_OUT_OF_MEMORY);
    launch_build_table(ctx, nullptr, 1, ctx->d_table_g, ctx->d_status);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess || cudaGetLastError() != cudaSuccess) return bail(EG_ERR_CUDA);
    *out = ctx;
    return EG_SUCCESS;
}

extern "C" void eg_ctx_destroy(eg_ctx *ctx) {
    if (!ctx) return;
    if (ctx_is_multi(ctx) || (!ctx->stream && !ctx->d_status)) {       // the parent of a multi-device context owns no device state
        for (eg_ctx *c : ctx->children) eg_ctx_destroy(c);
        delete ctx;
        return;
    }
    cudaSetDevice(ctx->device);
#ifndef EG_HOSTSIM
    if (ctx->comm) {
        cudaStreamSynchronize(ctx->stream);
        nccl_api *api = nccl_load();
        if (api) api->CommDestroy((ncclComm_t)ctx->comm);
        ctx->comm = nullptr;
    }
#endif
    dev_buf *bufs[] = {&ctx->pts, &ctx->enc, &ctx->commit, &ctx->chal, &ctx->flags, &ctx->res[0], &ctx->res[1], &ctx->res[2],
                       &ctx->in[0], &ctx->in[1], &ctx->in[2], &ctx->in[3], &ctx->verdicts, &ctx->partial, &ctx->running,
                       &ctx->adm, &ctx->misc, &ctx->slots, &ctx->consts, &ctx->res_big, &ctx->ring_scratch,
                       &ctx->in2[0], &ctx->in2[1], &ctx->in2[2], &ctx->term, &ctx->gather, &ctx->xtab};
    for (dev_buf *b : bufs) if (b->p) cudaFree(b->p);
    for (dev_buf &b : ctx->ws) if (b.p) cudaFree(b.p);
    if (ctx->d_table_g) cudaFree(ctx->d_table_g);
    if (ctx->d_table_k) cudaFree(ctx->d_table_k);
    if (ctx->d_table_h) cudaFree(ctx->d_table_h);
    if (ctx->d_status) cudaFree(ctx->d_status);
    for (auto &e : ctx->ev) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->commit_ev) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->ev_h2d) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->ev_pipe) if (e) cudaEventDestroy(e);
    for (auto &set : ctx->pp) for (dev_buf &b : set) if (b.p) cudaFree(b.p);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" eg_status eg_ctx_set_receiver(eg_ctx *ctx, const uint8_t key[32]) {
    if (!ctx || !key) return EG_ERR_INVALID_ARG;
    if (ctx_is_multi(ctx)) {
        ctx->has_receiver = false;
        for (eg_ctx *c : ctx->children) {
            eg_status st = eg_ctx_set_receiver(c, key);
            if (st != EG_SUCCESS) { ctx->err = c->err; return st; }
        }
        memcpy(ctx->key, key, 32);
        ctx->has_receiver = true;
        return EG_SUCCESS;
    }
    CU(cudaSetDevice(ctx->device));
    uint32_t *d_key = ctx->d_status + 8;
    CU(cudaMemcpyAsync(d_key, key, 32, cudaMemcpyHostToDevice, ctx->stream));
    launch_build_table(ctx, d_key, 0, ctx->d_table_k, ctx->d_status);
    uint32_t status = 0;
    CU(cudaMemcpyAsync(&status, ctx->d_status, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    if (status == 1) { ctx->has_receiver = false; return fail(ctx, EG_ERR_INVALID_ELEMENT, "receiver key does not represent a group element"); }
    if (status == 2) { ctx->has_receiver = false; return fail(ctx, EG_ERR_IDENTITY_KEY, "receiver key is the group identity"); }
    memcpy(ctx->key, key, 32);
    ctx->has_receiver = true;
    return EG_SUCCESS;
}

// Pedersen blinding base H of CommitmentEquivalenceProof (commitment.rs:140-145: `commitment_blinding_base`), e.g. the
// Bulletproofs base of tests/snapshots.rs:253-257.  Gets the same wide fixed-base table as G and K.
extern "C" eg_status eg_ctx_set_blinding_base(eg_ctx *ctx, const uint8_t base[32]) {
    if (!ctx || !base) return EG_ERR_INVALID_ARG;
    if (ctx_is_multi(ctx)) {
        ctx->has_blinding_base = false;
        for (eg_ctx *c : ctx->children) {
            eg_status st = eg_ctx_set_blinding_base(c, base);
            if (st != EG_SUCCESS) { ctx->err = c->err; return st; }
        }
        memcpy(ctx->blinding_base, base, 32);
        ctx->has_blinding_base = true;
        return EG_SUCCESS;
    }
    CU(cudaSetDevice(ctx->device));
    if (!ctx->d_table_h) {
        cudaError_t ce = cudaMalloc(&ctx->d_table_h, EG_TABLE_ALLOC_BYTES);
        if (ce != cudaSuccess) { cudaGetLastError(); ctx->d_table_h = nullptr; return fail(ctx, EG_ERR_OUT_OF_MEMORY, "cudaMalloc H table", ce); }
    }
    uint32_t *d_key = ctx->d_status + 16;
    CU(cudaMemcpyAsync(d_key, base, 32, cudaMemcpyHostToDevice, ctx->stream));
    launch_build_table(ctx, d_key, 0, ctx->d_table_h, ctx->d_status);
    uint32_t status = 0;
    CU(cudaMemcpyAsync(&status, ctx->d_status, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    ctx->has_blinding_base = false;
    if (status == 1) return fail(ctx, EG_ERR_INVALID_ELEMENT, "blinding base does not represent a group element");
    if (status == 2) return fail(ctx, EG_ERR_IDENTITY_KEY, "blinding base is the group identity");
    memcpy(ctx->blinding_base, base, 32);
    ctx->has_blinding_base = true;
    return EG_SUCCESS;
}

#include "api_ballots.inc"

#include "api_group.inc"

#include "api_range_qv.inc"

#include "api_sharing.inc"

#include "api_provers.inc"

#include "api_misc.inc"

#include "api_sigma.inc"

#include "api_decrypt.inc"

#include "api_decrypt_side.inc"

#include "api_sigma_provers.inc"

#include "api_weighted_sum.inc"

#include "api_group_sum.inc"

#include "api_multi.inc"
