// engine.cu -- host side of the sdpa_b200 engine: the B200 re-design of the body of
// attention() (attention-mpi.c:191-407).
//
//   reference (MPI ranks, AVX-512)                     here (GPUs, streams, NCCL)
//   ------------------------------------------------   -------------------------------------------
//   owner_count/owner_disp K/V row shards (:19-27,199)  one K/V shard per GPU, same map
//   root cvt_d2f of K,V + Bcast/Scatterv (:213-266)     per-GPU chunked H2D of its own rows, cast on
//                                                       the device (fp32 or bf16), shard stays resident
//   ping-pong Q batches via Ibcast (:268-330)           two Q buffers per GPU; H2D of batch i+1 on the
//                                                       copy stream overlaps the kernel of batch i
//   per-row online softmax loop (:333-338)              one fused kernel per batch (f32 SIMT / bf16 tcgen05)
//   Iallreduce MAX, rescale, Iallreduce SUM,            same three collectives with NCCL on a comm stream
//   normalise, Ireduce SUM to root (:340-380)           (overlapping the next batch), or one fused
//                                                       peer-memory merge kernel on the root GPU
//   cvt_f2d + copy into result (:365-376,387-399)       fused into the merge / kernel epilogue, D2H on the
//                                                       copy-out stream
#include "common.cuh"
#include "nccl_loader.h"

#include <dlfcn.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <atomic>
#include <string>
#include <vector>

namespace sdpa {

// ---------------------------------------------------------------------------
// error string (thread local)
// ---------------------------------------------------------------------------
static thread_local char g_error[1024] = "";

void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}
const char* get_error() { return g_error; }

static std::atomic<unsigned long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
unsigned long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

// ---------------------------------------------------------------------------
// NCCL loader
// ---------------------------------------------------------------------------
const NcclApi* nccl_api()
{
    static NcclApi api;
    static int state = 0;  // 0 = untried, 1 = ok, -1 = failed
    if (state == 1) return &api;
    if (state == -1) {
        set_error("NCCL is not loadable on this host (libnccl.so.2)");
        return nullptr;
    }
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
        state = -1;
        set_error("dlopen(libnccl.so.2) failed: %s", dlerror());
        return nullptr;
    }
    bool ok = true;
    auto sym = [&](const char* name) {
        void* p = dlsym(h, name);
        if (!p) ok = false;
        return p;
    };
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
    api.Reduce = (decltype(api.Reduce))sym("ncclReduce");
    api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
    api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
    api.Send = (decltype(api.Send))sym("ncclSend");
    api.Recv = (decltype(api.Recv))sym("ncclRecv");
    api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    api.GetVersion = (decltype(api.GetVersion))sym("ncclGetVersion");
    if (!ok) {
        state = -1;
        set_error("libnccl is missing a required symbol");
        return nullptr;
    }
    state = 1;
    return &api;
}

#define SDPA_NCCL_TRY(expr)                                                                   \
    do {                                                                                      \
        ::sdpa::ncclResult_t _r = (expr);                                                     \
        if (_r != ::sdpa::ncclSuccess) {                                                      \
            ::sdpa::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                   \
                              ::sdpa::nccl_api() ? ::sdpa::nccl_api()->GetErrorString(_r) : "?"); \
            return SDPA_ERR_NCCL;                                                             \
        }                                                                                     \
    } while (0)

// ---------------------------------------------------------------------------
// One K/V shard = one GPU.
// ---------------------------------------------------------------------------
// Device buffer.  Work buffers come from the device's stream-ordered memory pool (cudaMallocAsync) whose release threshold
// is lifted at context creation and which sdpa_runtime_init pre-fills (SDPA_PREALLOC_MB): inside the timed attention() call an
// allocation is then a pool hit (microseconds) instead of a cudaMalloc (a fraction of a millisecond each, ~25 of them on a
// first call).  Buffers exported over CUDA IPC must be plain cudaMalloc memory (`shareable`).  SDPA_MEM_POOL=0: cudaMalloc only.
static bool mem_pool_enabled()
{
    static const bool on = [] {
        const char* e = getenv("SDPA_MEM_POOL");
        return !(e && *e == '0');
    }();
    return on;
}
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    bool pooled = false;
    sdpa_status reserve(size_t want, bool shareable = false)
    {
        if (want <= bytes) return SDPA_OK;
        if (p) {
            SDPA_CUDA_TRY(cudaDeviceSynchronize());   // growth while earlier work may still read the old block (rare path)
            release();
        }
        size_t sz = (want + 255) & ~(size_t)255;
        if (!shareable && mem_pool_enabled()) {
            SDPA_CUDA_TRY(cudaMallocAsync(&p, sz, cudaStreamPerThread));
            SDPA_CUDA_TRY(cudaStreamSynchronize(cudaStreamPerThread));   // usable from every stream from here on
            pooled = true;
        } else {
            SDPA_CUDA_TRY(cudaMalloc(&p, sz));
            pooled = false;
        }
        bytes = sz;
        return SDPA_OK;
    }
    void release()
    {
        if (p) {
            if (pooled) {
                cudaFreeAsync(p, cudaStreamPerThread);
                cudaStreamSynchronize(cudaStreamPerThread);
            } else {
                cudaFree(p);
            }
        }
        p = nullptr;
        bytes = 0;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct Shard {
    int dev = 0;
    int grank = 0;  // global shard index (the reference's mpi_rank)
    cudaStream_t s_in = nullptr, s_compute = nullptr, s_comm = nullptr, s_out = nullptr;
    ncclComm_t comm = nullptr;

    // resident shard in compute precision
    DevBuf Kc, Vc;
    // Cast-ahead (queued device-resident passes): a second K/V set, so that the casts of pass i+1 (side stream s_cast,
    // small-footprint kernel) run under the fused kernel of pass i, which still reads the other set.  Kc / Vc always name
    // the set of the pass being issued (the sets swap per pass); kv_guard[set] = event behind the last kernel that read it.
    DevBuf KcAlt, VcAlt;
    cudaStream_t s_cast = nullptr;
    cudaEvent_t ev_cast_done = nullptr;
    cudaEvent_t kv_guard[2] = {nullptr, nullptr}, ev_kv_read[2] = {nullptr, nullptr};
    int kv_set = 0;
    bool ahead_call = false;                 // the pass being issued casts ahead (set by load_kv, consumed by attention_impl)
    cudaEvent_t ev_fence = nullptr;
    // Queued passes that do NOT cast ahead (several Q batches, another shape) keep their own slot order and record no per-slot
    // events: the end of each one is recorded here, and every later side-stream cast waits for it as well (a completed event
    // costs nothing), so that a cast never overwrites a K/V set or Q slot such a pass still reads.
    cudaEvent_t ev_plain_end = nullptr;
    bool ahead_ever = false, plain_end_recorded = false;
    size_t k_lo_off = 0, v_lo_off = 0, q_lo_off = 0;   // split precision: elements from an operand's hi array to its lo array
    int n_local = 0;
    // staging for fp64 uploads of K/V (two chunks in flight)
    DevBuf kv_stage[2];
    cudaEvent_t ev_stage_ready[2] = {nullptr, nullptr}, ev_stage_free[2] = {nullptr, nullptr};
    // ping-pong Q batches
    DevBuf q64[2], qc[2];
    cudaEvent_t ev_q_ready[2] = {nullptr, nullptr}, ev_q_free[2] = {nullptr, nullptr};
    // per-batch state
    DevBuf part_o, part_tmax, part_lsum;       // split-KV partials of the batch in flight
    DevBuf contrib[2], tmax[2], lsum[2];        // merged local state (ping-pong with the collectives)
    DevBuf gmax[2], gsum[2];                    // allreduce results
    DevBuf out32[2], out64[2];                  // root: reduced fp32 batch / fp64 batch for D2H
    cudaEvent_t ev_compute_done[2] = {nullptr, nullptr}, ev_slot_free[2] = {nullptr, nullptr};
    cudaEvent_t ev_comm_done[2] = {nullptr, nullptr};
    // what the fused kernel reads as K / V: the resident Kc / Vc, or the caller's arrays when they already are in compute
    // precision (typed passes: bf16 operands at BF16, fp32 operands at F32 -- no cast at all)
    const void* k_in = nullptr;
    const void* v_in = nullptr;
    // K/V casts of a device-resident call that wait for the first Q batch so that all three share one launch
    void* pend_dst[2] = {nullptr, nullptr};
    const void* pend_src[2] = {nullptr, nullptr};   // element type: sdpa_ctx::dtype
    size_t pend_cnt[2] = {0, 0};
    int npend = 0;
    cudaEvent_t ev_join[3] = {nullptr, nullptr, nullptr};
    // Stage timing: one pool of timestamp events ("marks"); each category -- casts [0], fused kernel [1],
    // merge + collectives [2], the whole call [3] -- keeps (begin, end) indices into it.  Adjacent stages on the
    // compute stream share a mark (the end of the cast IS the begin of the fused kernel), so a device-resident
    // single-GPU pass records 4 events, not 11.  Pairs accumulate call after call and are only turned into
    // numbers on demand (sdpa_last_timings / sdpa_accumulated_timings): the queries cost ~11 us of host time.
    std::vector<cudaEvent_t> marks;
    bool marks_on = true;                    // this call records stage marks (queued passes may sample: sdpa_ctx::mark_every)
    bool last_call_queued = false;           // the previous call ended without a host wait: its end mark is this call's begin mark
    cudaEvent_t ev_begin = nullptr;          // ordering-only begin event of an unmarked call (side streams fork from it)
    size_t marks_used = 0;
    int open_mark = -1;                      // last mark on s_compute with nothing enqueued behind it, or -1
    std::vector<int> tpair[4];               // begin, end, begin, end, ...
    size_t tpair_last[4] = {0, 0, 0, 0};     // where the last call's pairs start
    double acc_ms[4] = {0, 0, 0, 0};        // folded (already queried) time since the last reset
    UmmaPlan* plan = nullptr;
    int sm_count = 148;
};

}  // namespace sdpa

using namespace sdpa;

// Root form of the device-side exchange: in-stream (one merge kernel on the root per batch) or on the comm stream.
// "auto": single-batch passes take instream at two GPUs and pushsync beyond; passes of several Q batches take overlap (the
// comm-stream merge, measured on c4 at 4 GPUs).
static constexpr const char* kRootMergeDefault = "auto";
// Deferred guard repair on contexts with several K/V shards (agreement by all-reduce at sdpa_synchronize): default.
static constexpr bool kDeferAcrossGpus = false;

struct sdpa_ctx {
    sdpa_config cfg;
    std::vector<Shard> shards;
    int world = 1;
    int rank_base = 0;
    int dk = 0, dv = 0;
    int prec = SDPA_PREC_F32;   // resolved precision of the resident shard
    int dtype = SDPA_DTYPE_F64; // element type of the operands and the result of the pass the shard was loaded for
    bool zero_copy = false;     // the fused kernel reads the caller's K/V/Q in place (Shard::k_in / v_in, Q per batch)
    int q_batch = 0;
    bool peer_ok = false;
    float last_timing[6] = {0, 0, 0, 0, 0, 0};
    bool last_timing_valid = true;          // false: last_timing[0..3] still have to be computed from the event pairs
    double acc_fused_launches = 0, acc_calls = 0;   // over the calls that recorded stage marks
    // Deferred guard repair (queued passes): the exact twin is not launched behind every fast kernel; sdpa_synchronize reads the
    // guard rings once, the processes agree (MAX all-reduce) on the passes in which ANY shard raised its guard, and those
    // passes are re-run with the exact variant -- their arrays are still valid then (contract of sdpa_enqueue_device_full; with
    // several processes sdpa_synchronize is collective like the passes themselves).  SDPA_DEFER_TWIN=0 keeps the twin in the stream.
    struct GuardRef { int shard; unsigned int slot, epoch; };
    struct PendingPass {
        int dtype;                           // re-run as the same typed pass
        std::vector<const void*> K, V, Q;     // per local shard
        std::vector<int> n_local;
        int dk, dv;
        void* result; int m;
        std::vector<GuardRef> guards;         // every fused launch of the pass
    };
    std::vector<PendingPass> pending;
    std::vector<GuardRef> call_guards;        // collected by the attention call in flight
    bool defer_twin = true, deferring = false, repairing = false;
    bool defer_multi = kDeferAcrossGpus;    // contexts with several shards: SDPA_DEFER_TWIN=2 / 1 overrides
    unsigned int ring_use = 0;              // fused launches since the pending passes were last resolved (the guard ring has kGuardRing words)
    int mark_every = 1;                     // queued passes: stage marks on every mark_every-th pass (SDPA_STAGE_TIMING_EVERY); blocking: always
    unsigned long long queued_seq = 0;
    const char* last_kernel = "none";
    // Queued passes of a one-GPU-per-process context (sdpa_enqueue_device_full) alternate exchange slots and are not joined at
    // the end of the call, so the comm stream merges pass i while the compute stream already runs the cast and fused kernel
    // of pass i+1 (SDPA_OVERLAP_PASSES=0 turns that off).  Blocking calls always join.
    bool qshard = false;                    // SDPA_DIST_Q in effect: every shard holds ALL K/V rows, Q rows are sharded, no exchange
    bool overlap_passes = false;
    DevBuf cast_trace;                      // SDPA_CAST_TRACE=<path> (developer aid, single-GPU contexts): per-CTA stamps of the background cast
    std::string cast_trace_path;            // + [600..603] begin/end stamps of the fused kernels of the last two passes, dumped at destroy
    unsigned long long trace_pass = 0;
    struct ByteRange { const char* p; size_t n; };
    std::vector<ByteRange> queued_results;  // results of the queued passes still in flight (a pass that reads one of them cannot cast ahead)
    bool cast_ahead = true;                 // SDPA_CAST_AHEAD=0: the casts of a queued pass stay on the compute stream
    unsigned long long batch_seq = 0;       // batches issued by queued passes with sequence slots (slot = batch_seq & 1)
    bool exchange_pending = false;          // overlap mode left exchange work behind: drain before freeing / reallocating slots
    // device-side exchange across processes (one GPU per process): state buffers + flags shared through CUDA IPC
    struct Ipc {
        bool ready = false;
        int cap_rows = 0, dv = 0, slice_cap = 0;
        DevBuf xbuf[2];                 // [contrib rows*dv | tmax rows | lsum rows], one per ping-pong slot
        // uint32 flags: [0..1] ready[slot] (root merge), [2..3] consumed[slot] (root's copy is the one polled), block
        // counters [4..5] root merge, [6..7] slice merge, [8..9] collect, [10..11] routed split merge;
        // [kFlagStaged + slot*64 + r] "rank r's rows of the batch are staged" (root's copy, written by rank r over NVLink);
        // [kFlagDelivered + slot*64 + r] "source rank r has delivered its state of my rows into my inbox" (written by rank r)
        static constexpr int kFlagStaged = 256, kFlagDelivered = 512;   // two slots x 64 ranks each; 4096-byte block
        DevBuf flags;
        DevBuf stage[2];                // fp64 batch assembled from every rank's slice (the root's copy is the one used)
        std::vector<void*> peer_x[2];   // every rank's xbuf (own pointer for itself)
        std::vector<unsigned int*> peer_flags;  // every rank's flag block
        unsigned int* root_flags = nullptr;     // the root's flag block (== peer_flags[0])
        double* root_stage[2] = {nullptr, nullptr};
        bool sliced = false;            // the root merges all rows (default) / every rank merges its share of the rows
        bool instream = false;          // root form: the root merges its own pieces and the peers' states in ONE kernel of its compute stream
        bool push = false;              // root form: every shard PUSHES its state into the root's inbox (xbuf = world segments), flags are
                                        // pushed too (ready[r] lives on the root, consumed on every rank): nobody reads or polls over NVLink;
                                        // the root's merge is a small-footprint kernel beside the next pass's fused kernel
        bool push_sync = false;         // push form whose final merge runs on the root's COMPUTE stream (full-size kernel, local reads) instead of in the background
        bool auto_form = false;         // default: pushsync for single-batch passes, overlap for passes of several Q batches (chosen per call)
        bool inbox = false;             // the slots are sized (and mapped) as inboxes: any root form may be chosen
        static constexpr int kFlagReady = 768;   // [kFlagReady + slot*64 + r] "shard r's state of the batch is in the root's inbox" (root's copy)
        std::vector<void*> opened;      // IPC mappings to close
        unsigned int epoch = 0;         // global batch counter, identical on every rank
        unsigned int slot_epoch[2] = {0, 0};
        DevBuf trace;                   // SDPA_EXCHANGE_TRACE=<path>: kTraceEpochs x 4 u64 %globaltimer stamps, dumped to <path>.rank<r>
        static constexpr unsigned int kTraceEpochs = 4096, kTraceWords = 12;   // [0] published [1] merge begin [2] all flags seen [3] done [4+r] flag r seen
        unsigned long long* trace_slot(unsigned int e) { return trace.p ? trace.as<unsigned long long>() + (size_t)(e % kTraceEpochs) * kTraceWords : nullptr; }
    } ipc;
    bool has_root() const { return rank_base == 0; }
};

extern "C" { static sdpa_status resolve_pending(sdpa_ctx* ctx); }   // deferred guard repair (defined with the C ABI below)

namespace sdpa {

static sdpa_status new_mark(Shard& s, cudaStream_t st, int* idx)
{
    if (s.marks_used == s.marks.size()) {
        cudaEvent_t e;
        SDPA_CUDA_TRY(cudaEventCreate(&e));
        s.marks.push_back(e);
    }
    SDPA_CUDA_TRY(cudaEventRecord(s.marks[s.marks_used], st));
    *idx = (int)s.marks_used++;
    return SDPA_OK;
}
// Work enqueued on the compute stream outside a timed stage (event waits, flag kernels) must call this:
// the next stage may then not reuse the previous stage's end mark as its begin.
static inline void compute_stream_touched(Shard& s) { s.open_mark = -1; }

// SDPA_STAGE_TIMING=0 (developer knob): no per-stage timestamp events, only the whole-call bracket -- quantifies what the
// stage marks cost inside a queued loop.
static bool stage_timing_enabled()
{
    static const bool on = [] {
        const char* e = getenv("SDPA_STAGE_TIMING");
        return !(e && *e == '0');
    }();
    return on;
}

static sdpa_status time_begin(Shard& s, int which, cudaStream_t st)
{
    if (!s.marks_on || (which != 3 && !stage_timing_enabled())) return SDPA_OK;
    int idx = -1;
    if (st == s.s_compute && s.open_mark >= 0) idx = s.open_mark;
    else SDPA_TRY(new_mark(s, st, &idx));
    if (st == s.s_compute) s.open_mark = idx;   // still nothing behind it until the stage's work is enqueued
    s.tpair[which].push_back(idx);
    return SDPA_OK;
}
static sdpa_status time_end(Shard& s, int which, cudaStream_t st, bool may_share = false)
{
    if (!s.marks_on || (which != 3 && !stage_timing_enabled())) return SDPA_OK;
    int idx = -1;
    if (may_share && st == s.s_compute && s.open_mark >= 0) idx = s.open_mark;   // nothing ran since the last end mark
    else SDPA_TRY(new_mark(s, st, &idx));
    if (st == s.s_compute) s.open_mark = idx;
    s.tpair[which].push_back(idx);
    return SDPA_OK;
}

// Developer aid: SDPA_HOST_PROFILE=1 prints host-side timestamps (us) of one attention call's phases.
static double host_now_us()
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}

// Turn the pending pairs [from, end) of category w into milliseconds (the recorded work must be complete).
static sdpa_status sum_pairs(Shard& s, int w, size_t from, double* out)
{
    double acc = 0.0;
    const std::vector<int>& p = s.tpair[w];
    for (size_t k = from; k + 1 < p.size(); k += 2) {
        float ms = 0.f;
        if (p[k] != p[k + 1]) SDPA_CUDA_TRY(cudaEventElapsedTime(&ms, s.marks[p[k]], s.marks[p[k + 1]]));
        acc += ms;
    }
    *out = acc;
    return SDPA_OK;
}
// Fold everything recorded so far into acc_ms and recycle the marks.
static sdpa_status fold_timings(Shard& s)
{
    SDPA_CUDA_TRY(cudaSetDevice(s.dev));
    SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));   // queued passes (sdpa_enqueue_*) must have finished
    SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_comm));
    for (int w = 0; w < 4; ++w) {
        double ms = 0.0;
        SDPA_TRY(sum_pairs(s, w, 0, &ms));
        s.acc_ms[w] += ms;
        s.tpair[w].clear();
        s.tpair_last[w] = 0;
    }
    s.marks_used = 0;
    s.open_mark = -1;
    return SDPA_OK;
}

// Resident storage per element: fp32 4 B, bf16 2 B, split precision 2 + 2 B (a hi array and, lo_off elements behind it, a lo array).
static size_t elem_size(int prec) { return prec == SDPA_PREC_BF16 ? 2 : 4; }
static size_t unit_size(int prec) { return prec == SDPA_PREC_F32 ? 4 : 2; }   // bytes per element of ONE array
static bool is_umma(int prec) { return prec == SDPA_PREC_BF16 || prec == SDPA_PREC_BF16X3; }
static int prec_hl(int prec) { return prec == SDPA_PREC_BF16X3 ? 2 : 1; }
static const char* kernel_name(int prec, int dk, int dv)
{
    if (prec == SDPA_PREC_BF16X3) return "bf16x3_umma";
    if (prec == SDPA_PREC_BF16) return (dk == 128 && dv == 128) ? "bf16_umma" : "bf16_umma_general";
    return "f32_simt";
}

// Cast `count` fp64 elements into the operand that starts at `dst` (element offset `at`); lo_off: split precision only.
static sdpa_status cast_in(int prec, void* dst, size_t lo_off, size_t at, const double* src, size_t count, cudaStream_t st)
{
    if (prec == SDPA_PREC_BF16X3) {
        __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(dst) + at;
        return launch_cvt_d2bf16x2(hi, hi + lo_off, src, count, st);
    }
    if (prec == SDPA_PREC_BF16) return launch_cvt_d2bf16(reinterpret_cast<__nv_bfloat16*>(dst) + at, src, count, st);
    return launch_cvt_d2f(reinterpret_cast<float*>(dst) + at, src, count, st);
}

// AUTO keeps the reference's accuracy class (fp32, attention-mpi.c:168-189): the split-precision tensor-core kernel where
// the shape allows it, else the fp32 CUDA-core kernel.  Plain bf16 is opt-in only for fp64 and fp32 operands: its operand
// rounding can move peaky scores beyond the reference's own 0.02 acceptance gate (attention-mpi.c:476).  bf16 operands have
// been rounded by the caller already, so for them AUTO is the bf16 kernel, which reads them in place.
static int resolve_precision(int dtype, int requested, int dk, int dv)
{
    if (requested == SDPA_PREC_BF16 || requested == SDPA_PREC_F32 || requested == SDPA_PREC_BF16X3) return requested;
    if (dtype == SDPA_DTYPE_BF16) return attn_umma_supported(dk, dv, 1) ? SDPA_PREC_BF16 : SDPA_PREC_F32;
    return attn_umma_supported(dk, dv, 2) ? SDPA_PREC_BF16X3 : SDPA_PREC_F32;
}
static bool dtype_valid(int dtype) { return dtype == SDPA_DTYPE_F64 || dtype == SDPA_DTYPE_F32 || dtype == SDPA_DTYPE_BF16; }
static size_t dtype_size(int dtype) { return dtype == SDPA_DTYPE_F64 ? 8 : (dtype == SDPA_DTYPE_F32 ? 4 : 2); }
static const char* dtype_name(int dtype) { return dtype == SDPA_DTYPE_F64 ? "fp64" : (dtype == SDPA_DTYPE_F32 ? "fp32" : "bf16"); }
// Operands that already are in compute precision: the fused kernel reads the caller's arrays, no cast kernel runs.
static bool reads_in_place(int dtype, int prec)
{
    return (dtype == SDPA_DTYPE_BF16 && prec == SDPA_PREC_BF16) || (dtype == SDPA_DTYPE_F32 && prec == SDPA_PREC_F32);
}
static sdpa_status check_precision(int prec, int dk, int dv)
{
    if (is_umma(prec) && !attn_umma_supported(dk, dv, prec_hl(prec))) {
        set_error("%s tensor-core kernel: dk and dv must be multiples of 8, %s (got dk=%d dv=%d)",
                  prec == SDPA_PREC_BF16X3 ? "bf16x3" : "bf16",
                  prec == SDPA_PREC_BF16X3 ? "dk <= 128 and dv <= 128, or dk <= 64 and dv <= 256" : "up to 256", dk, dv);
        return SDPA_ERR_UNSUPPORTED;
    }
    if (prec == SDPA_PREC_F32 && !attn_f32_supported(dk, dv)) {
        set_error("fp32 kernel supports 1 <= dk, dv <= 256 (got dk=%d dv=%d)", dk, dv);
        return SDPA_ERR_UNSUPPORTED;
    }
    return SDPA_OK;
}

static sdpa_status shard_init(Shard& s)
{
    SDPA_CUDA_TRY(cudaSetDevice(s.dev));
    SDPA_CUDA_TRY(cudaStreamCreateWithFlags(&s.s_in, cudaStreamNonBlocking));
    SDPA_CUDA_TRY(cudaStreamCreateWithFlags(&s.s_compute, cudaStreamNonBlocking));
    SDPA_CUDA_TRY(cudaStreamCreateWithFlags(&s.s_comm, cudaStreamNonBlocking));
    SDPA_CUDA_TRY(cudaStreamCreateWithFlags(&s.s_out, cudaStreamNonBlocking));
    auto mk = [](cudaEvent_t* e) { return cudaEventCreateWithFlags(e, cudaEventDisableTiming); };
    for (int b = 0; b < 2; ++b) {
        SDPA_CUDA_TRY(mk(&s.ev_stage_ready[b]));
        SDPA_CUDA_TRY(mk(&s.ev_stage_free[b]));
        SDPA_CUDA_TRY(mk(&s.ev_q_ready[b]));
        SDPA_CUDA_TRY(mk(&s.ev_q_free[b]));
        if (getenv("SDPA_PASS_FENCE") && atoi(getenv("SDPA_PASS_FENCE")) == 2) SDPA_CUDA_TRY(cudaEventCreate(&s.ev_compute_done[b]));
        else SDPA_CUDA_TRY(mk(&s.ev_compute_done[b]));
        SDPA_CUDA_TRY(mk(&s.ev_slot_free[b]));
        SDPA_CUDA_TRY(mk(&s.ev_comm_done[b]));
    }
    for (int j = 0; j < 3; ++j) SDPA_CUDA_TRY(mk(&s.ev_join[j]));
    SDPA_CUDA_TRY(cudaStreamCreateWithFlags(&s.s_cast, cudaStreamNonBlocking));
    SDPA_CUDA_TRY(mk(&s.ev_cast_done));
    for (int b = 0; b < 2; ++b) SDPA_CUDA_TRY(mk(&s.ev_kv_read[b]));
    if (mem_pool_enabled()) {   // keep freed blocks in the pool instead of returning them to the driver at every synchronisation
        cudaMemPool_t pool;
        unsigned long long keep = ~0ull;
        if (cudaDeviceGetDefaultMemPool(&pool, s.dev) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        cudaGetLastError();
    }
    int sms = 0;
    SDPA_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s.dev));
    s.sm_count = sms > 0 ? sms : 148;
    return SDPA_OK;
}

static void shard_destroy(Shard& s, const NcclApi* api)
{
    cudaSetDevice(s.dev);
    cudaDeviceSynchronize();
    if (s.comm && api) api->CommDestroy(s.comm);
    if (s.plan) umma_plan_destroy(s.plan);
    DevBuf* bufs[] = {&s.Kc, &s.Vc, &s.KcAlt, &s.VcAlt, &s.kv_stage[0], &s.kv_stage[1], &s.q64[0], &s.q64[1], &s.qc[0], &s.qc[1],
                      &s.part_o, &s.part_tmax, &s.part_lsum, &s.contrib[0], &s.contrib[1], &s.tmax[0],
                      &s.tmax[1], &s.lsum[0], &s.lsum[1], &s.gmax[0], &s.gmax[1], &s.gsum[0], &s.gsum[1],
                      &s.out32[0], &s.out32[1], &s.out64[0], &s.out64[1]};
    for (DevBuf* b : bufs) b->release();
    cudaEvent_t evs[] = {s.ev_stage_ready[0], s.ev_stage_ready[1], s.ev_stage_free[0], s.ev_stage_free[1],
                         s.ev_q_ready[0], s.ev_q_ready[1], s.ev_q_free[0], s.ev_q_free[1],
                         s.ev_compute_done[0], s.ev_compute_done[1], s.ev_slot_free[0], s.ev_slot_free[1],
                         s.ev_comm_done[0], s.ev_comm_done[1],
                         s.ev_join[0], s.ev_join[1], s.ev_join[2], s.ev_cast_done, s.ev_kv_read[0], s.ev_kv_read[1]};
    for (cudaEvent_t e : evs)
        if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s.marks) cudaEventDestroy(e);
    if (s.ev_begin) cudaEventDestroy(s.ev_begin);
    if (s.ev_fence) cudaEventDestroy(s.ev_fence);
    if (s.ev_plain_end) cudaEventDestroy(s.ev_plain_end);
    cudaStream_t sts[] = {s.s_in, s.s_compute, s.s_comm, s.s_out, s.s_cast};
    for (cudaStream_t st : sts)
        if (st) cudaStreamDestroy(st);
}

// K/V chunk size for the fp64 staging buffers (elements).
static const size_t kStageElems = (size_t)4 << 20;  // 32 MiB of fp64 per chunk

// Upload (or read in place) one operand of the shard and cast it into `dst`.
static sdpa_status upload_cast(Shard& s, int prec, void* dst, size_t lo_off, const double* src, size_t count, bool src_on_device)
{
    if (src_on_device) {
        SDPA_TRY(cast_in(prec, dst, lo_off, 0, src, count, s.s_compute));
        return SDPA_OK;
    }
    size_t done = 0;
    int c = 0;
    while (done < count) {
        const size_t len = std::min(kStageElems, count - done);
        const int b = c & 1;
        SDPA_TRY(s.kv_stage[b].reserve(std::min(kStageElems, count) * sizeof(double)));
        SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_in, s.ev_stage_free[b], 0));
        SDPA_TRY(h2d_any(s.kv_stage[b].p, src + done, len * sizeof(double), s.s_in));   // pinned: direct; pageable: staged
        SDPA_CUDA_TRY(cudaEventRecord(s.ev_stage_ready[b], s.s_in));
        SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_compute, s.ev_stage_ready[b], 0));
        SDPA_TRY(cast_in(prec, dst, lo_off, done, s.kv_stage[b].as<double>(), len, s.s_compute));
        SDPA_CUDA_TRY(cudaEventRecord(s.ev_stage_free[b], s.s_compute));
        done += len;
        ++c;
    }
    return SDPA_OK;
}

static sdpa_status load_kv(sdpa_ctx* ctx, int dtype, const void* const* K_shards, const void* const* V_shards,
                           const int* n_local, int dk, int dv, bool on_device, bool defer_casts = false, bool ahead = false)
{
    if (!ctx || !n_local || dk < 1 || dv < 1) {
        set_error("load_kv: bad arguments");
        return SDPA_ERR_INVALID;
    }
    const int prec = resolve_precision(dtype, ctx->cfg.precision, dk, dv);
    SDPA_TRY(check_precision(prec, dk, dv));
    // typed passes (device arrays, deferred casts) whose operands already are in compute precision: no resident copy
    const bool zero_copy = on_device && defer_casts && reads_in_place(dtype, prec);
    ctx->dk = dk;
    ctx->dv = dv;
    ctx->prec = prec;
    ctx->dtype = dtype;
    ctx->zero_copy = zero_copy;
    ctx->qshard = false;   // sdpa_load_kv_host_full sets it again when it replicates
    const size_t esz = elem_size(prec);
    for (size_t i = 0; i < ctx->shards.size(); ++i) {
        Shard& s = ctx->shards[i];
        if (n_local[i] < 0 || (n_local[i] > 0 && (!K_shards || !V_shards || !K_shards[i] || !V_shards[i]))) {
            set_error("load_kv: shard %zu has n_local=%d but a NULL K/V pointer", i, n_local[i]);
            return SDPA_ERR_INVALID;
        }
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        s.n_local = n_local[i];
        s.ahead_call = ahead && defer_casts && on_device && s.n_local > 0;
        if (s.ahead_call) {   // this pass fills (and its kernels read) the other K/V set
            std::swap(s.Kc, s.KcAlt);
            std::swap(s.Vc, s.VcAlt);
            s.kv_set ^= 1;
        }
        s.npend = 0;
        if (zero_copy && s.n_local > 0) {
            // the kernels read the caller's rows; TMA zero-fills the boxes past row n_local, the fp32 kernel masks them
            s.k_in = K_shards[i];
            s.v_in = V_shards[i];
        } else {
            // +128 rows of slack so TMA boxes / vector loads past the last row stay in bounds
            SDPA_TRY(s.Kc.reserve(((size_t)s.n_local + 128) * dk * esz));
            SDPA_TRY(s.Vc.reserve(((size_t)s.n_local + 128) * dv * esz));
            s.k_lo_off = ((size_t)s.n_local + 128) * dk;
            s.v_lo_off = ((size_t)s.n_local + 128) * dv;
            s.k_in = s.Kc.p;
            s.v_in = s.Vc.p;
        }
        if (zero_copy || s.n_local == 0) {
            // nothing to cast
        } else if (on_device && defer_casts) {
            // sdpa_attention_device_full / _typed: the sources stay valid for the whole call, so the casts ride with Q's
            s.pend_dst[0] = s.Kc.p, s.pend_src[0] = K_shards[i], s.pend_cnt[0] = (size_t)s.n_local * dk;
            s.pend_dst[1] = s.Vc.p, s.pend_src[1] = V_shards[i], s.pend_cnt[1] = (size_t)s.n_local * dv;
            s.npend = 2;
        } else {   // fp64 only: sdpa_load_kv_host / sdpa_load_kv_device
            SDPA_TRY(upload_cast(s, prec, s.Kc.p, s.k_lo_off, static_cast<const double*>(K_shards[i]), (size_t)s.n_local * dk, on_device));
            SDPA_TRY(upload_cast(s, prec, s.Vc.p, s.v_lo_off, static_cast<const double*>(V_shards[i]), (size_t)s.n_local * dv, on_device));
        }
        if (is_umma(prec)) {
            if (!s.plan) SDPA_TRY(umma_plan_create(&s.plan));
            SDPA_TRY(umma_plan_bind_kv(s.plan, static_cast<const __nv_bfloat16*>(s.k_in), static_cast<const __nv_bfloat16*>(s.v_in),
                                       s.n_local, dk, dv, prec_hl(prec), s.k_lo_off, s.v_lo_off));
        }
    }
    // Host sources: block until the uploads have been consumed (the caller may reuse its arrays).
    // Device sources: stream-ordered -- the casts are queued on the compute stream that the next
    // sdpa_attention_* call uses, so no host round trip is spent here (see include/sdpa_b200.h).
    if (!on_device)
        for (Shard& s : ctx->shards) {
            SDPA_CUDA_TRY(cudaSetDevice(s.dev));
            SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));
        }
    return SDPA_OK;
}

// Cast-ahead needs the end of a pass to be visible to the side stream AT ONCE: behind an event without a timestamp the cast of
// pass i+2 was seen to start only when the fused kernel of pass i+1 had finished (239 us per c3 step instead of 216;
// profiles/r02/visit17_*).  A timing-enabled event record at the end of the pass (what the stage marks do on a marked pass)
// restores the overlap.  SDPA_PASS_FENCE=0: off; 1 (default): one extra timing event per cast-ahead batch; 2: the gate event
// itself carries the timestamp.
static int pass_fence()
{
    static const int mode = [] {
        const char* e = getenv("SDPA_PASS_FENCE");
        return e ? atoi(e) : 1;
    }();
    return mode;
}
static int pick_q_batch(const sdpa_ctx* ctx, int m);
// Pieces per row block when the persistent fused kernel takes the pass (dk = dv = 128 bf16, automatic splits, every shard the
// same number of keys, enough work per SM pair), else 0.
static int persistent_pieces(const sdpa_ctx* ctx, int prec, int dk, int dv, int B, const int* n_local)
{
    if (prec != SDPA_PREC_BF16 || dk != 128 || dv != 128 || ctx->cfg.kv_splits > 0) return 0;
    for (size_t i = 1; i < ctx->shards.size(); ++i)
        if (n_local[i] != n_local[0]) return 0;
    const int pieces = attn_umma_v8_pieces(B, n_local[0], ctx->shards[0].sm_count);
    return pieces > 1 ? pieces : 0;
}

static int pick_q_batch(const sdpa_ctx* ctx, int m)
{
    int B = ctx->cfg.q_batch;
    if (B <= 0) {
        // Engine default: the reference's B=512 (mpi.c:200) is sized for MPI latency on CPUs.
        // On NVLink the per-batch exchange is ~tens of microseconds, so batches are made as large
        // as the buffers allow (8192 rows); the ping-pong overlap matters once m exceeds one batch (c4, c5).
        B = 8192;
        // (Measured on 2 GPUs: halving the batch to overlap the exchange with the next kernel does not pay --
        // the fused kernel holds every SM, so the NCCL kernels queue behind it anyway, and two half-size
        // launches lose more in the tail than the overlap wins.  m > 8192 still ping-pongs, as c4/c5 do.)
    }
    if (B > m) B = m;
    if (B < 1) B = 1;
    return B;
}

static sdpa_status reserve_batch_buffers(sdpa_ctx* ctx, Shard& s, int B, int splits, bool root)
{
    const size_t esz = elem_size(ctx->prec);
    const int dk = ctx->dk, dv = ctx->dv;
    const int Bpad = (B + 127) & ~127;
    for (int b = 0; b < 2; ++b) {
        SDPA_TRY(s.q64[b].reserve((size_t)B * dk * sizeof(double)));
        SDPA_TRY(s.qc[b].reserve((size_t)(Bpad + 128) * dk * esz));
        SDPA_TRY(s.contrib[b].reserve(((size_t)B * dv + B) * sizeof(float)));   // + lsum tail for the 2-collective merge
        SDPA_TRY(s.tmax[b].reserve((size_t)B * sizeof(float)));
        SDPA_TRY(s.lsum[b].reserve((size_t)B * sizeof(float)));
        SDPA_TRY(s.gmax[b].reserve((size_t)B * sizeof(float)));
        SDPA_TRY(s.gsum[b].reserve((size_t)B * sizeof(float)));
        if (root) {
            SDPA_TRY(s.out32[b].reserve(((size_t)B * dv + B) * sizeof(float)));
            SDPA_TRY(s.out64[b].reserve((size_t)B * dv * sizeof(double)));
        }
    }
    SDPA_TRY(s.part_o.reserve((size_t)splits * B * dv * sizeof(float)));
    SDPA_TRY(s.part_tmax.reserve((size_t)splits * B * sizeof(float)));
    SDPA_TRY(s.part_lsum.reserve((size_t)splits * B * sizeof(float)));
    return SDPA_OK;
}

// The fused kernel for one batch on one shard: fills the split partials, or writes fp64 directly.  q_f32: the fp32 Q rows of
// the batch (the fp32 kernel; the tensor-core kernels read Q through the plan's map of the slot).
static sdpa_status run_fused(sdpa_ctx* ctx, Shard& s, int slot, const float* q_f32, int rows, int splits, Partials part, double* direct_out)
{
    if (is_umma(ctx->prec)) {
        return launch_attn_umma(s.plan, slot, rows, splits, part, direct_out, s.sm_count, s.s_compute);
    }
    return launch_attn_f32(q_f32, static_cast<const float*>(s.k_in), static_cast<const float*>(s.v_in), rows, s.n_local, ctx->dk,
                           ctx->dv, splits, part, direct_out, s.s_compute);
}

// ---------------------------------------------------------------------------
// Device-side exchange for one process per GPU: every rank exports its per-slot state buffer and flag
// block with cudaIpcGetMemHandle; the handles are all-gathered over the (already bootstrapped) NCCL
// communicator; the root maps everybody's buffers, the others map the root's flags.  After this no
// collective runs on the data path: shards publish an epoch flag, the root's merge kernel polls the
// flags and reads the states over NVLink, and publishes "consumed" for buffer reuse.
// ---------------------------------------------------------------------------
static void ipc_close(sdpa_ctx* ctx)
{
    for (void* p : ctx->ipc.opened) cudaIpcCloseMemHandle(p);
    ctx->ipc.opened.clear();
    ctx->ipc.peer_x[0].clear();
    ctx->ipc.peer_x[1].clear();
    ctx->ipc.peer_flags.clear();
    ctx->ipc.root_flags = nullptr;
    ctx->ipc.root_stage[0] = ctx->ipc.root_stage[1] = nullptr;
    ctx->ipc.ready = false;
}

// Overlap mode: wait until the root has consumed every slot this rank published and all streams are idle.
static sdpa_status drain_exchange(sdpa_ctx* ctx)
{
    if (!ctx->exchange_pending) return SDPA_OK;
    for (Shard& s : ctx->shards) {
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        if (ctx->ipc.ready && s.grank != 0) {
            for (int b = 0; b < 2; ++b)
                if (ctx->ipc.slot_epoch[b] != 0)
                    SDPA_TRY(launch_wait_flag(ctx->ipc.root_flags + 2 + b, ctx->ipc.slot_epoch[b], s.s_compute));
            compute_stream_touched(s);
        }
        SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));
        SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_comm));
        SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_out));
    }
    ctx->exchange_pending = false;
    return SDPA_OK;
}

static bool ipc_sliced_requested()
{
    const char* mode = getenv("SDPA_IPC_MERGE");
    return mode && !strcmp(mode, "sliced");
}

static sdpa_status ipc_setup(sdpa_ctx* ctx, int rows_cap, int dv)
{
    sdpa_ctx::Ipc& x = ctx->ipc;
    if (x.ready && x.cap_rows >= rows_cap && x.dv == dv) return SDPA_OK;
    const NcclApi* api = nccl_api();
    if (!api) return SDPA_ERR_NCCL;
    SDPA_TRY(drain_exchange(ctx));
    Shard& s = ctx->shards[0];
    SDPA_CUDA_TRY(cudaSetDevice(s.dev));
    SDPA_CUDA_TRY(cudaDeviceSynchronize());
    ipc_close(ctx);
    // every rank re-allocates together (the decision depends only on arguments all ranks share)
    // root merge: [o rows*dv | tmax rows | lsum rows]; sliced merge: one inbox segment per source rank,
    // [o slice*dv | tmax slice | lsum slice] each, slice = rows of one rank's share (rounded up to a multiple of 4)
    if (!x.flags.p) {
        // "root" (default): the root GPU merges every row; "sliced": every rank merges its share of the rows from an inbox the
        // others push into.  Root forms (SDPA_ROOT_MERGE): overlap = comm-stream merge reading the states over NVLink,
        // instream = one merge on the root's compute stream, push = states pushed into the root's inbox + background merge.
        x.sliced = ipc_sliced_requested();
        const char* rm = getenv("SDPA_ROOT_MERGE");   // push | instream | overlap
        const char* form = rm ? rm : kRootMergeDefault;
        x.instream = !x.sliced && !strcmp(form, "instream");
        x.push = !x.sliced && (!strcmp(form, "push") || !strcmp(form, "pushsync"));
        x.push_sync = x.push && !strcmp(form, "pushsync");
        x.auto_form = !x.sliced && !strcmp(form, "auto");
        x.inbox = x.push || x.auto_form;
    }
    const int slice_cap = ((rows_cap + ctx->world - 1) / ctx->world + 3) & ~3;
    const size_t state_floats = (size_t)rows_cap * dv + 2 * (size_t)rows_cap;
    const size_t xbytes = std::max(x.inbox ? (size_t)ctx->world * state_floats : state_floats,
                                   (size_t)ctx->world * slice_cap * ((size_t)dv + 2)) * sizeof(float);
    x.slice_cap = slice_cap;
    for (int b = 0; b < 2; ++b) {
        x.xbuf[b].release();
        SDPA_TRY(x.xbuf[b].reserve(xbytes, true));
    }
    for (int b = 0; b < 2; ++b) {
        x.stage[b].release();
        SDPA_TRY(x.stage[b].reserve((size_t)rows_cap * dv * sizeof(double), true));
    }
    if (!x.flags.p) {
        SDPA_TRY(x.flags.reserve(4096, true));
        SDPA_CUDA_TRY(cudaMemset(x.flags.p, 0, 4096));
        if (const char* ts = getenv("SDPA_FLAG_TIMEOUT_S"); ts && atof(ts) > 0.0) SDPA_TRY(set_flag_timeout_seconds(atof(ts)));
        if (const char* tp = getenv("SDPA_EXCHANGE_TRACE"); tp && *tp) {
            SDPA_TRY(x.trace.reserve((size_t)sdpa_ctx::Ipc::kTraceEpochs * sdpa_ctx::Ipc::kTraceWords * sizeof(unsigned long long)));
            SDPA_CUDA_TRY(cudaMemset(x.trace.p, 0, x.trace.bytes));
        }
        x.epoch = 0;
        x.slot_epoch[0] = x.slot_epoch[1] = 0;
    }
    struct Handles { cudaIpcMemHandle_t x0, x1, fl, s0, s1; };
    Handles mine;
    SDPA_CUDA_TRY(cudaIpcGetMemHandle(&mine.x0, x.xbuf[0].p));
    SDPA_CUDA_TRY(cudaIpcGetMemHandle(&mine.x1, x.xbuf[1].p));
    SDPA_CUDA_TRY(cudaIpcGetMemHandle(&mine.fl, x.flags.p));
    SDPA_CUDA_TRY(cudaIpcGetMemHandle(&mine.s0, x.stage[0].p));
    SDPA_CUDA_TRY(cudaIpcGetMemHandle(&mine.s1, x.stage[1].p));
    const int world = ctx->world;
    DevBuf dsend, drecv;
    SDPA_TRY(dsend.reserve(sizeof(Handles)));
    SDPA_TRY(drecv.reserve(sizeof(Handles) * world));
    SDPA_CUDA_TRY(cudaMemcpyAsync(dsend.p, &mine, sizeof(Handles), cudaMemcpyHostToDevice, s.s_comm));
    SDPA_NCCL_TRY(api->AllGather(dsend.p, drecv.p, sizeof(Handles), ncclUint8, s.comm, s.s_comm));
    std::vector<Handles> all(world);
    SDPA_CUDA_TRY(cudaMemcpyAsync(all.data(), drecv.p, sizeof(Handles) * world, cudaMemcpyDeviceToHost, s.s_comm));
    SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_comm));
    dsend.release();
    drecv.release();
    auto open = [&](const cudaIpcMemHandle_t& h, void** out) -> sdpa_status {
        SDPA_CUDA_TRY(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
        x.opened.push_back(*out);
        return SDPA_OK;
    };
    // every rank maps every other rank's state slots and flags (sliced merge: all-to-all reads), and the root's staging
    x.peer_x[0].assign(world, nullptr);
    x.peer_x[1].assign(world, nullptr);
    x.peer_flags.assign(world, nullptr);
    for (int r = 0; r < world; ++r) {
        if (r == s.grank) {
            x.peer_x[0][r] = x.xbuf[0].p;
            x.peer_x[1][r] = x.xbuf[1].p;
            x.peer_flags[r] = x.flags.as<unsigned int>();
            continue;
        }
        if (s.grank != 0 && r != 0 && !x.sliced) continue;   // root merge: non-root ranks only need the root's flags
        void* p = nullptr;
        if (s.grank == 0 || x.sliced || (x.inbox && r == 0)) {
            SDPA_TRY(open(all[r].x0, &p));
            x.peer_x[0][r] = p;
            SDPA_TRY(open(all[r].x1, &p));
            x.peer_x[1][r] = p;
        }
        SDPA_TRY(open(all[r].fl, &p));
        x.peer_flags[r] = reinterpret_cast<unsigned int*>(p);
    }
    x.root_flags = x.peer_flags[0];
    if (s.grank == 0) {
        x.root_stage[0] = x.stage[0].as<double>();
        x.root_stage[1] = x.stage[1].as<double>();
    } else if (x.sliced) {
        void* p = nullptr;
        SDPA_TRY(open(all[0].s0, &p));
        x.root_stage[0] = reinterpret_cast<double*>(p);
        SDPA_TRY(open(all[0].s1, &p));
        x.root_stage[1] = reinterpret_cast<double*>(p);
    }
    x.cap_rows = rows_cap;
    x.dv = dv;
    x.ready = true;
    return SDPA_OK;
}

// Q_dev / result: element type `dtype` (device arrays; host arrays are fp64).  A typed result is merged into the root's fp64
// batch slot and rounded from there into the caller's array.
static sdpa_status attention_impl(sdpa_ctx* ctx, const double* Q_host, const void* const* Q_dev,
                                  void* result, bool result_on_device, int m, bool q_from_root = false,
                                  bool blocking = true, int dtype = SDPA_DTYPE_F64)
{
    if (!ctx || m < 0) {
        set_error("attention: bad arguments");
        return SDPA_ERR_INVALID;
    }
    if (ctx->dk == 0) {
        set_error("attention: no K/V shard loaded (call sdpa_load_kv_* first)");
        return SDPA_ERR_INVALID;
    }
    if (dtype != ctx->dtype) {
        set_error("attention: the K/V shard was loaded for %s operands, this call passes %s arrays", dtype_name(ctx->dtype), dtype_name(dtype));
        return SDPA_ERR_INVALID;
    }
    const bool on_device = Q_dev != nullptr;
    if (m > 0 && !on_device && !Q_host && !(q_from_root && !ctx->has_root())) {
        set_error("attention: Q is NULL");
        return SDPA_ERR_INVALID;
    }
    if (m > 0 && ctx->has_root() && !result) {
        set_error("attention: result is NULL on the process that owns shard 0");
        return SDPA_ERR_INVALID;
    }
    const int dk = ctx->dk, dv = ctx->dv;
    const int world = ctx->world;
    const int L = (int)ctx->shards.size();
    const NcclApi* api = nullptr;
    const bool use_peer = world > 1 && ctx->cfg.merge == SDPA_MERGE_PEER && ctx->peer_ok && world == L;
    const bool use_ipc = world > 1 && ctx->cfg.merge == SDPA_MERGE_PEER && L == 1 && world > L;   // one GPU per process
    const bool overlap = !blocking && use_ipc && ctx->overlap_passes && Q_dev != nullptr && result_on_device;
    const bool two_coll = ctx->cfg.merge != SDPA_MERGE_NCCL;   // NCCL2 (default) unless the reference's 3-collective form is asked for
    if ((world > 1 && !use_peer && !use_ipc) || q_from_root) {
        api = nccl_api();
        if (!api) return SDPA_ERR_NCCL;
    }
    ctx->last_kernel = kernel_name(ctx->prec, dk, dv);
    for (float& t : ctx->last_timing) t = 0.f;
    if (m == 0) {
        ctx->last_timing_valid = true;   // nothing ran: all-zero stage times
        for (Shard& s : ctx->shards) {   // K/V casts deferred by sdpa_attention_device_full still have to happen
            if (s.npend == 0) continue;
            SDPA_CUDA_TRY(cudaSetDevice(s.dev));
            const size_t lo[2] = {s.k_lo_off, s.v_lo_off};
            SDPA_TRY(launch_cvt_in_batch(ctx->dtype, ctx->prec, s.pend_dst, s.pend_src, s.pend_cnt, lo, 2, s.s_compute));
            s.npend = 0;
            s.ahead_call = false;
            s.kv_guard[s.kv_set] = nullptr;
        }
        return SDPA_OK;
    }

    static const bool host_prof = getenv("SDPA_HOST_PROFILE") != nullptr;
    const double hp0 = host_prof ? host_now_us() : 0.0;
    const int B = pick_q_batch(ctx, m);
    const int num_iter = ceil_div(m, B);

    // split-KV factor (same on every shard so the partial buffers match)
    int splits = ctx->cfg.kv_splits;
    if (splits <= 0) {
        int nmax = 0;
        for (Shard& s : ctx->shards) nmax = std::max(nmax, s.n_local);
        splits = is_umma(ctx->prec) ? attn_umma_pick_splits(B, nmax, ctx->shards[0].sm_count)
                                    : attn_f32_pick_splits(B, nmax, ctx->shards[0].sm_count);
    }
    splits = std::max(1, std::min(splits, 64));
    // The persistent fused kernel (dk = dv = 128 bf16, enough work per SM pair) cuts every row block into pieces; its piece
    // count replaces the split count and the split merge reads pieces per row block (launch_merge_pieces).  Every shard must
    // own the same number of keys (the partial buffers and the piece count are shared).
    bool by_pieces = false;
    {
        std::vector<int> nl;
        for (Shard& s : ctx->shards) nl.push_back(s.n_local);
        const int pieces = persistent_pieces(ctx, ctx->prec, dk, dv, B, nl.data());
        if (pieces > 1) {
            splits = pieces;
            by_pieces = true;
        }
    }
    // cast-ahead pass (decided by sdpa_enqueue_device_full): the first cast runs on the side stream; Q slots follow the batch sequence
    bool ahead = false;
    for (Shard& s : ctx->shards) ahead = ahead || s.ahead_call;
    const bool seq_slots = overlap || ahead;
    if (is_umma(ctx->prec))
        for (Shard& s : ctx->shards)
            if (s.plan) umma_plan_allow_v8(s.plan, by_pieces);

    // guard twin: in the stream behind every fast tensor-core launch, except for queued passes of a single-GPU context
    if (!ctx->repairing && !ctx->pending.empty() && ctx->ring_use + (unsigned int)num_iter + 8 >= kGuardRing)
        SDPA_TRY(resolve_pending(ctx));   // the guard words of the pending passes must not be reused before they are read
    ctx->ring_use += (unsigned int)num_iter;
    ctx->deferring = ctx->defer_twin && (world == 1 || ctx->defer_multi) && !blocking && !ctx->repairing && is_umma(ctx->prec) && on_device &&
                     (result_on_device || !ctx->has_root());
    ctx->call_guards.clear();
    // stage marks: every blocking call; queued passes on every mark_every-th pass (each timestamp event costs ~2 us of stream time)
    const bool marked = blocking || ctx->mark_every <= 1 || (ctx->queued_seq++ % (unsigned long long)ctx->mark_every) == 0;
    // which side streams this call touches (the others are neither forked nor joined: every stream operation
    // between two kernels costs front-end time on the GPU)
    const bool use_in = !on_device;                                  // H2D of the Q batches
    const bool use_comm = world > 1;                                 // collectives / peer merge
    const bool use_out = world > 1 || !result_on_device;             // D2H of the result, slot recycling
    // where the merged fp64 rows go: straight into an fp64 device result, else the root's batch slot out64[b] (then D2H, or
    // rounded into the typed result)
    const bool direct = result_on_device && dtype == SDPA_DTYPE_F64;
    double* const res64 = static_cast<double*>(result);
    for (int i = 0; i < L; ++i) {
        Shard& s = ctx->shards[i];
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        SDPA_TRY(reserve_batch_buffers(ctx, s, B, splits, s.grank == 0));
        if (s.marks_used > 2048) {   // long unmeasured loops: keep the pool bounded
            ctx->last_timing_valid = true;   // the last call's detail is dropped with the fold
            SDPA_TRY(fold_timings(s));
        }
        for (int w = 0; w < 4; ++w) s.tpair_last[w] = s.tpair[w].size();
        // Whatever ran before this call is not part of it -- except when both this and the previous call are queued passes:
        // nothing separates them on the compute stream, so the previous end mark IS this call's begin mark (one event less).
        if (!(s.last_call_queued && !blocking && s.marks_on && marked)) compute_stream_touched(s);
        s.marks_on = marked;
        s.q_lo_off = (size_t)(((B + 127) & ~127) + 128) * dk;
        if (is_umma(ctx->prec) && dtype == SDPA_DTYPE_F64)   // typed passes bind their Q rows batch by batch (below)
            for (int b = 0; b < 2; ++b)
                SDPA_TRY(umma_plan_bind_q(s.plan, b, s.qc[b].as<__nv_bfloat16>(), (B + 127) & ~127, dk, prec_hl(ctx->prec), s.q_lo_off));
        SDPA_TRY(time_begin(s, 3, s.s_compute));
        // the side streams this call uses start after the begin mark, so that "total" brackets everything
        if (use_in || use_comm || use_out) {
            cudaEvent_t begun = nullptr;
            if (marked) begun = s.marks[s.tpair[3].back()];
            else {
                if (!s.ev_begin) SDPA_CUDA_TRY(cudaEventCreateWithFlags(&s.ev_begin, cudaEventDisableTiming));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_begin, s.s_compute));
                begun = s.ev_begin;
            }
            if (use_in) SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_in, begun, 0));
            if (use_comm) SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_comm, begun, 0));
            if (use_out) SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_out, begun, 0));
        }
    }

    if (use_ipc) {
        SDPA_TRY(ipc_setup(ctx, std::max(B, 8192), dv));
        if (ctx->ipc.auto_form) {
            // The forms share slots, epochs and the "consumed" flag, and the other shards cannot tell `instream` from `overlap`.
            // Single-batch passes: two GPUs -> instream (257 us per c3 step against 269 for pushsync), more -> pushsync (265 us at
            // four GPUs against 312); passes of several Q batches -> overlap.
            const bool single_batch = num_iter == 1;
            ctx->ipc.instream = single_batch && world == 2;
            ctx->ipc.push = ctx->ipc.push_sync = single_batch && world > 2;
        }
    }

    int fused_launches = 0, all_launches = 0;
    const unsigned long long launches_before = launch_count();

    for (int ii = 0; ii < num_iter; ++ii) {
        const int row0 = ii * B;
        const int bs = std::min(B, m - row0);
        const int b = seq_slots ? (int)(ctx->batch_seq & 1) : (ii & 1);

        // ---- per shard: Q batch in, cast, fused kernel, split merge -------------------------
        for (int i = 0; i < L; ++i) {
            Shard& s = ctx->shards[i];
            SDPA_CUDA_TRY(cudaSetDevice(s.dev));
            const bool single = (world == 1);
            const void* q_src_dev = nullptr;   // element type `dtype`
            const bool have_q = !q_from_root || s.grank == 0;  // q_from_root: only shard 0's process holds Q
            if (on_device) {
                q_src_dev = static_cast<const char*>(Q_dev[i]) + (size_t)row0 * dk * dtype_size(dtype);
            } else if (have_q) {
                // copy stream: wait until the cast of batch ii-2 released this buffer
                if (ii >= 2) SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_in, s.ev_q_free[b], 0));
                SDPA_TRY(h2d_any(s.q64[b].p, Q_host + (size_t)row0 * dk, (size_t)bs * dk * sizeof(double), s.s_in));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_q_ready[b], s.s_in));
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_compute, s.ev_q_ready[b], 0));
                compute_stream_touched(s);
                q_src_dev = s.q64[b].as<double>();
            }
            // slot b (contrib/out buffers) must have been drained by batch ii-2's collectives / D2H
            if ((seq_slots ? ctx->batch_seq >= 2 : ii >= 2) && use_out) {
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_compute, s.ev_slot_free[b], 0));
                compute_stream_touched(s);
            }

            // cast-ahead: K, V and the first Q batch of this pass are cast on the side stream by the small-footprint kernel --
            // gated by the last readers of the K/V set (two passes back) and of the Q slot (two batches back), not by the pass
            // in front, whose fused kernel it runs beside
            const bool cast_aside = s.ahead_call && s.npend > 0;
            cudaStream_t cst = cast_aside ? s.s_cast : s.s_compute;
            if (cast_aside) {
                if (s.kv_guard[s.kv_set]) SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_cast, s.kv_guard[s.kv_set], 0));
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_cast, s.ev_compute_done[b], 0));
                if (s.plain_end_recorded) SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_cast, s.ev_plain_end, 0));
                s.ahead_ever = true;
            }
            // Typed passes: the tensor-core kernels get a map of exactly this batch's Q rows -- the caller's (zero copy: no cast
            // stage at all) or the slot's -- so the rows of a 256-row block past the batch are zero-filled by TMA and never
            // stale slot contents (which the overflow guard would look at too).  Zero copy on the fp32 kernel: Q read in place.
            if (dtype != SDPA_DTYPE_F64 && is_umma(ctx->prec))
                SDPA_TRY(umma_plan_bind_q(s.plan, b, ctx->zero_copy ? static_cast<const __nv_bfloat16*>(q_src_dev) : s.qc[b].as<__nv_bfloat16>(),
                                          bs, dk, prec_hl(ctx->prec), s.q_lo_off));
            if (!ctx->zero_copy) SDPA_TRY(time_begin(s, 0, cst));
            if (ctx->zero_copy) {
                // nothing to cast
            } else if (s.npend > 0) {
                void* cd[3] = {s.pend_dst[0], s.pend_dst[1], s.qc[b].p};
                const void* cs[3] = {s.pend_src[0], s.pend_src[1], q_src_dev};
                const size_t cc[3] = {s.pend_cnt[0], s.pend_cnt[1], (size_t)bs * dk};
                const size_t lo[3] = {s.k_lo_off, s.v_lo_off, s.q_lo_off};
                SDPA_TRY(launch_cvt_in_batch(dtype, ctx->prec, cd, cs, cc, lo, have_q ? 3 : 2, cst, cast_aside ? s.sm_count : 0));
                s.npend = 0;
                ++all_launches;
            } else if (have_q && dtype != SDPA_DTYPE_F64) {
                void* cd[1] = {s.qc[b].p};
                const size_t cc[1] = {(size_t)bs * dk}, lo[1] = {s.q_lo_off};
                SDPA_TRY(launch_cvt_in_batch(dtype, ctx->prec, cd, &q_src_dev, cc, lo, 1, s.s_compute));
                ++all_launches;
            } else if (have_q) {
                SDPA_TRY(cast_in(ctx->prec, s.qc[b].p, s.q_lo_off, 0, static_cast<const double*>(q_src_dev), (size_t)bs * dk, s.s_compute));
                ++all_launches;
            }
            if (q_from_root) {  // the Q batch travels in compute precision (mpi.c:305,327: Ibcast of the fp32 batch)
                SDPA_NCCL_TRY(api->Broadcast(s.qc[b].p, s.qc[b].p, (size_t)bs * dk * unit_size(ctx->prec), ncclUint8, 0,
                                             s.comm, s.s_compute));
                if (ctx->prec == SDPA_PREC_BF16X3) {   // ... and the lo half of the split operand
                    void* lo = s.qc[b].as<__nv_bfloat16>() + s.q_lo_off;
                    SDPA_NCCL_TRY(api->Broadcast(lo, lo, (size_t)bs * dk * 2, ncclUint8, 0, s.comm, s.s_compute));
                }
            }
            if (!ctx->zero_copy) SDPA_TRY(time_end(s, 0, cst));
            if (cast_aside) {
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_cast_done, s.s_cast));
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_compute, s.ev_cast_done, 0));
                compute_stream_touched(s);
            }
            if (!on_device && have_q) SDPA_CUDA_TRY(cudaEventRecord(s.ev_q_free[b], s.s_compute));

            Partials part{s.part_o.as<float>(), s.part_tmax.as<float>(), s.part_lsum.as<float>(), splits, B};
            double* final_dst = nullptr;  // where the fp64 rows of this batch go when no cross-GPU merge is needed
            if (single) final_dst = direct ? res64 + (size_t)row0 * dv : s.out64[b].as<double>();

            SDPA_TRY(time_begin(s, 1, s.s_compute));
            if (ctx->cast_trace.p) SDPA_TRY(launch_stamp(ctx->cast_trace.as<unsigned long long>() + 600 + 2 * (ctx->trace_pass & 1), s.s_compute));
            const float* q_f32 = ctx->zero_copy ? static_cast<const float*>(q_src_dev) : s.qc[b].as<float>();
            SDPA_TRY(run_fused(ctx, s, b, q_f32, bs, splits, part, (single && splits == 1) ? final_dst : nullptr));
            if (ctx->cast_trace.p) SDPA_TRY(launch_stamp(ctx->cast_trace.as<unsigned long long>() + 601 + 2 * (ctx->trace_pass++ & 1), s.s_compute));
            SDPA_TRY(time_end(s, 1, s.s_compute));
            ++fused_launches;
            ++all_launches;
            // the guard twin of a tensor-core launch belongs to the merge stage ("guard twin + split merge"): the fused stage is
            // the duration of the fused kernel alone
            const bool twin = is_umma(ctx->prec) && !ctx->deferring;
            if (ctx->deferring) {
                unsigned int slot = 0, ep = 0;
                umma_plan_last_guard(s.plan, &slot, &ep);
                ctx->call_guards.push_back({i, slot, ep});
            }
            if (twin && single && splits == 1)
                SDPA_TRY(launch_attn_umma_twin(s.plan, b, bs, splits, part, final_dst, s.s_compute));

            if (!(single && splits == 1)) {
                SDPA_TRY(time_begin(s, 2, s.s_compute));
                if (twin) SDPA_TRY(launch_attn_umma_twin(s.plan, b, bs, splits, part, nullptr, s.s_compute));
                WorkMap wm;
                int max_pieces = 0;
                const unsigned int* guard = nullptr;
                unsigned int guard_epoch = 0;
                const bool pieces = by_pieces && umma_plan_last_v8(s.plan, &wm, &max_pieces, &guard, &guard_epoch);
                if (pieces) ctx->last_kernel = "bf16_umma_v8";
                // the shard's own partial states -> one state: normalised fp64 rows (single GPU) or (contrib, tmax, lsum)
                auto merge_local = [&](double* out64, float* c, float* t, float* l, const PublishSync* pub = nullptr) -> sdpa_status {
                    if (pieces) return launch_merge_pieces(part, wm, max_pieces, bs, dv, out64, c, t, l, guard, guard_epoch, s.s_compute, pub);
                    return launch_merge_splits(part, bs, dv, out64, c, t, l, false, s.s_compute, pub);
                };
                if (single) {
                    SDPA_TRY(merge_local(final_dst, nullptr, nullptr, nullptr));
                } else {
                    if (use_ipc) {
                        // publish this shard's state in its IPC-shared slot, then raise the epoch flag
                        sdpa_ctx::Ipc& x = ctx->ipc;
                        float* xc = x.xbuf[b].as<float>();
                        float* xt = xc + (size_t)x.cap_rows * dv;
                        float* xl = xt + x.cap_rows;
                        if (i == 0) ++x.epoch;
                        if (x.sliced && s.grank != 0 && x.slot_epoch[b] != 0)   // the root must have consumed the slot's previous content
                            SDPA_TRY(launch_wait_flag(x.root_flags + 2 + b, x.slot_epoch[b], s.s_compute));
                        if (x.sliced) {
                            // push: every row's merged state goes straight into the inbox of the rank that owns its slice
                            RouteTargets to;
                            const size_t seg = (size_t)x.slice_cap * ((size_t)dv + 2);
                            for (int r = 0; r < world; ++r) {
                                float* in = reinterpret_cast<float*>(x.peer_x[b][r]) + (size_t)s.grank * seg;
                                to.o[r] = in;
                                to.tmax[r] = in + (size_t)x.slice_cap * dv;
                                to.lsum[r] = to.tmax[r] + x.slice_cap;
                                to.flag[r] = x.peer_flags[r] + sdpa_ctx::Ipc::kFlagDelivered + b * 64 + s.grank;
                            }
                            to.block_counter = x.flags.as<unsigned int>() + 10 + b;
                            to.epoch = x.epoch;
                            to.world = world;
                            SDPA_TRY(launch_merge_splits_routed(part, bs, dv, to, s.s_compute, pieces ? &wm : nullptr, max_pieces, guard, guard_epoch));
                        } else if (x.instream && s.grank == 0) {
                            // the root: its own partial states and every other shard's published state in ONE merge, right here in
                            // the compute stream (no state of its own to publish, no second merge on the comm stream)
                            const float* cp[64];
                            const float* tp[64];
                            const float* lp[64];
                            PeerSync sync;
                            for (int r = 1; r < world; ++r) {
                                const float* base = reinterpret_cast<const float*>(x.peer_x[b][r]);
                                cp[r - 1] = base;
                                tp[r - 1] = base + (size_t)x.cap_rows * dv;
                                lp[r - 1] = tp[r - 1] + x.cap_rows;
                                sync.ready[r - 1] = x.peer_flags[r] + b;
                            }
                            sync.consumed = x.flags.as<unsigned int>() + 2 + b;
                            sync.block_counter = x.flags.as<unsigned int>() + 4 + b;
                            sync.epoch = x.epoch;
                            sync.trace = x.trace_slot(x.epoch);
                            double* dst = direct ? res64 + (size_t)row0 * dv : s.out64[b].as<double>();
                            SDPA_TRY(launch_merge_root_instream(part, pieces ? &wm : nullptr, max_pieces, guard, guard_epoch, cp, tp, lp, world - 1, bs,
                                                                dv, dst, sync, s.s_compute));
                        } else if (x.push) {
                            // one launch: wait until the root's merge has handed the slot back (consumed, pushed into THIS rank's
                            // flag block), merge the shard's partial states straight into segment grank of the root's inbox
                            // (posted stores over NVLink; local on the root), raise ready[grank] on the root
                            const size_t seg = (size_t)x.cap_rows * ((size_t)dv + 2);
                            float* ic = reinterpret_cast<float*>(x.peer_x[b][0]) + (size_t)s.grank * seg;
                            float* it = ic + (size_t)x.cap_rows * dv;
                            float* il = it + x.cap_rows;
                            PublishSync pub;
                            if (x.slot_epoch[b] != 0 && !(x.push_sync && s.grank == 0)) {
                                // background form: `consumed` is pushed into every rank's own flag block; in-stream form: the root's
                                // final merge releases its own copy only (its own publish is ordered behind it by the stream)
                                pub.wait_flag = (x.push_sync ? x.root_flags : x.flags.as<unsigned int>()) + 2 + b;
                                pub.wait_epoch = x.slot_epoch[b];
                            }
                            pub.flag = x.root_flags + sdpa_ctx::Ipc::kFlagReady + b * 64 + s.grank;
                            pub.epoch = x.epoch;
                            pub.block_counter = x.flags.as<unsigned int>() + 12 + b;
                            pub.trace = x.trace_slot(x.epoch);
                            SDPA_TRY(merge_local(nullptr, ic, it, il, &pub));
                        } else {
                            // one launch: wait for the root's "consumed" flag of this slot, merge the shard's partial states
                            // into the slot, publish the epoch flag
                            PublishSync pub;
                            if (s.grank != 0 && x.slot_epoch[b] != 0) {
                                pub.wait_flag = x.root_flags + 2 + b;
                                pub.wait_epoch = x.slot_epoch[b];
                            }
                            pub.flag = x.flags.as<unsigned int>() + b;
                            pub.epoch = x.epoch;
                            pub.block_counter = x.flags.as<unsigned int>() + 12 + b;
                            pub.trace = x.trace_slot(x.epoch);
                            SDPA_TRY(merge_local(nullptr, xc, xt, xl, &pub));
                        }
                        x.slot_epoch[b] = x.epoch;
                    } else {
                    float* lsum_dst = (two_coll && !use_peer) ? s.contrib[b].as<float>() + (size_t)bs * dv : s.lsum[b].as<float>();
                    SDPA_TRY(merge_local(nullptr, s.contrib[b].as<float>(), s.tmax[b].as<float>(), lsum_dst));
                    }
                }
                SDPA_TRY(time_end(s, 2, s.s_compute));
                ++all_launches;
            }
            if (use_comm || use_out || ahead) SDPA_CUDA_TRY(cudaEventRecord(s.ev_compute_done[b], s.s_compute));
            if (ahead && pass_fence() == 1) {
                if (!s.ev_fence) SDPA_CUDA_TRY(cudaEventCreate(&s.ev_fence));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_fence, s.s_compute));
            }
            if (ii == num_iter - 1) {
                // who read this pass's K/V set last: the batch just issued
                if (!ahead) s.kv_guard[s.kv_set] = nullptr;   // not a cast-ahead context / a blocking call (ends with a wait)
                else if (num_iter == 1) s.kv_guard[s.kv_set] = s.ev_compute_done[b];
                else {
                    SDPA_CUDA_TRY(cudaEventRecord(s.ev_kv_read[s.kv_set], s.s_compute));
                    s.kv_guard[s.kv_set] = s.ev_kv_read[s.kv_set];
                }
            }
        }

        // ---- cross-shard merge ----------------------------------------------------------------
        if (use_ipc) {
            Shard& s = ctx->shards[0];
            sdpa_ctx::Ipc& x = ctx->ipc;
            SDPA_CUDA_TRY(cudaSetDevice(s.dev));
            if (x.sliced) {
                // every rank merges its share of the batch rows from its inbox (filled by all ranks' routed split merges:
                // all-to-all posted stores over NVLink), writes the fp64 rows into the root's staging buffer and raises its
                // "staged" flag there; the root then moves the assembled batch to its destination and releases the slots.
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_comm, s.ev_compute_done[b], 0));
                const int base = bs / world, rem = bs % world;
                const int my_rows = base + (s.grank < rem ? 1 : 0);
                const int my_first = s.grank * base + std::min(s.grank, rem);
                const float* cp[64];
                const float* tp[64];
                const float* lp[64];
                PeerSync sync;
                const size_t seg = (size_t)x.slice_cap * ((size_t)dv + 2);
                for (int r = 0; r < world; ++r) {   // local inbox: segment r holds source r's state of my rows
                    const float* in = x.xbuf[b].as<float>() + (size_t)r * seg;
                    cp[r] = in;
                    tp[r] = in + (size_t)x.slice_cap * dv;
                    lp[r] = tp[r] + x.slice_cap;
                    sync.ready[r] = x.flags.as<unsigned int>() + sdpa_ctx::Ipc::kFlagDelivered + b * 64 + r;
                }
                sync.consumed = x.root_flags + sdpa_ctx::Ipc::kFlagStaged + b * 64 + s.grank;   // "rank grank's rows are staged", in the root's memory
                sync.block_counter = x.flags.as<unsigned int>() + 6 + b;
                sync.epoch = x.epoch;
                SDPA_TRY(time_begin(s, 2, s.s_comm));
                SDPA_TRY(launch_merge_peers_synced(cp, tp, lp, world, my_rows, dv, x.root_stage[b] + (size_t)my_first * dv, sync,
                                                   s.s_comm));
                if (s.grank == 0) {
                    PeerSync col;
                    for (int r = 0; r < world; ++r) col.ready[r] = x.flags.as<unsigned int>() + sdpa_ctx::Ipc::kFlagStaged + b * 64 + r;
                    col.consumed = x.flags.as<unsigned int>() + 2 + b;
                    col.block_counter = x.flags.as<unsigned int>() + 8 + b;
                    col.epoch = x.epoch;
                    double* dst = direct ? res64 + (size_t)row0 * dv : s.out64[b].as<double>();
                    SDPA_TRY(launch_collect_slices(dst, x.stage[b].as<double>(), bs, dv, col, world, s.s_comm));
                }
                SDPA_TRY(time_end(s, 2, s.s_comm));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_comm_done[b], s.s_comm));
                if (s.grank != 0) SDPA_CUDA_TRY(cudaEventRecord(s.ev_slot_free[b], s.s_comm));
            } else if (s.grank == 0 && x.push_sync) {
                // final merge of the inbox right behind the root's own publish, on the compute stream: every read and every flag
                // poll is local; what it waits for is the other shards' pushes (posted NVLink stores issued when THEIR fused kernels ended)
                const float* cp[64];
                const float* tp[64];
                const float* lp[64];
                PeerSync sync;
                const size_t seg = (size_t)x.cap_rows * ((size_t)dv + 2);
                for (int r = 0; r < world; ++r) {
                    const float* base = x.xbuf[b].as<float>() + (size_t)r * seg;
                    cp[r] = base;
                    tp[r] = base + (size_t)x.cap_rows * dv;
                    lp[r] = tp[r] + x.cap_rows;
                    sync.ready[r] = x.flags.as<unsigned int>() + sdpa_ctx::Ipc::kFlagReady + b * 64 + r;
                }
                sync.consumed = x.flags.as<unsigned int>() + 2 + b;
                sync.block_counter = x.flags.as<unsigned int>() + 4 + b;
                sync.epoch = x.epoch;
                sync.trace = x.trace_slot(x.epoch);
                double* dst = direct ? res64 + (size_t)row0 * dv : s.out64[b].as<double>();
                SDPA_TRY(time_begin(s, 2, s.s_compute));
                SDPA_TRY(launch_merge_peers_synced(cp, tp, lp, world, bs, dv, dst, sync, s.s_compute));
                SDPA_TRY(time_end(s, 2, s.s_compute));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_comm_done[b], s.s_compute));
                if (ahead) {
                    // The side stream's gate moves behind this merge: a background cast released while the merge still runs is
                    // placed on whatever SMs have room -- several of its CTAs on one SM, which then cannot take a CTA of the next
                    // fused kernel (measured: that kernel ran in two waves, 336 us instead of 190).  Released together with the
                    // fused kernel on an empty GPU its CTAs land one per SM.
                    SDPA_CUDA_TRY(cudaEventRecord(s.ev_compute_done[b], s.s_compute));
                    if (pass_fence() == 1 && s.ev_fence) SDPA_CUDA_TRY(cudaEventRecord(s.ev_fence, s.s_compute));
                }
            } else if (s.grank == 0 && x.push) {
                // background merge of the inbox on the comm stream (after the root's own state is in): all reads local
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_comm, s.ev_compute_done[b], 0));
                unsigned int* consumed[64];
                for (int r = 0; r < world; ++r) consumed[r] = x.peer_flags[r] + 2 + b;
                double* dst = direct ? res64 + (size_t)row0 * dv : s.out64[b].as<double>();
                SDPA_TRY(time_begin(s, 2, s.s_comm));
                SDPA_TRY(launch_merge_inbox_background(x.xbuf[b].as<float>(), (size_t)x.cap_rows * ((size_t)dv + 2), x.cap_rows, world,
                                                       x.flags.as<unsigned int>() + sdpa_ctx::Ipc::kFlagReady + b * 64, consumed,
                                                       x.flags.as<unsigned int>() + 4 + b, x.epoch, x.trace_slot(x.epoch), bs, dv, dst,
                                                       s.sm_count, s.s_comm));
                SDPA_TRY(time_end(s, 2, s.s_comm));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_comm_done[b], s.s_comm));
            } else if (s.grank == 0 && x.instream) {
                // the merge already ran in the compute stream
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_comm_done[b], s.s_compute));
            } else if (s.grank == 0) {
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_comm, s.ev_compute_done[b], 0));
                const float* cp[64];
                const float* tp[64];
                const float* lp[64];
                PeerSync sync;
                for (int r = 0; r < world; ++r) {
                    const float* base = reinterpret_cast<const float*>(x.peer_x[b][r]);
                    cp[r] = base;
                    tp[r] = base + (size_t)x.cap_rows * dv;
                    lp[r] = tp[r] + x.cap_rows;
                    sync.ready[r] = x.peer_flags[r] + b;
                }
                sync.consumed = x.flags.as<unsigned int>() + 2 + b;
                sync.block_counter = x.flags.as<unsigned int>() + 4 + b;
                sync.epoch = x.epoch;
                sync.trace = x.trace_slot(x.epoch);
                double* dst = direct ? res64 + (size_t)row0 * dv : s.out64[b].as<double>();
                SDPA_TRY(time_begin(s, 2, s.s_comm));
                SDPA_TRY(launch_merge_peers_synced(cp, tp, lp, world, bs, dv, dst, sync, s.s_comm));
                SDPA_TRY(time_end(s, 2, s.s_comm));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_comm_done[b], s.s_comm));
            } else {
                // nothing to wait for on the host: slot reuse is guarded on the device by the root's "consumed" flag
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_comm_done[b], s.s_compute));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_slot_free[b], s.s_compute));
            }
        } else if (world > 1 && use_peer) {
            // fused device-side exchange: the root GPU reads every shard's state over NVLink
            Shard& r = ctx->shards[0];
            SDPA_CUDA_TRY(cudaSetDevice(r.dev));
            const float* cp[64];
            const float* tp[64];
            const float* lp[64];
            for (int i = 0; i < L; ++i) {
                SDPA_CUDA_TRY(cudaStreamWaitEvent(r.s_comm, ctx->shards[i].ev_compute_done[b], 0));
                cp[i] = ctx->shards[i].contrib[b].as<float>();
                tp[i] = ctx->shards[i].tmax[b].as<float>();
                lp[i] = ctx->shards[i].lsum[b].as<float>();
            }
            double* dst = direct ? res64 + (size_t)row0 * dv : r.out64[b].as<double>();
            SDPA_TRY(time_begin(r, 2, r.s_comm));
            SDPA_TRY(launch_merge_peers(cp, tp, lp, L, bs, dv, dst, r.s_comm));
            SDPA_TRY(time_end(r, 2, r.s_comm));
            ++all_launches;
            SDPA_CUDA_TRY(cudaEventRecord(r.ev_comm_done[b], r.s_comm));
            for (int i = 1; i < L; ++i) {
                Shard& s = ctx->shards[i];
                SDPA_CUDA_TRY(cudaSetDevice(s.dev));
                // shard i's slot is free once the root has read it
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_comm, r.ev_comm_done[b], 0));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_slot_free[b], s.s_comm));
            }
        } else if (world > 1) {
            for (int i = 0; i < L; ++i) {
                Shard& s = ctx->shards[i];
                SDPA_CUDA_TRY(cudaSetDevice(s.dev));
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_comm, s.ev_compute_done[b], 0));
                SDPA_TRY(time_begin(s, 2, s.s_comm));
            }
            // (1) global max (mpi.c:342)
            SDPA_NCCL_TRY(api->GroupStart());
            for (int i = 0; i < L; ++i) {
                Shard& s = ctx->shards[i];
                SDPA_NCCL_TRY(api->AllReduce(s.tmax[b].p, s.gmax[b].p, (size_t)bs, ncclFloat32, ncclMax, s.comm, s.s_comm));
            }
            SDPA_NCCL_TRY(api->GroupEnd());
            if (two_coll) {
                // (2) scale contrib and lsum to the global max (mpi.c:346-351); lsum lives right behind contrib,
                // so ONE reduce(SUM) carries both (mpi.c:354 + mpi.c:380); normalisation (mpi.c:358-362) and the
                // fp64 cast (mpi.c:373) run once on the root after it.
                for (int i = 0; i < L; ++i) {
                    Shard& s = ctx->shards[i];
                    SDPA_CUDA_TRY(cudaSetDevice(s.dev));
                    float* lsum_tail = s.contrib[b].as<float>() + (size_t)bs * dv;
                    SDPA_TRY(launch_rescale_to_gmax(s.contrib[b].as<float>(), lsum_tail, s.tmax[b].as<float>(),
                                                    s.gmax[b].as<float>(), bs, dv, s.s_comm));
                }
                SDPA_NCCL_TRY(api->GroupStart());
                for (int i = 0; i < L; ++i) {
                    Shard& s = ctx->shards[i];
                    void* recv = s.grank == 0 ? s.out32[b].p : nullptr;
                    SDPA_NCCL_TRY(api->Reduce(s.contrib[b].p, recv, (size_t)bs * dv + bs, ncclFloat32, ncclSum, 0, s.comm, s.s_comm));
                }
                SDPA_NCCL_TRY(api->GroupEnd());
                for (int i = 0; i < L; ++i) {
                    Shard& s = ctx->shards[i];
                    SDPA_CUDA_TRY(cudaSetDevice(s.dev));
                    if (s.grank == 0) {
                        double* dst = direct ? res64 + (size_t)row0 * dv : s.out64[b].as<double>();
                        SDPA_TRY(launch_finalize_reduced(dst, s.out32[b].as<float>(), s.out32[b].as<float>() + (size_t)bs * dv, bs, dv, s.s_comm));
                    }
                    SDPA_TRY(time_end(s, 2, s.s_comm));
                    SDPA_CUDA_TRY(cudaEventRecord(s.ev_comm_done[b], s.s_comm));
                    if (s.grank != 0) SDPA_CUDA_TRY(cudaEventRecord(s.ev_slot_free[b], s.s_comm));
                }
            } else {
            // the reference's three collectives (mpi.c:342,354,380), one NCCL group per step
            for (int i = 0; i < L; ++i) {
                Shard& s = ctx->shards[i];
                SDPA_CUDA_TRY(cudaSetDevice(s.dev));
                SDPA_TRY(launch_rescale_to_gmax(s.contrib[b].as<float>(), s.lsum[b].as<float>(), s.tmax[b].as<float>(),
                                                s.gmax[b].as<float>(), bs, dv, s.s_comm));
            }
            SDPA_NCCL_TRY(api->GroupStart());
            for (int i = 0; i < L; ++i) {
                Shard& s = ctx->shards[i];
                SDPA_NCCL_TRY(api->AllReduce(s.lsum[b].p, s.gsum[b].p, (size_t)bs, ncclFloat32, ncclSum, s.comm, s.s_comm));
            }
            SDPA_NCCL_TRY(api->GroupEnd());
            for (int i = 0; i < L; ++i) {
                Shard& s = ctx->shards[i];
                SDPA_CUDA_TRY(cudaSetDevice(s.dev));
                SDPA_TRY(launch_normalize(s.contrib[b].as<float>(), s.gsum[b].as<float>(), bs, dv, s.s_comm));
            }
            SDPA_NCCL_TRY(api->GroupStart());
            for (int i = 0; i < L; ++i) {
                Shard& s = ctx->shards[i];
                void* recv = s.grank == 0 ? s.out32[b].p : nullptr;
                SDPA_NCCL_TRY(api->Reduce(s.contrib[b].p, recv, (size_t)bs * dv, ncclFloat32, ncclSum, 0, s.comm, s.s_comm));
            }
            SDPA_NCCL_TRY(api->GroupEnd());
            for (int i = 0; i < L; ++i) {
                Shard& s = ctx->shards[i];
                SDPA_CUDA_TRY(cudaSetDevice(s.dev));
                if (s.grank == 0) {
                    double* dst = direct ? res64 + (size_t)row0 * dv : s.out64[b].as<double>();
                    SDPA_TRY(launch_cvt_f2d(dst, s.out32[b].as<float>(), (size_t)bs * dv, s.s_comm));  // mpi.c:373
                }
                SDPA_TRY(time_end(s, 2, s.s_comm));
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_comm_done[b], s.s_comm));
                if (s.grank != 0) SDPA_CUDA_TRY(cudaEventRecord(s.ev_slot_free[b], s.s_comm));
            }
            }
        }

        // ---- root: fp64 rows of this batch back to the host, or rounded into the typed result ------------
        for (int i = 0; i < L; ++i) {
            Shard& s = ctx->shards[i];
            if (s.grank != 0) continue;
            // one GPU writing to device memory: all on the compute stream (fp64 rows are in place already)
            cudaStream_t st = use_out ? s.s_out : s.s_compute;
            if (!use_out && direct) continue;
            SDPA_CUDA_TRY(cudaSetDevice(s.dev));
            if (use_out) SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_out, world > 1 ? s.ev_comm_done[b] : s.ev_compute_done[b], 0));
            if (!result_on_device)
                SDPA_CUDA_TRY(cudaMemcpyAsync(res64 + (size_t)row0 * dv, s.out64[b].p, (size_t)bs * dv * sizeof(double),
                                              cudaMemcpyDeviceToHost, s.s_out));
            else if (dtype == SDPA_DTYPE_F32)
                SDPA_TRY(launch_cvt_d2f(static_cast<float*>(result) + (size_t)row0 * dv, s.out64[b].as<double>(), (size_t)bs * dv, st));
            else if (dtype == SDPA_DTYPE_BF16)
                SDPA_TRY(launch_cvt_d2bf16(static_cast<__nv_bfloat16*>(result) + (size_t)row0 * dv, s.out64[b].as<double>(), (size_t)bs * dv, st));
            if (use_out) SDPA_CUDA_TRY(cudaEventRecord(s.ev_slot_free[b], s.s_out));
            else compute_stream_touched(s);
        }
        if (seq_slots) ++ctx->batch_seq;
    }

    if (use_ipc && ctx->shards[0].grank != 0 && !overlap) {
        // do not return (and possibly free or overwrite the slots) before the root has read them
        Shard& s = ctx->shards[0];
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        for (int b = 0; b < 2; ++b)
            if (ctx->ipc.slot_epoch[b] != 0)
                SDPA_TRY(launch_wait_flag(ctx->ipc.root_flags + 2 + b, ctx->ipc.slot_epoch[b], s.s_compute));
        compute_stream_touched(s);
    }

    const double hp1 = host_prof ? host_now_us() : 0.0;
    // ---- join: every stream back into the compute stream, then wait ----------------------------
    for (int i = 0; i < L; ++i) {
        Shard& s = ctx->shards[i];
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        cudaStream_t side[3] = {s.s_in, s.s_comm, s.s_out};
        const bool used[3] = {use_in, use_comm && !overlap, use_out && !overlap};   // overlap: the slots' own guards order the passes
        for (int j = 0; j < 3; ++j) {
            if (!used[j]) continue;
            SDPA_CUDA_TRY(cudaEventRecord(s.ev_join[j], side[j]));
            SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_compute, s.ev_join[j], 0));
            compute_stream_touched(s);
        }
        SDPA_TRY(time_end(s, 3, s.s_compute, true));
    }
    for (int i = 0; i < L && blocking; ++i) {
        Shard& s = ctx->shards[i];
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));
    }

    const double hp2 = host_prof ? host_now_us() : 0.0;
    if (overlap) ctx->exchange_pending = true;
    for (Shard& s : ctx->shards) {
        s.last_call_queued = !blocking;
        s.ahead_call = false;
        if (!ahead && !blocking && s.ahead_ever) {   // a queued pass outside the cast-ahead scheme on a context that uses it
            SDPA_CUDA_TRY(cudaSetDevice(s.dev));
            if (!s.ev_plain_end) SDPA_CUDA_TRY(cudaEventCreateWithFlags(&s.ev_plain_end, cudaEventDisableTiming));
            SDPA_CUDA_TRY(cudaEventRecord(s.ev_plain_end, s.s_compute));
            s.plain_end_recorded = true;
        }
    }
    if (marked) {
        ctx->last_timing_valid = false;   // evaluated lazily by sdpa_last_timings / sdpa_accumulated_timings
        ctx->acc_fused_launches += fused_launches;
        ctx->acc_calls += 1;
    }
    if (host_prof) {
        const double hp3 = host_now_us();
        fprintf(stderr, "sdpa host profile: enqueue %.1f us, join+sync %.1f us, event queries %.1f us (device total %.1f us)\n",
                hp1 - hp0, hp2 - hp1, hp3 - hp2, 0.0);
    }
    ctx->last_timing[4] = (float)fused_launches;
    (void)all_launches;
    ctx->last_timing[5] = (float)(launch_count() - launches_before);
    return SDPA_OK;
}


// ---------------------------------------------------------------------------
// SDPA_DIST_Q: K/V replicated on every local GPU (sdpa_load_kv_host_full), Q rows sharded by
// owner_count/owner_disp over the GPUs, every GPU writes its own rows of the result -- no exchange at all.
// The GPU analogue of the reference's small-problem branch (Bcast of the whole K/V, mpi.c:213-231); SURVEY 8(f) rank 3.
// Same per-batch pipeline as attention_impl (H2D on the copy-in stream, cast + fused kernel + split merge on the
// compute stream, D2H on the copy-out stream, two slots), once per GPU.
// ---------------------------------------------------------------------------
static sdpa_status attention_qshard_host(sdpa_ctx* ctx, const double* Q, double* result, int m)
{
    if (!ctx || m < 0 || (m > 0 && (!Q || !result))) {
        set_error("attention (Q-sharded): bad arguments");
        return SDPA_ERR_INVALID;
    }
    const int dk = ctx->dk, dv = ctx->dv;
    const int L = (int)ctx->shards.size();
    ctx->last_kernel = kernel_name(ctx->prec, dk, dv);
    for (float& t : ctx->last_timing) t = 0.f;
    ctx->last_timing_valid = true;
    if (m == 0) return SDPA_OK;

    int most_rows = 0;
    for (int i = 0; i < L; ++i) most_rows = std::max(most_rows, sdpa_owner_count(m, L, i));
    const int B = pick_q_batch(ctx, most_rows);
    int splits = ctx->cfg.kv_splits;
    if (splits <= 0)
        splits = is_umma(ctx->prec) ? attn_umma_pick_splits(B, ctx->shards[0].n_local, ctx->shards[0].sm_count)
                                    : attn_f32_pick_splits(B, ctx->shards[0].n_local, ctx->shards[0].sm_count);
    splits = std::max(1, std::min(splits, 64));
    const unsigned long long launches_before = launch_count();
    int fused_launches = 0;

    for (int i = 0; i < L; ++i) {
        Shard& s = ctx->shards[i];
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        SDPA_TRY(reserve_batch_buffers(ctx, s, B, splits, true));   // every GPU delivers rows: all need the fp64 out buffers
        if (s.marks_used > 2048) SDPA_TRY(fold_timings(s));
        for (int w = 0; w < 4; ++w) s.tpair_last[w] = s.tpair[w].size();
        s.marks_on = true;
        s.last_call_queued = false;
        compute_stream_touched(s);
        s.q_lo_off = (size_t)(((B + 127) & ~127) + 128) * dk;
        if (is_umma(ctx->prec)) {
            umma_plan_allow_v8(s.plan, false);   // this path merges by splits
            for (int b = 0; b < 2; ++b)
                SDPA_TRY(umma_plan_bind_q(s.plan, b, s.qc[b].as<__nv_bfloat16>(), (B + 127) & ~127, dk, prec_hl(ctx->prec), s.q_lo_off));
        }
        SDPA_TRY(time_begin(s, 3, s.s_compute));
        cudaEvent_t begun = s.marks[s.tpair[3].back()];
        SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_in, begun, 0));
        SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_out, begun, 0));
    }

    const int num_iter = ceil_div(most_rows, B);
    for (int ii = 0; ii < num_iter; ++ii) {
        const int b = ii & 1;
        for (int i = 0; i < L; ++i) {
            Shard& s = ctx->shards[i];
            const int my_rows = sdpa_owner_count(m, L, i);
            const int row0 = ii * B;
            if (row0 >= my_rows) continue;
            const int bs = std::min(B, my_rows - row0);
            const size_t grow0 = (size_t)sdpa_owner_disp(m, L, i) + row0;   // first global row of this batch
            SDPA_CUDA_TRY(cudaSetDevice(s.dev));
            if (ii >= 2) SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_in, s.ev_q_free[b], 0));
            SDPA_TRY(h2d_any(s.q64[b].p, Q + grow0 * dk, (size_t)bs * dk * sizeof(double), s.s_in));
            SDPA_CUDA_TRY(cudaEventRecord(s.ev_q_ready[b], s.s_in));
            SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_compute, s.ev_q_ready[b], 0));
            if (ii >= 2) SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_compute, s.ev_slot_free[b], 0));   // out64[b] has been copied out
            compute_stream_touched(s);

            SDPA_TRY(time_begin(s, 0, s.s_compute));
            SDPA_TRY(cast_in(ctx->prec, s.qc[b].p, s.q_lo_off, 0, s.q64[b].as<double>(), (size_t)bs * dk, s.s_compute));
            SDPA_TRY(time_end(s, 0, s.s_compute));
            SDPA_CUDA_TRY(cudaEventRecord(s.ev_q_free[b], s.s_compute));

            Partials part{s.part_o.as<float>(), s.part_tmax.as<float>(), s.part_lsum.as<float>(), splits, B};
            double* dst = s.out64[b].as<double>();
            SDPA_TRY(time_begin(s, 1, s.s_compute));
            SDPA_TRY(run_fused(ctx, s, b, s.qc[b].as<float>(), bs, splits, part, splits == 1 ? dst : nullptr));
            SDPA_TRY(time_end(s, 1, s.s_compute));
            if (is_umma(ctx->prec)) SDPA_TRY(launch_attn_umma_twin(s.plan, b, bs, splits, part, splits == 1 ? dst : nullptr, s.s_compute));
            ++fused_launches;
            if (splits > 1) {
                SDPA_TRY(time_begin(s, 2, s.s_compute));
                SDPA_TRY(launch_merge_splits(part, bs, dv, dst, nullptr, nullptr, nullptr, false, s.s_compute));
                SDPA_TRY(time_end(s, 2, s.s_compute));
            }
            SDPA_CUDA_TRY(cudaEventRecord(s.ev_compute_done[b], s.s_compute));
            SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_out, s.ev_compute_done[b], 0));
            SDPA_CUDA_TRY(cudaMemcpyAsync(result + grow0 * dv, dst, (size_t)bs * dv * sizeof(double), cudaMemcpyDeviceToHost, s.s_out));
            SDPA_CUDA_TRY(cudaEventRecord(s.ev_slot_free[b], s.s_out));
        }
    }

    for (int i = 0; i < L; ++i) {
        Shard& s = ctx->shards[i];
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        cudaStream_t side[2] = {s.s_in, s.s_out};
        for (int j = 0; j < 2; ++j) {
            SDPA_CUDA_TRY(cudaEventRecord(s.ev_join[j], side[j]));
            SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_compute, s.ev_join[j], 0));
        }
        compute_stream_touched(s);
        SDPA_TRY(time_end(s, 3, s.s_compute));
    }
    for (int i = 0; i < L; ++i) {
        Shard& s = ctx->shards[i];
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));
    }
    ctx->last_timing_valid = false;
    ctx->acc_fused_launches += fused_launches;
    ctx->acc_calls += 1;
    ctx->last_timing[4] = (float)fused_launches;
    ctx->last_timing[5] = (float)(launch_count() - launches_before);
    return SDPA_OK;
}

// ---------------------------------------------------------------------------
// One process per GPU, data on rank 0 only: the reference's own calling convention
// (mpi.c:193-197 dims Bcast, mpi.c:213-266 K/V distribution, mpi.c:305,327 Q Ibcast).
// Rank 0 uploads each destination's rows in fp64 chunks, casts them on its GPU and
// ncclSend()s the compute-precision chunk; rank r ncclRecv()s straight into its shard.
// ---------------------------------------------------------------------------
static sdpa_status scatter_operand(sdpa_ctx* ctx, Shard& s, const NcclApi* api, int prec, void* my_dst, size_t my_lo_off,
                                   const double* src_full, int n, int width, DevBuf* sendbuf)
{
    const size_t usz = unit_size(prec);
    const bool split = prec == SDPA_PREC_BF16X3;
    const int world = ctx->world;
    if (s.grank == 0) {
        for (int r = 0; r < world; ++r) {
            const size_t count = (size_t)sdpa_owner_count(n, world, r) * width;
            const double* src = src_full + (size_t)sdpa_owner_disp(n, world, r) * width;
            size_t done = 0;
            int c = 0;
            while (done < count) {
                const size_t len = std::min(kStageElems, count - done);
                const int b = c & 1;
                SDPA_TRY(s.kv_stage[b].reserve(kStageElems * sizeof(double)));
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_in, s.ev_stage_free[b], 0));
                SDPA_TRY(h2d_any(s.kv_stage[b].p, src + done, len * sizeof(double), s.s_in));   // pinned: direct; pageable: staged
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_stage_ready[b], s.s_in));
                SDPA_CUDA_TRY(cudaStreamWaitEvent(s.s_compute, s.ev_stage_ready[b], 0));
                if (r == 0) {
                    SDPA_TRY(cast_in(prec, my_dst, my_lo_off, done, s.kv_stage[b].as<double>(), len, s.s_compute));
                } else {
                    // chunk in compute precision: [hi (or the only) array | lo array of the split precision]
                    SDPA_TRY(sendbuf[b].reserve(kStageElems * usz * (split ? 2 : 1)));
                    SDPA_TRY(cast_in(prec, sendbuf[b].p, kStageElems, 0, s.kv_stage[b].as<double>(), len, s.s_compute));
                    SDPA_NCCL_TRY(api->Send(sendbuf[b].p, len * usz, ncclUint8, r, s.comm, s.s_compute));
                    if (split)
                        SDPA_NCCL_TRY(api->Send((char*)sendbuf[b].p + kStageElems * usz, len * usz, ncclUint8, r, s.comm, s.s_compute));
                }
                SDPA_CUDA_TRY(cudaEventRecord(s.ev_stage_free[b], s.s_compute));
                done += len;
                ++c;
            }
        }
    } else {
        const size_t count = (size_t)sdpa_owner_count(n, world, s.grank) * width;
        size_t done = 0;
        while (done < count) {
            const size_t len = std::min(kStageElems, count - done);
            SDPA_NCCL_TRY(api->Recv((char*)my_dst + done * usz, len * usz, ncclUint8, 0, s.comm, s.s_compute));
            if (split) SDPA_NCCL_TRY(api->Recv((char*)my_dst + (my_lo_off + done) * usz, len * usz, ncclUint8, 0, s.comm, s.s_compute));
            done += len;
        }
    }
    return SDPA_OK;
}

static sdpa_status scatter_attention_impl(sdpa_ctx* ctx, const double* Q, const double* K, const double* V,
                                          double* result, int m, int n, int dk, int dv)
{
    if (!ctx || ctx->shards.size() != 1 || ctx->world < 2) {
        set_error("scatter attention needs a one-GPU-per-process context with world_size > 1");
        return SDPA_ERR_INVALID;
    }
    const NcclApi* api = nccl_api();
    if (!api) return SDPA_ERR_NCCL;
    Shard& s = ctx->shards[0];
    SDPA_CUDA_TRY(cudaSetDevice(s.dev));
    // dims from rank 0 (mpi.c:193-197), together with rank 0's verdict on its own arguments: every rank leaves with the same
    // error instead of the others blocking in a receive that rank 0 never posts
    int dims[5] = {m, n, dk, dv, 1};
    if (s.grank == 0 && (m < 0 || n < 0 || dk < 1 || dv < 1 || (n > 0 && (!K || !V)) || (m > 0 && (!Q || !result)))) dims[4] = 0;
    SDPA_TRY(s.gmax[0].reserve(256));
    if (s.grank == 0) SDPA_CUDA_TRY(cudaMemcpyAsync(s.gmax[0].p, dims, sizeof(dims), cudaMemcpyHostToDevice, s.s_compute));
    SDPA_NCCL_TRY(api->Broadcast(s.gmax[0].p, s.gmax[0].p, 5, ncclInt32, 0, s.comm, s.s_compute));
    SDPA_CUDA_TRY(cudaMemcpyAsync(dims, s.gmax[0].p, sizeof(dims), cudaMemcpyDeviceToHost, s.s_compute));
    SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));
    m = dims[0]; n = dims[1]; dk = dims[2]; dv = dims[3];
    if (!dims[4]) {
        set_error("attention(): bad dimensions or NULL input on rank 0 (m=%d n=%d dk=%d dv=%d)", m, n, dk, dv);
        return SDPA_ERR_INVALID;
    }
    const int prec = resolve_precision(SDPA_DTYPE_F64, ctx->cfg.precision, dk, dv);
    SDPA_TRY(check_precision(prec, dk, dv));
    ctx->dk = dk;
    ctx->dv = dv;
    ctx->prec = prec;
    ctx->dtype = SDPA_DTYPE_F64;
    ctx->zero_copy = false;
    const size_t esz = elem_size(prec);
    s.n_local = sdpa_owner_count(n, ctx->world, s.grank);
    SDPA_TRY(s.Kc.reserve(((size_t)s.n_local + 128) * dk * esz));
    SDPA_TRY(s.Vc.reserve(((size_t)s.n_local + 128) * dv * esz));
    s.k_in = s.Kc.p;
    s.v_in = s.Vc.p;
    s.k_lo_off = ((size_t)s.n_local + 128) * dk;
    s.v_lo_off = ((size_t)s.n_local + 128) * dv;
    DevBuf sendbuf[2];
    sdpa_status st = scatter_operand(ctx, s, api, prec, s.Kc.p, s.k_lo_off, K, n, dk, sendbuf);
    if (st == SDPA_OK) st = scatter_operand(ctx, s, api, prec, s.Vc.p, s.v_lo_off, V, n, dv, sendbuf);
    if (st == SDPA_OK && cudaStreamSynchronize(s.s_compute) != cudaSuccess) {
        set_error("K/V scatter failed: %s", cudaGetErrorString(cudaGetLastError()));
        st = SDPA_ERR_CUDA;
    }
    sendbuf[0].release();
    sendbuf[1].release();
    SDPA_TRY(st);
    if (is_umma(prec)) {
        if (!s.plan) SDPA_TRY(umma_plan_create(&s.plan));
        SDPA_TRY(umma_plan_bind_kv(s.plan, s.Kc.as<__nv_bfloat16>(), s.Vc.as<__nv_bfloat16>(), s.n_local, dk, dv, prec_hl(prec),
                                   s.k_lo_off, s.v_lo_off));
    }
    return attention_impl(ctx, Q, nullptr, result, false, m, /*q_from_root=*/true);
}

}  // namespace sdpa

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

const char* sdpa_last_error(void) { return sdpa::get_error(); }
const char* sdpa_version(void) { return "sdpa_b200 0.1 (sm_100a)"; }

int sdpa_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

/* mpi.c:19-22 */
int sdpa_owner_count(int n, int size, int rank)
{
    if (size <= 0) return 0;
    const int q = n / size, r = n % size;
    return q + (rank < r ? 1 : 0);
}

/* mpi.c:24-27 */
int sdpa_owner_disp(int n, int size, int rank)
{
    if (size <= 0) return 0;
    const int q = n / size, r = n % size;
    return rank * q + (rank < r ? rank : r);
}

int sdpa_precision_supported(int precision, int dk, int dv, int* resolved)
{
    return sdpa_precision_supported_for(SDPA_DTYPE_F64, precision, dk, dv, resolved);
}

int sdpa_precision_supported_for(int dtype, int precision, int dk, int dv, int* resolved)
{
    if (!dtype_valid(dtype) || precision < SDPA_PREC_AUTO || precision > SDPA_PREC_BF16X3 || dk < 1 || dv < 1) return 0;
    const int prec = resolve_precision(dtype, precision, dk, dv);
    if (resolved) *resolved = prec;
    if (is_umma(prec)) return attn_umma_supported(dk, dv, prec_hl(prec)) ? 1 : 0;
    return attn_f32_supported(dk, dv) ? 1 : 0;
}

void sdpa_config_init(sdpa_config* cfg)
{
    if (!cfg) return;
    memset(cfg, 0, sizeof(*cfg));
    cfg->precision = SDPA_PREC_AUTO;
    cfg->merge = SDPA_MERGE_NCCL2;
    cfg->num_local = 1;
}

sdpa_status sdpa_get_unique_id(void* out128)
{
    if (!out128) {
        set_error("sdpa_get_unique_id: NULL output");
        return SDPA_ERR_INVALID;
    }
    const NcclApi* api = nccl_api();
    if (!api) return SDPA_ERR_NCCL;
    ncclUniqueId id;
    SDPA_NCCL_TRY(api->GetUniqueId(&id));
    memcpy(out128, &id, sizeof(id));
    return SDPA_OK;
}

sdpa_status sdpa_ctx_create(sdpa_ctx** out, const sdpa_config* cfg_in, const void* nccl_id)
{
    if (!out) {
        set_error("sdpa_ctx_create: NULL output");
        return SDPA_ERR_INVALID;
    }
    *out = nullptr;
    sdpa_config cfg;
    if (cfg_in) cfg = *cfg_in;
    else sdpa_config_init(&cfg);
    const int L = cfg.num_local > 0 ? cfg.num_local : 1;
    const int world = cfg.world_size > 0 ? cfg.world_size : L;
    if (cfg.rank_base < 0 || cfg.rank_base + L > world || L > 64 || world > 64) {
        set_error("sdpa_ctx_create: inconsistent shard layout (num_local=%d rank_base=%d world=%d; max 64)", L,
                  cfg.rank_base, world);
        return SDPA_ERR_INVALID;
    }
    int ndev = sdpa_device_count();
    if (ndev <= 0) {
        set_error("no CUDA device visible: this engine has no CPU fallback");
        return SDPA_ERR_CUDA;
    }
    if (cfg.first_device < 0 || cfg.first_device + L > ndev) {
        set_error("sdpa_ctx_create: devices [%d,%d) requested but %d visible", cfg.first_device, cfg.first_device + L, ndev);
        return SDPA_ERR_INVALID;
    }
    if (world > L && !nccl_id) {
        set_error("sdpa_ctx_create: world_size %d > num_local %d needs a shared ncclUniqueId", world, L);
        return SDPA_ERR_INVALID;
    }
    sdpa_ctx* ctx = new sdpa_ctx();
    ctx->cfg = cfg;
    ctx->world = world;
    ctx->rank_base = cfg.rank_base;
    {
        if (const char* me = getenv("SDPA_STAGE_TIMING_EVERY")) ctx->mark_every = std::max(1, atoi(me));
        if (const char* dt = getenv("SDPA_DEFER_TWIN")) {   // 0: twin always in the stream; 1: deferred on single-shard contexts only; 2: everywhere
            ctx->defer_twin = *dt != '0';
            ctx->defer_multi = *dt == '2' ? true : (*dt == '1' ? false : ctx->defer_multi);
        }
        const char* ov = getenv("SDPA_OVERLAP_PASSES");   // SDPA_OVERLAP_PASSES=0: every queued pass joins its exchange before the next starts
        ctx->overlap_passes = !(ov && *ov == '0');
        const char* ca = getenv("SDPA_CAST_AHEAD");
        ctx->cast_ahead = !(ca && *ca == '0');
    }
    ctx->shards.resize(L);
    sdpa_status st = SDPA_OK;
    for (int i = 0; i < L && st == SDPA_OK; ++i) {
        ctx->shards[i].dev = cfg.first_device + i;
        ctx->shards[i].grank = cfg.rank_base + i;
        st = shard_init(ctx->shards[i]);
    }
    if (const char* tp = getenv("SDPA_CAST_TRACE"); st == SDPA_OK && tp && *tp && L == 1 && world == 1) {
        ctx->cast_trace_path = tp;
        cudaSetDevice(ctx->shards[0].dev);
        st = ctx->cast_trace.reserve(1024 * sizeof(unsigned long long));
        if (st == SDPA_OK) {
            cudaMemset(ctx->cast_trace.p, 0, ctx->cast_trace.bytes);
            set_cast_trace(ctx->cast_trace.as<unsigned long long>());
        }
    }
    // peer access among the local GPUs (for the fused exchange)
    if (st == SDPA_OK && L > 1) {
        bool all = true;
        for (int i = 0; i < L; ++i)
            for (int j = 0; j < L; ++j) {
                if (i == j) continue;
                int can = 0;
                cudaDeviceCanAccessPeer(&can, ctx->shards[i].dev, ctx->shards[j].dev);
                if (!can) { all = false; continue; }
                cudaSetDevice(ctx->shards[i].dev);
                cudaError_t e = cudaDeviceEnablePeerAccess(ctx->shards[j].dev, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) all = false;
                cudaGetLastError();
            }
        ctx->peer_ok = all;
        // work buffers live in the devices' stream-ordered memory pools: peers read each other's exchange state, so every
        // local device gets read/write access to every other local device's pool (cudaDeviceEnablePeerAccess does not cover pools)
        if (all && mem_pool_enabled()) {
            for (int i = 0; i < L; ++i) {
                cudaMemPool_t pool;
                if (cudaDeviceGetDefaultMemPool(&pool, ctx->shards[i].dev) != cudaSuccess) continue;
                std::vector<cudaMemAccessDesc> desc;
                for (int j = 0; j < L; ++j) {
                    if (i == j) continue;
                    cudaMemAccessDesc d{};
                    d.location.type = cudaMemLocationTypeDevice;
                    d.location.id = ctx->shards[j].dev;
                    d.flags = cudaMemAccessFlagsProtReadWrite;
                    desc.push_back(d);
                }
                if (!desc.empty() && cudaMemPoolSetAccess(pool, desc.data(), desc.size()) != cudaSuccess) ctx->peer_ok = false;
            }
            cudaGetLastError();
        }
    }
    // NCCL communicator(s)
    const bool need_nccl = world > 1 && !(cfg.merge == SDPA_MERGE_PEER && ctx->peer_ok && world == L);
    if (st == SDPA_OK && need_nccl) {
        const NcclApi* api = nccl_api();
        if (!api) st = SDPA_ERR_NCCL;
        else {
            ncclUniqueId id;
            if (nccl_id) memcpy(&id, nccl_id, sizeof(id));
            else if (api->GetUniqueId(&id) != ncclSuccess) st = SDPA_ERR_NCCL;
            if (st == SDPA_OK) {
                ncclResult_t r = api->GroupStart();
                for (int i = 0; i < L && r == ncclSuccess; ++i) {
                    cudaSetDevice(ctx->shards[i].dev);
                    r = api->CommInitRank(&ctx->shards[i].comm, world, id, ctx->shards[i].grank);
                }
                ncclResult_t r2 = api->GroupEnd();
                if (r != ncclSuccess || r2 != ncclSuccess) {
                    set_error("ncclCommInitRank failed: %s", api->GetErrorString(r != ncclSuccess ? r : r2));
                    st = SDPA_ERR_NCCL;
                }
            }
        }
    }
    if (st != SDPA_OK) {
        for (Shard& s : ctx->shards) shard_destroy(s, nullptr);
        delete ctx;
        return st;
    }
    *out = ctx;
    return SDPA_OK;
}

sdpa_status sdpa_ctx_destroy(sdpa_ctx* ctx)
{
    if (!ctx) return SDPA_OK;
    const NcclApi* api = nullptr;
    for (Shard& s : ctx->shards)
        if (s.comm) api = nccl_api();
    if (!ctx->shards.empty()) {
        drain_exchange(ctx);
        cudaSetDevice(ctx->shards[0].dev);
        cudaDeviceSynchronize();
        if (ctx->cast_trace.p) {   // developer aid: per-CTA stamps of the last background cast + the last two fused kernels
            std::vector<unsigned long long> host(1024);
            if (cudaMemcpy(host.data(), ctx->cast_trace.p, host.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost) == cudaSuccess)
                if (FILE* f = fopen(ctx->cast_trace_path.c_str(), "w")) {
                    fprintf(f, "fused %llu %llu %llu %llu passes %llu\n", host[600], host[601], host[602], host[603], ctx->trace_pass);
                    for (int c = 0; c < 300; ++c)
                        if (host[2 * c]) fprintf(f, "cta %d %llu %llu\n", c, host[2 * c], host[2 * c + 1]);
                    fclose(f);
                }
            set_cast_trace(nullptr);
            ctx->cast_trace.release();
        }
        if (ctx->ipc.trace.p) {   // developer aid: dump the exchange timeline of this rank
            const char* tp = getenv("SDPA_EXCHANGE_TRACE");
            const unsigned int W = sdpa_ctx::Ipc::kTraceWords;
            std::vector<unsigned long long> host((size_t)sdpa_ctx::Ipc::kTraceEpochs * W);
            if (tp && cudaMemcpy(host.data(), ctx->ipc.trace.p, host.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost) == cudaSuccess) {
                char path[1024];
                snprintf(path, sizeof(path), "%s.rank%d", tp, ctx->rank_base);
                if (FILE* f = fopen(path, "w")) {
                    fprintf(f, "epoch published_ns merge_begin_ns flags_seen_ns merge_done_ns flag_seen_ns[0..7]   (last epoch %u; every GPU has its own clock)\n", ctx->ipc.epoch);
                    for (unsigned int e = 0; e < sdpa_ctx::Ipc::kTraceEpochs; ++e)
                        if (host[e * W] || host[e * W + 1]) {
                            fprintf(f, "%u", e);
                            for (unsigned int k = 0; k < W; ++k) fprintf(f, " %llu", host[e * W + k]);
                            fprintf(f, "\n");
                        }
                    fclose(f);
                }
            }
            ctx->ipc.trace.release();
        }
        ipc_close(ctx);
        ctx->ipc.xbuf[0].release();
        ctx->ipc.xbuf[1].release();
        ctx->ipc.flags.release();
        ctx->ipc.stage[0].release();
        ctx->ipc.stage[1].release();
    }
    for (Shard& s : ctx->shards) shard_destroy(s, api);
    delete ctx;
    return SDPA_OK;
}

sdpa_status sdpa_load_kv_host(sdpa_ctx* ctx, const double* const* K_shards, const double* const* V_shards,
                              const int* n_local, int dk, int dv)
{
    return load_kv(ctx, SDPA_DTYPE_F64, reinterpret_cast<const void* const*>(K_shards), reinterpret_cast<const void* const*>(V_shards),
                   n_local, dk, dv, false);
}

sdpa_status sdpa_load_kv_device(sdpa_ctx* ctx, const double* const* K_shards, const double* const* V_shards,
                                const int* n_local, int dk, int dv)
{
    return load_kv(ctx, SDPA_DTYPE_F64, reinterpret_cast<const void* const*>(K_shards), reinterpret_cast<const void* const*>(V_shards),
                   n_local, dk, dv, true);
}

sdpa_status sdpa_load_kv_host_full(sdpa_ctx* ctx, const double* K, const double* V, int n, int dk, int dv)
{
    if (!ctx || n < 0) {
        set_error("sdpa_load_kv_host_full: bad arguments");
        return SDPA_ERR_INVALID;
    }
    if (ctx->world != (int)ctx->shards.size()) {
        set_error("sdpa_load_kv_host_full needs a single-process context (world == num_local)");
        return SDPA_ERR_INVALID;
    }
    const int L = (int)ctx->shards.size();
    std::vector<const void*> kp(L), vp(L);
    std::vector<int> cnt(L);
    // Distribution policy, the GPU analogue of the reference's Bcast-vs-Scatterv switch (mpi.c:213-215: K/V under 64 MiB
    // in fp32 are broadcast whole): with K/V replicated the Q rows can be sharded instead and no exchange is needed.
    const int mode = ctx->cfg.distribution;
    const bool small = (size_t)n * ((size_t)dk + dv) * sizeof(float) < ((size_t)64 << 20);
    const bool replicate = L > 1 && n > 0 && (mode == SDPA_DIST_Q || (mode == SDPA_DIST_AUTO && small));
    for (int i = 0; i < L; ++i) {
        cnt[i] = replicate ? n : sdpa_owner_count(n, L, i);
        const int d = replicate ? 0 : sdpa_owner_disp(n, L, i);
        kp[i] = K ? K + (size_t)d * dk : nullptr;
        vp[i] = V ? V + (size_t)d * dv : nullptr;
    }
    SDPA_TRY(load_kv(ctx, SDPA_DTYPE_F64, kp.data(), vp.data(), cnt.data(), dk, dv, false));
    ctx->qshard = replicate;
    return SDPA_OK;
}

sdpa_status sdpa_attention_host(sdpa_ctx* ctx, const double* Q, double* result, int m)
{
    if (ctx && ctx->qshard && ctx->dk != 0) return attention_qshard_host(ctx, Q, result, m);
    return attention_impl(ctx, Q, nullptr, result, false, m);
}

sdpa_status sdpa_attention_device(sdpa_ctx* ctx, const double* const* Q_dev, double* result_dev, int m)
{
    if (m > 0 && !Q_dev) {
        set_error("sdpa_attention_device: Q_dev is NULL");
        return SDPA_ERR_INVALID;
    }
    if (ctx && ctx->qshard) {
        set_error("sdpa_attention_device: the resident K/V is replicated (SDPA_DIST_Q); that distribution serves host arrays only");
        return SDPA_ERR_UNSUPPORTED;
    }
    return attention_impl(ctx, nullptr, reinterpret_cast<const void* const*>(Q_dev), result_dev, true, m);
}

/* One pass on device-resident arrays of element type `dtype`: K/V shard cast (or none, where the fused kernel reads the arrays in
 * place) + Q batches + merge.  blocking = false: queued (sdpa_enqueue_device_*), repaired at sdpa_synchronize. */
static sdpa_status device_pass(sdpa_ctx* ctx, int dtype, const void* const* K_shards, const void* const* V_shards, const int* n_local,
                               int dk, int dv, const void* const* Q_dev, void* result_dev, int m, bool blocking, const char* what)
{
    if (!dtype_valid(dtype)) {
        set_error("%s: unknown dtype %d", what, dtype);
        return SDPA_ERR_INVALID;
    }
    if (m > 0 && !Q_dev) {
        set_error("%s: Q_dev is NULL", what);
        return SDPA_ERR_INVALID;
    }
    const size_t esz = dtype_size(dtype);
    if (ctx && n_local && dk >= 1 && dv >= 1) {
        // Operands read in place: the tensor-core kernels load them through TMA, whose global addresses must be 16-byte aligned;
        // the fp32 kernel takes any fp32 array.  A misaligned operand is refused, not copied.
        const int prec = resolve_precision(dtype, ctx->cfg.precision, dk, dv);
        const size_t align = is_umma(prec) ? 16 : esz;
        auto bad = [&](const void* p) { return p && (uintptr_t)p % align != 0; };
        for (size_t i = 0; i < ctx->shards.size() && reads_in_place(dtype, prec); ++i)
            if ((n_local[i] > 0 && K_shards && V_shards && (bad(K_shards[i]) || bad(V_shards[i]))) || (m > 0 && bad(Q_dev[i]))) {
                set_error("%s: %s operands are read in place by the %s kernel, which needs K, V and Q aligned to %zu bytes "
                          "(shard %zu: K=%p V=%p Q=%p)", what, dtype_name(dtype), kernel_name(prec, dk, dv), align, i,
                          K_shards ? K_shards[i] : nullptr, V_shards ? V_shards[i] : nullptr, m > 0 ? Q_dev[i] : nullptr);
                return SDPA_ERR_INVALID;
            }
    }
    // Cast-ahead (queued fp64 passes): where the persistent fused kernel takes the pass (it leaves room on every SM for one small
    // CTA), on one GPU or with the overlapped device-side exchange, the casts of this pass run beside the previous pass's fused
    // kernel.  Typed passes never cast ahead: they are "plain" queued passes (ev_plain_end).
    bool ahead = false;
    if (!blocking && dtype == SDPA_DTYPE_F64 && ctx && ctx->cast_ahead && !ctx->repairing && n_local && m > 0 && dk == 128 && dv == 128) {
        const int L = (int)ctx->shards.size();
        const bool ipc = ctx->world > 1 && ctx->cfg.merge == SDPA_MERGE_PEER && L == 1 && ctx->overlap_passes;
        const int prec = resolve_precision(dtype, ctx->cfg.precision, dk, dv);
        // single-batch passes only: between two batches of one pass the side kernel would be released while other kernels
        // still run, and its CTAs pile up on the SMs that happen to have room (see the gate of the pushsync root form)
        const int B = pick_q_batch(ctx, m);
        ahead = (ctx->world == 1 || ipc) && m <= B && persistent_pieces(ctx, prec, dk, dv, B, n_local) > 1;
        // a pass whose operands ARE an earlier queued pass's result (chained passes) must see that result: its casts stay in
        // the compute stream, behind the merge that writes it
        auto aliases_result = [&](const void* ptr, size_t bytes) {
            const char* a = static_cast<const char*>(ptr);
            for (const sdpa_ctx::ByteRange& r : ctx->queued_results)
                if (a && a < r.p + r.n && r.p < a + bytes) return true;
            return false;
        };
        for (int i = 0; i < L && ahead; ++i)
            if ((K_shards && aliases_result(K_shards[i], (size_t)n_local[i] * dk * esz)) ||
                (V_shards && aliases_result(V_shards[i], (size_t)n_local[i] * dv * esz)) ||
                aliases_result(Q_dev[i], (size_t)m * dk * esz))
                ahead = false;
    }
    SDPA_TRY(load_kv(ctx, dtype, K_shards, V_shards, n_local, dk, dv, true, true, ahead));
    SDPA_TRY(attention_impl(ctx, nullptr, Q_dev, result_dev, true, m, false, blocking, dtype));
    if (blocking) return SDPA_OK;
    if (result_dev && m > 0) {
        if (ctx->queued_results.size() >= 64) ctx->queued_results.erase(ctx->queued_results.begin());   // bounded: older ones are long complete
        ctx->queued_results.push_back({reinterpret_cast<const char*>(result_dev), (size_t)m * dv * esz});
    }
    if (ctx->deferring && !ctx->call_guards.empty()) {
        const size_t L = ctx->shards.size();
        sdpa_ctx::PendingPass p;
        p.dtype = dtype;
        p.K.assign(K_shards, K_shards + L);
        p.V.assign(V_shards, V_shards + L);
        p.Q.assign(Q_dev, Q_dev + L);
        p.n_local.assign(n_local, n_local + L);
        p.dk = dk;
        p.dv = dv;
        p.result = result_dev;
        p.m = m;
        p.guards = ctx->call_guards;
        ctx->pending.push_back(std::move(p));
    }
    return SDPA_OK;
}

/* attention() on device-resident fp64 arrays in one call: K/V shard cast + Q batches + merge. */
sdpa_status sdpa_attention_device_full(sdpa_ctx* ctx, const double* const* K_shards, const double* const* V_shards,
                                       const int* n_local, int dk, int dv, const double* const* Q_dev, double* result_dev, int m)
{
    return device_pass(ctx, SDPA_DTYPE_F64, reinterpret_cast<const void* const*>(K_shards), reinterpret_cast<const void* const*>(V_shards),
                       n_local, dk, dv, reinterpret_cast<const void* const*>(Q_dev), result_dev, m, true, "sdpa_attention_device_full");
}

/* The same pass, queued: returns as soon as the work is enqueued (stream order keeps consecutive passes and their
 * shared buffers in sequence); sdpa_synchronize() waits.  All arrays must stay valid until then. */
sdpa_status sdpa_enqueue_device_full(sdpa_ctx* ctx, const double* const* K_shards, const double* const* V_shards,
                                     const int* n_local, int dk, int dv, const double* const* Q_dev, double* result_dev, int m)
{
    return device_pass(ctx, SDPA_DTYPE_F64, reinterpret_cast<const void* const*>(K_shards), reinterpret_cast<const void* const*>(V_shards),
                       n_local, dk, dv, reinterpret_cast<const void* const*>(Q_dev), result_dev, m, false, "sdpa_enqueue_device_full");
}

sdpa_status sdpa_attention_device_typed(sdpa_ctx* ctx, int dtype, const void* const* K_shards, const void* const* V_shards,
                                        const int* n_local, int dk, int dv, const void* const* Q_dev, void* result_dev, int m)
{
    return device_pass(ctx, dtype, K_shards, V_shards, n_local, dk, dv, Q_dev, result_dev, m, true, "sdpa_attention_device_typed");
}

sdpa_status sdpa_enqueue_device_typed(sdpa_ctx* ctx, int dtype, const void* const* K_shards, const void* const* V_shards,
                                      const int* n_local, int dk, int dv, const void* const* Q_dev, void* result_dev, int m)
{
    return device_pass(ctx, dtype, K_shards, V_shards, n_local, dk, dv, Q_dev, result_dev, m, false, "sdpa_enqueue_device_typed");
}

/* Deferred guard repair: wait for the queued passes, read the guard rings once, agree across processes, re-run (exact variant
 * alone, blocking) every pass one of whose launches raised its guard on any shard. */
static sdpa_status resolve_pending(sdpa_ctx* ctx)
{
    if (ctx->pending.empty()) return SDPA_OK;
    const int L = (int)ctx->shards.size();
    SDPA_TRY(drain_exchange(ctx));
    std::vector<std::vector<unsigned int>> ring(L, std::vector<unsigned int>(kGuardRing, 0u));
    for (int i = 0; i < L; ++i) {
        Shard& s = ctx->shards[i];
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));
        const unsigned int* dev_ring = umma_plan_guard_ring(s.plan);
        if (dev_ring) SDPA_CUDA_TRY(cudaMemcpy(ring[i].data(), dev_ring, kGuardRing * sizeof(unsigned int), cudaMemcpyDeviceToHost));
    }
    std::vector<int> fired(ctx->pending.size(), 0);
    for (size_t p = 0; p < ctx->pending.size(); ++p)
        for (const sdpa_ctx::GuardRef& g : ctx->pending[p].guards)
            if (ring[g.shard][g.slot] == g.epoch) fired[p] = 1;
    if (ctx->world > L) {
        // one process per GPU: every process queued the same passes; a pass is repaired by all of them if any shard fired
        const NcclApi* api = nccl_api();
        if (!api) return SDPA_ERR_NCCL;
        Shard& s = ctx->shards[0];
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        DevBuf buf;
        SDPA_TRY(buf.reserve(fired.size() * sizeof(int), true));
        SDPA_CUDA_TRY(cudaMemcpyAsync(buf.p, fired.data(), fired.size() * sizeof(int), cudaMemcpyHostToDevice, s.s_comm));
        SDPA_NCCL_TRY(api->AllReduce(buf.p, buf.p, fired.size(), ncclInt32, ncclMax, s.comm, s.s_comm));
        SDPA_CUDA_TRY(cudaMemcpyAsync(fired.data(), buf.p, fired.size() * sizeof(int), cudaMemcpyDeviceToHost, s.s_comm));
        SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_comm));
        buf.release();
    }
    std::vector<sdpa_ctx::PendingPass> todo;
    for (size_t p = 0; p < ctx->pending.size(); ++p)
        if (fired[p]) todo.push_back(ctx->pending[p]);
    ctx->pending.clear();
    ctx->ring_use = 0;
    if (todo.empty()) return SDPA_OK;
    ctx->repairing = true;
    for (Shard& s : ctx->shards) umma_plan_force_exact(s.plan, true);
    sdpa_status st = SDPA_OK;
    for (sdpa_ctx::PendingPass& p : todo) {
        st = device_pass(ctx, p.dtype, p.K.data(), p.V.data(), p.n_local.data(), p.dk, p.dv, p.Q.data(), p.result, p.m, true,
                         "sdpa_synchronize (repair)");
        if (st != SDPA_OK) break;
    }
    for (Shard& s : ctx->shards) umma_plan_force_exact(s.plan, false);
    ctx->repairing = false;
    return st;
}

sdpa_status sdpa_synchronize(sdpa_ctx* ctx)
{
    if (!ctx) {
        set_error("sdpa_synchronize: ctx is NULL");
        return SDPA_ERR_INVALID;
    }
    SDPA_TRY(drain_exchange(ctx));
    for (Shard& s : ctx->shards) {
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));
    }
    ctx->queued_results.clear();
    return resolve_pending(ctx);   // collective when the context spans several processes
}

sdpa_status sdpa_online_softmax_partials(sdpa_ctx* ctx, int local, const float* Qf_dev, int m, float* contrib_dev,
                                         float* lmax_dev, float* lsum_dev)
{
    if (!ctx || local < 0 || local >= (int)ctx->shards.size() || m < 0) {
        set_error("sdpa_online_softmax_partials: bad arguments");
        return SDPA_ERR_INVALID;
    }
    if (ctx->dk == 0 || ctx->prec != SDPA_PREC_F32 || ctx->zero_copy) {
        set_error("sdpa_online_softmax_partials needs a resident fp32 K/V shard (precision f32)");
        return SDPA_ERR_INVALID;
    }
    if (m == 0) return SDPA_OK;
    Shard& s = ctx->shards[local];
    SDPA_CUDA_TRY(cudaSetDevice(s.dev));
    int splits = ctx->cfg.kv_splits > 0 ? ctx->cfg.kv_splits : attn_f32_pick_splits(m, s.n_local, s.sm_count);
    splits = std::max(1, std::min(splits, 64));
    SDPA_TRY(s.part_o.reserve((size_t)splits * m * ctx->dv * sizeof(float)));
    SDPA_TRY(s.part_tmax.reserve((size_t)splits * m * sizeof(float)));
    SDPA_TRY(s.part_lsum.reserve((size_t)splits * m * sizeof(float)));
    Partials part{s.part_o.as<float>(), s.part_tmax.as<float>(), s.part_lsum.as<float>(), splits, m};
    SDPA_TRY(launch_attn_f32(Qf_dev, s.Kc.as<float>(), s.Vc.as<float>(), m, s.n_local, ctx->dk, ctx->dv, splits, part,
                             nullptr, s.s_compute));
    SDPA_TRY(launch_merge_splits(part, m, ctx->dv, nullptr, contrib_dev, lmax_dev, lsum_dev, true, s.s_compute));
    SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));
    return SDPA_OK;
}

sdpa_status sdpa_scatter_attention(sdpa_ctx* ctx, const double* Q, const double* K, const double* V, double* result,
                                   int m, int n, int dk, int dv)
{
    return scatter_attention_impl(ctx, Q, K, V, result, m, n, dk, dv);
}

sdpa_status sdpa_last_timings(sdpa_ctx* ctx, float* out6)
{
    if (!ctx || !out6) {
        set_error("sdpa_last_timings: bad arguments");
        return SDPA_ERR_INVALID;
    }
    if (!ctx->last_timing_valid) {
        for (int k = 0; k < 4; ++k) ctx->last_timing[k] = 0.f;
        for (Shard& s : ctx->shards) {
            SDPA_CUDA_TRY(cudaSetDevice(s.dev));
            SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_compute));   // queued passes (sdpa_enqueue_*) must have finished
            SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_comm));
            const int slot[4] = {3, 0, 1, 2};   // out[0] total, [1] casts, [2] fused, [3] merge
            for (int k = 0; k < 4; ++k) {
                double ms = 0.0;
                SDPA_TRY(sum_pairs(s, slot[k], s.tpair_last[slot[k]], &ms));
                ctx->last_timing[k] = std::max(ctx->last_timing[k], (float)ms);
            }
        }
        ctx->last_timing_valid = true;
    }
    memcpy(out6, ctx->last_timing, sizeof(ctx->last_timing));
    return SDPA_OK;
}

/* Device time summed over every sdpa_attention_* call since the last reset, evaluated now (no host work is spent
 * on timing inside the calls): out[0] total, [1] casts, [2] fused kernel(s), [3] merge, [4] fused launches, [5] calls. */
sdpa_status sdpa_accumulated_timings(sdpa_ctx* ctx, double* out6, int reset)
{
    if (!ctx || !out6) {
        set_error("sdpa_accumulated_timings: bad arguments");
        return SDPA_ERR_INVALID;
    }
    float last[6];
    SDPA_TRY(sdpa_last_timings(ctx, last));   // keep the last call's detail before the events are recycled
    for (int k = 0; k < 6; ++k) out6[k] = 0.0;
    for (Shard& s : ctx->shards) {
        SDPA_TRY(fold_timings(s));
        const int slot[4] = {3, 0, 1, 2};
        for (int k = 0; k < 4; ++k) out6[k] = std::max(out6[k], s.acc_ms[slot[k]]);
        if (reset) for (int w = 0; w < 4; ++w) s.acc_ms[w] = 0.0;
    }
    out6[4] = ctx->acc_fused_launches;
    out6[5] = ctx->acc_calls;
    if (reset) ctx->acc_fused_launches = ctx->acc_calls = 0;
    return SDPA_OK;
}

const char* sdpa_last_kernel(sdpa_ctx* ctx) { return ctx ? ctx->last_kernel : "none"; }

/* Untimed preparation of a context, the analogue of what MPI_Init does for the reference before its timed region
 * (mpi.c:504,519): fill the memory pool of every local GPU with `pool_bytes` (later allocations become pool hits), load the
 * kernels (CUDA loads a kernel's code lazily at its first launch), start the host staging pool. */
sdpa_status sdpa_ctx_prewarm(sdpa_ctx* ctx, size_t pool_bytes)
{
    if (!ctx) {
        set_error("sdpa_ctx_prewarm: ctx is NULL");
        return SDPA_ERR_INVALID;
    }
    for (Shard& s : ctx->shards) {
        SDPA_CUDA_TRY(cudaSetDevice(s.dev));
        if (mem_pool_enabled() && pool_bytes > 0) {
            void* p = nullptr;
            if (cudaMallocAsync(&p, pool_bytes, cudaStreamPerThread) == cudaSuccess) {
                cudaMemsetAsync(p, 0, pool_bytes, cudaStreamPerThread);   // touch: the physical pages are mapped now
                cudaFreeAsync(p, cudaStreamPerThread);
            }
            cudaStreamSynchronize(cudaStreamPerThread);
            cudaGetLastError();
        }
        preload_cast_kernels();
        preload_merge_kernels();
        preload_attn_f32_kernels();
        preload_attn_umma_kernels();
    }
    host_staging_warm();
    return SDPA_OK;
}

/* MAX of a double over every process of the context (mpi.c:524); collective. */
sdpa_status sdpa_ctx_max(sdpa_ctx* ctx, double* value)
{
    if (!ctx || !value) {
        set_error("sdpa_ctx_max: bad arguments");
        return SDPA_ERR_INVALID;
    }
    if (ctx->world == (int)ctx->shards.size()) return SDPA_OK;   // one process: nothing to reduce over
    const NcclApi* api = nccl_api();
    if (!api) return SDPA_ERR_NCCL;
    Shard& s = ctx->shards[0];
    if (!s.comm) {
        set_error("sdpa_ctx_max: the context has no communicator");
        return SDPA_ERR_INVALID;
    }
    SDPA_CUDA_TRY(cudaSetDevice(s.dev));
    SDPA_TRY(s.gsum[0].reserve(256));
    SDPA_CUDA_TRY(cudaMemcpyAsync(s.gsum[0].p, value, sizeof(double), cudaMemcpyHostToDevice, s.s_comm));
    SDPA_NCCL_TRY(api->AllReduce(s.gsum[0].p, s.gsum[0].p, 1, ncclFloat64, ncclMax, s.comm, s.s_comm));
    SDPA_CUDA_TRY(cudaMemcpyAsync(value, s.gsum[0].p, sizeof(double), cudaMemcpyDeviceToHost, s.s_comm));
    SDPA_CUDA_TRY(cudaStreamSynchronize(s.s_comm));
    return SDPA_OK;
}

unsigned long long sdpa_launch_count(void) { return sdpa::launch_count(); }

sdpa_status sdpa_cvt_d2f(float* dst_dev, const double* src_dev, size_t count, void* stream)
{
    return launch_cvt_d2f(dst_dev, src_dev, count, (cudaStream_t)stream);
}
sdpa_status sdpa_cvt_f2d(double* dst_dev, const float* src_dev, size_t count, void* stream)
{
    return launch_cvt_f2d(dst_dev, src_dev, count, (cudaStream_t)stream);
}
sdpa_status sdpa_cvt_d2bf16(uint16_t* dst_dev, const double* src_dev, size_t count, void* stream)
{
    return launch_cvt_d2bf16(reinterpret_cast<__nv_bfloat16*>(dst_dev), src_dev, count, (cudaStream_t)stream);
}
sdpa_status sdpa_cvt_d2bf16x2(uint16_t* hi_dev, uint16_t* lo_dev, const double* src_dev, size_t count, void* stream)
{
    return launch_cvt_d2bf16x2(reinterpret_cast<__nv_bfloat16*>(hi_dev), reinterpret_cast<__nv_bfloat16*>(lo_dev), src_dev, count,
                               (cudaStream_t)stream);
}

}  // extern "C"
