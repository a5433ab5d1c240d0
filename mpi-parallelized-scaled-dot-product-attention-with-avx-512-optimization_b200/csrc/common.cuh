// common.cuh -- shared declarations of the sdpa_b200 engine (host + device).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stddef.h>
#include <stdio.h>
#include <string>

#include "../../include/sdpa_b200.h"

namespace sdpa {

// ---- error plumbing -------------------------------------------------------
void set_error(const char* fmt, ...);
const char* get_error();

#define SDPA_CUDA_TRY(expr)                                                          \
    do {                                                                             \
        cudaError_t _e = (expr);                                                     \
        if (_e != cudaSuccess) {                                                     \
            ::sdpa::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,          \
                              cudaGetErrorString(_e));                               \
            return SDPA_ERR_CUDA;                                                    \
        }                                                                            \
    } while (0)

#define SDPA_TRY(expr)                                                               \
    do {                                                                             \
        sdpa_status _s = (expr);                                                     \
        if (_s != SDPA_OK) return _s;                                                \
    } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// process-wide count of kernels this library has launched (bench.py reports it as gpu_launches)
void count_launch(int n = 1);
unsigned long long launch_count();

// ---- partial softmax state -------------------------------------------------
// One fused-kernel launch covers `rows` query rows against `splits` contiguous
// key ranges of the resident shard and leaves, per (split,row):
//   o    [split][row][dv]  un-normalised  sum_j 2^(t_j - tmax) V_j
//   tmax [split][row]      running max of t_j = (q.k_j) * scale * log2(e)   (log2 domain)
//   lsum [split][row]      sum_j 2^(t_j - tmax)
// tmax * ln2 is the reference's lmax (mpi.c:188); lsum is identical.
struct Partials {
    float* o;
    float* tmax;
    float* lsum;
    int splits;
    int rows_capacity;
};

// ---- kernel launchers (each returns after enqueueing on `stream`) ----------
sdpa_status launch_cvt_d2f(float* dst, const double* src, size_t count, cudaStream_t stream);
sdpa_status launch_cvt_f2d(double* dst, const float* src, size_t count, cudaStream_t stream);
sdpa_status launch_cvt_d2bf16(__nv_bfloat16* dst, const double* src, size_t count, cudaStream_t stream);
// fp64 -> (hi, lo) bf16 pair of the split precision SDPA_PREC_BF16X3: hi = bf16(fp32(x)), lo = bf16(fp32(x) - hi)
sdpa_status launch_cvt_d2bf16x2(__nv_bfloat16* dst_hi, __nv_bfloat16* dst_lo, const double* src, size_t count, cudaStream_t stream);
struct CastBatch {
    void* dst[3];
    const void* src[3];   // element type: the launch's source dtype
    size_t units[3];   // 2-element units per segment
    size_t lo_off[3];  // split precision: distance from the hi to the lo array, in 2-element units
    unsigned long long* trace;   // developer aid (background form): per CTA [start, end] %globaltimer stamps, or NULL
};
// Developer aid: where the background cast kernel leaves its per-CTA stamps (NULL = off), and a one-thread kernel that
// stamps %globaltimer into *dst in stream order.
void set_cast_trace(unsigned long long* buf);
sdpa_status launch_stamp(unsigned long long* dst, cudaStream_t stream);
// src_dtype: sdpa_dtype of the sources (fp64, fp32 or bf16); prec: the compute precision written.
// lo_off (elements, per segment) is read for SDPA_PREC_BF16X3 only and may be NULL otherwise.
sdpa_status launch_cvt_in_batch(int src_dtype, int prec, void* const* dst, const void* const* src, const size_t* count,
                                const size_t* lo_off, int nseg, cudaStream_t stream, int background_ctas = 0);
// background_ctas > 0 (fp64 sources only): the small-footprint form (that many CTAs of 128 threads, 40 KB of shared memory,
// <= 32 registers) that fits on an SM beside a resident CTA of the persistent fused kernel.

// fp32 CUDA-core fused attention.  Q [rows x dk], K [n x dk], V [n x dv] fp32 row-major.
// If out64 != nullptr (requires splits == 1) the normalised result is written as fp64
// and no partials are produced.
sdpa_status launch_attn_f32(const float* Q, const float* K, const float* V, int rows, int n, int dk,
                            int dv, int splits, Partials part, double* out64, cudaStream_t stream);
bool attn_f32_supported(int dk, int dv);
int attn_f32_pick_splits(int rows, int n, int sm_count);

// tcgen05 fused attention (attn_umma_bf16.cu: dk = dv = 128 bf16; attn_umma_general.cu: every other shape and the
// split precision).  Q, K [.. x dk], V [n x dv] bf16 row-major.
struct UmmaPlan;  // holds the TMA descriptors for one (Q buffer, K/V shard) binding
sdpa_status umma_plan_create(UmmaPlan** plan);
void umma_plan_destroy(UmmaPlan* plan);
// hl = 1: bf16 operands; hl = 2: hi/lo split (the lo array of an operand starts *_lo_off ELEMENTS behind its hi array).
sdpa_status umma_plan_bind_kv(UmmaPlan* plan, const __nv_bfloat16* K, const __nv_bfloat16* V, int n,
                              int dk, int dv, int hl, size_t k_lo_off, size_t v_lo_off);
sdpa_status umma_plan_bind_q(UmmaPlan* plan, int slot, const __nv_bfloat16* Q, int rows_capacity, int dk, int hl,
                             size_t q_lo_off);
sdpa_status launch_attn_umma(UmmaPlan* plan, int q_slot, int rows, int splits, Partials part,
                             double* out64, int sm_count, cudaStream_t stream);
// Overflow-guard ring of a plan: launch epoch e owns word e % kGuardRing; the word equals e iff that launch raised its guard.
constexpr unsigned int kGuardRing = 4096;
void umma_plan_last_guard(const UmmaPlan* plan, unsigned int* slot, unsigned int* epoch);
const unsigned int* umma_plan_guard_ring(const UmmaPlan* plan);
void umma_plan_force_exact(UmmaPlan* plan, bool on);   // the next launches run the exact variant alone (host-side repair)
// the exact two-phase variant behind the fast launch above (exits at once unless its overflow guard fired)
sdpa_status launch_attn_umma_twin(UmmaPlan* plan, int q_slot, int rows, int splits, Partials part, double* out64, cudaStream_t stream);
bool attn_umma_supported(int dk, int dv, int hl);
int attn_umma_pick_splits(int rows, int n, int sm_count);
// Persistent fused kernel (EXPERIMENTAL, SDPA_UMMA_V8=1): partial slots per row block for (rows, n), 0 = not applicable.
struct WorkMap;
int attn_umma_v8_pieces(int rows, int n, int sm_count);
void umma_plan_allow_v8(UmmaPlan* plan, bool allow);   // the caller will merge with launch_merge_pieces
bool umma_plan_last_v8(const UmmaPlan* plan, WorkMap* wm, int* max_pieces, const unsigned int** guard, unsigned int* epoch);

// Merge of partial states (the arithmetic of mpi.c:340-362 in the log2 domain).
//   mode FINAL   : out64[row][d] = sum_s o_s w_s / sum_s lsum_s w_s     (gsum==0 -> 0)
//   mode PARTIAL : contrib/tmax/lsum of the merged state, un-normalised (feeds the cross-GPU merge)
//   mode PUBLIC  : like PARTIAL but lmax is converted to the reference's natural-log units
// Exchange-slot hand-over of one shard, fused into its split merge: wait until *wait_flag >= wait_epoch (the root has
// consumed what the slot held; NULL = nothing to wait for), merge into the slot, release *flag = epoch (state published).
struct PublishSync {
    const unsigned int* wait_flag = nullptr;
    unsigned int wait_epoch = 0;
    unsigned int* flag = nullptr;
    unsigned int epoch = 0;
    unsigned int* block_counter = nullptr;   // local scratch word
    unsigned long long* trace = nullptr;
};
sdpa_status launch_merge_splits(Partials part, int rows, int dv, double* out64, float* contrib,
                                float* tmax_out, float* lsum_out, bool natural_log_max,
                                cudaStream_t stream, const PublishSync* publish = nullptr);
// Cross-shard steps of the NCCL merge (mpi.c:346-351 and mpi.c:358-362).
sdpa_status launch_rescale_to_gmax(float* contrib, float* lsum, const float* tmax, const float* gmax,
                                   int rows, int dv, cudaStream_t stream);
sdpa_status launch_normalize(float* contrib, const float* gsum, int rows, int dv, cudaStream_t stream);
// out64[row][d] = reduced[row][d] / gsum[row]  (gsum == 0 -> 0): normalise + fp32->fp64 after the single SUM reduce
sdpa_status launch_finalize_reduced(double* out64, const float* reduced, const float* gsum, int rows, int dv,
                                    cudaStream_t stream);
// Fused device-side exchange: root reads every shard's (contrib,tmax,lsum) through peer pointers.
sdpa_status launch_merge_peers(const float* const* contrib_ptrs, const float* const* tmax_ptrs,
                               const float* const* lsum_ptrs, int shards, int rows, int dv,
                               double* out64, cudaStream_t stream);


// ---- device-side exchange across processes (CUDA IPC peer memory + flags in device memory) ----------
// A flag holds the epoch (global batch counter) of the last completed step.
sdpa_status launch_signal_flag(unsigned int* flag, unsigned int epoch, cudaStream_t stream,
                               unsigned long long* trace = nullptr);                                // release-store after prior work
sdpa_status launch_wait_flag(const unsigned int* flag, unsigned int epoch, cudaStream_t stream);   // spin until *flag >= epoch
sdpa_status set_flag_timeout_seconds(double seconds);   // bound of those spins on the current device (default 120 s)
struct PeerSync {
    const unsigned int* ready[64];   // per shard: its "state of epoch e is complete" flag (local or IPC-mapped)
    unsigned int* consumed;          // root-local: set to epoch once every block has merged (peers poll it before reuse)
    unsigned int* block_counter;     // root-local scratch
    unsigned int epoch;
    unsigned long long* trace = nullptr;   // SDPA_EXCHANGE_TRACE: 4 x u64 of this epoch (see merge_kernels.cu)
};
// Root GPU: wait for every shard's flag, merge their (contrib,tmax,lsum) read through peer pointers, write fp64.
sdpa_status launch_merge_peers_synced(const float* const* contrib_ptrs, const float* const* tmax_ptrs,
                                      const float* const* lsum_ptrs, int shards, int rows, int dv, double* out64,
                                      const PeerSync& sync, cudaStream_t stream);
// Root GPU, push form: merge the `world` states the shards have pushed into the root's local inbox (segment r at r * seg_floats:
// [o cap_rows*dv | tmax cap_rows | lsum cap_rows]) once ready[r] >= epoch for every r; write fp64 rows; release `consumed[r]`
// (every rank's own flag word) = epoch.  Small-footprint kernel (`ctas` CTAs x 128 threads, <= 32 registers): runs beside
// the persistent fused kernel of the next queued pass.
sdpa_status launch_merge_inbox_background(const float* inbox, size_t seg_floats, int cap_rows, int world, const unsigned int* ready,
                                          unsigned int* const* consumed, unsigned int* block_counter, unsigned int epoch,
                                          unsigned long long* trace, int rows, int dv, double* out64, int ctas, cudaStream_t stream);
// Root GPU, in-stream cross-GPU merge: own partial states (pieces if wm != NULL, else part.splits) + the peers' published states.
sdpa_status launch_merge_root_instream(Partials part, const WorkMap* wm, int max_pieces, const unsigned int* guard, unsigned int guard_epoch,
                                       const float* const* peer_c, const float* const* peer_t, const float* const* peer_l, int npeers,
                                       int rows, int dv, double* out64, const PeerSync& sync, cudaStream_t stream);
// Split merge behind the persistent fused kernel: per row, wm_pieces(row block) states (all max_pieces if *guard == epoch).
// out64 != NULL: normalised fp64 rows; else the merged un-normalised state (contrib, tmax, lsum) for the cross-GPU merge.
sdpa_status launch_merge_pieces(Partials part, const WorkMap& wm, int max_pieces, int rows, int dv, double* out64, float* contrib,
                                float* tmax_out, float* lsum_out, const unsigned int* guard, unsigned int epoch, cudaStream_t stream,
                                const PublishSync* publish = nullptr);
// Sliced merge, source side: merge the split states of `rows` rows and write each row's state into the inbox segment of
// the rank owning its slice (slice r = rows/world + (r < rows%world) consecutive rows), then raise flag[r] = epoch at every rank.
struct RouteTargets {
    float* o[64];
    float* tmax[64];
    float* lsum[64];
    unsigned int* flag[64];
    unsigned int* block_counter;   // local scratch
    unsigned int epoch;
    int world;
};
// wm != NULL: the partials come from the persistent fused kernel (pieces per row block, see launch_merge_pieces)
sdpa_status launch_merge_splits_routed(Partials part, int rows, int dv, const RouteTargets& to, cudaStream_t stream, const WorkMap* wm = nullptr,
                                       int max_pieces = 0, const unsigned int* guard = nullptr, unsigned int guard_epoch = 0);
// Sliced merge, root side: wait for every rank's "my rows are staged" flag (sync.ready), copy the staged fp64 batch
// to dst, then raise sync.consumed.
sdpa_status launch_collect_slices(double* dst, const double* staged, int rows, int dv, const PeerSync& sync, int ranks,
                                  cudaStream_t stream);

// Work decomposition of the persistent fused kernel (attn_umma_kernel_v8): the linear space (row block of 256 rows, key
// tile) has W = RB*T units; cluster c of C owns units [c*W/C, (c+1)*W/C).  A row block is therefore cut into
// wm_pieces(rb) consecutive pieces, piece p computed by cluster wm_cluster_of(rb*T) + p and stored in partial slot p.
struct WorkMap {
    int T;    // key tiles per row block
    int C;    // clusters (CTA pairs) in the grid
    int RB;   // row blocks of 256 rows
};
__host__ __device__ inline long long wm_total(const WorkMap& w) { return (long long)w.RB * w.T; }
__host__ __device__ inline long long wm_begin(const WorkMap& w, int c) { return (long long)c * wm_total(w) / w.C; }
// the cluster whose range contains `unit`: the largest c with floor(c*W/C) <= unit
__host__ __device__ inline int wm_cluster_of(const WorkMap& w, long long unit)
{
    const long long W = wm_total(w);
    return (int)(((unit + 1) * w.C + W - 1) / W) - 1;
}
__host__ __device__ inline int wm_pieces(const WorkMap& w, int rb)
{
    return wm_cluster_of(w, (long long)(rb + 1) * w.T - 1) - wm_cluster_of(w, (long long)rb * w.T) + 1;
}

// Force the (lazily loaded) kernels of each translation unit onto the current device: cudaFuncGetAttributes loads the function.
void preload_cast_kernels();
void preload_merge_kernels();
void preload_attn_f32_kernels();
void preload_attn_umma_kernels();
void host_staging_warm();   // pinned ring + copy threads of the pageable-source path, ahead of the first timed call

// host_staging.cu: host -> device copies that run at the pinned rate for pageable sources too (pinned ring + copy threads)
bool host_ptr_is_pageable(const void* p);
sdpa_status h2d_any(void* dst_dev, const void* src_host, size_t bytes, cudaStream_t stream);
int host_staging_lanes();

}  // namespace sdpa
