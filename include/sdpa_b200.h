/*
 * sdpa_b200.h -- C ABI of the B200-native scaled-dot-product-attention engine.
 *
 * This library is a drop-in for the hot path of
 * lynchu/MPI-parallelized-Scaled-Dot-Product-Attention-with-AVX-512-optimization:
 * the body of attention() in attention-mpi.c:191-407 (K/V row sharding, fp64->fp32
 * casts, per-row online softmax attention, the MAX/SUM/SUM merge, fp32->fp64
 * write-back).  Everything is plain C: pointers, ints and sizes, no C++ or torch
 * types.  Citations below are reference file:line ("mpi.c" = attention-mpi.c,
 * "ser.c" = attention.c).
 *
 * Error model.  The reference entry point is `void` and its harness treats every
 * fatal condition as fprintf(stderr)+exit(1) (mpi.c:419-422,436-448); the drop-in
 * attention() below keeps that behaviour.  Every other function returns an
 * sdpa_status and leaves a message retrievable with sdpa_last_error().
 * There is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef SDPA_B200_H
#define SDPA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum sdpa_status {
    SDPA_OK = 0,
    SDPA_ERR_INVALID = 1,     /* bad argument / unsupported shape              */
    SDPA_ERR_CUDA = 2,        /* CUDA runtime or driver error                  */
    SDPA_ERR_NCCL = 3,        /* NCCL error or NCCL not loadable               */
    SDPA_ERR_UNSUPPORTED = 4, /* shape/precision combination has no kernel     */
    SDPA_ERR_NOMEM = 5
} sdpa_status;

/* Arithmetic of the fused QK^T -> softmax -> .V kernel. */
typedef enum sdpa_precision {
    SDPA_PREC_AUTO = 0,  /* fp32-class accuracy, like the reference (mpi.c:168-189): BF16X3 where that kernel takes the shape,
                            else F32.  Never BF16 for fp64 / fp32 operands: the reference's 0.02 gate (mpi.c:476) must hold on
                            peaky inputs.  bf16 operands (typed passes): BF16 where it takes the shape, else F32           */
    SDPA_PREC_F32 = 1,   /* fp32 CUDA-core kernel: the reference's own arithmetic; any dk, dv <= 256                        */
    SDPA_PREC_BF16 = 2,  /* opt-in: bf16 operands, fp32 accumulate, tcgen05; dk, dv multiples of 8 up to 256                */
    SDPA_PREC_BF16X3 = 3 /* fp32 operands split into bf16 hi + lo, three tcgen05.mma per contraction into one fp32
                            accumulator (<= 1e-5 on N(0,1) inputs); dk, dv multiples of 8 with dk <= 128 and dv <= 128, or
                            dk <= 64 and dv <= 256 (what fits the 227 KiB of shared memory)                                */
} sdpa_precision;

/* Element type of the device arrays of a typed pass (sdpa_attention_device_typed); the result has the same type. */
typedef enum sdpa_dtype {
    SDPA_DTYPE_F64 = 0,  /* the reference's own operands: the same pass as sdpa_attention_device_full                         */
    SDPA_DTYPE_F32 = 1,
    SDPA_DTYPE_BF16 = 2  /* raw bfloat16 (1 sign, 8 exponent, 7 mantissa bits), e.g. torch.bfloat16                            */
} sdpa_dtype;

/* How the per-shard softmax states are merged across GPUs (mpi.c:340-380). */
typedef enum sdpa_merge {
    SDPA_MERGE_NCCL = 0, /* allreduce(MAX), allreduce(SUM), reduce(SUM): the reference's three collectives */
    SDPA_MERGE_PEER = 1, /* fused device-side exchange over NVLink peer memory: one process driving several GPUs (peer
                            access), or one process per GPU (slots and flags shared through CUDA IPC)                */
    SDPA_MERGE_NCCL2 = 2 /* same arithmetic in two collectives: allreduce(MAX), then ONE reduce(SUM) over
                            [contrib | lsum] with the normalisation + fp64 cast fused after it (default)   */
} sdpa_merge;

/* How one process spreads the problem over its GPUs -- the GPU analogue of the reference's Bcast-vs-Scatterv
 * switch for K/V (mpi.c:213-215).  Applies to sdpa_load_kv_host_full / attention() with num_local > 1. */
typedef enum sdpa_distribution {
    SDPA_DIST_KV = 0,  /* K/V rows sharded by owner_count/owner_disp, Q replicated, one exchange per batch (the reference's way) */
    SDPA_DIST_Q = 1,   /* K/V replicated on every GPU, Q rows sharded, no exchange: pays when n is small                        */
    SDPA_DIST_AUTO = 2 /* DIST_Q when n*(dk+dv)*4 bytes < 64 MiB (the reference's own threshold), else DIST_KV                  */
} sdpa_distribution;

typedef struct sdpa_config {
    int precision;   /* sdpa_precision                                              */
    int q_batch;     /* Q rows per ping-pong batch (reference: B=512, mpi.c:200); 0 = engine default */
    int kv_splits;   /* split-KV factor inside one GPU; 0 = auto (fill the 148 SMs) */
    int merge;       /* sdpa_merge                                                  */
    int num_local;   /* GPUs driven by THIS process (K/V shards it owns); 0 = 1     */
    int first_device;/* CUDA ordinal of the first local GPU                         */
    int world_size;  /* total K/V shards over all processes; 0 = num_local          */
    int rank_base;   /* global shard index of this process's first local GPU        */
    int distribution;/* sdpa_distribution (single-process contexts)                 */
    int reserved[7];
} sdpa_config;

typedef struct sdpa_ctx sdpa_ctx;

/* Whether a kernel exists for (precision, dk, dv); for SDPA_PREC_AUTO always 1 when dk, dv are in [1, 256], and
 * *resolved (may be NULL) receives the precision AUTO selects.  Pure host function; usable without a GPU. */
int sdpa_precision_supported(int precision, int dk, int dv, int* resolved);
/* The same for operands of element type `dtype` (sdpa_dtype).  fp64 and fp32 operands: the rule above.  bf16 operands: AUTO
 * resolves to BF16 where the bf16 tensor-core kernel takes (dk, dv), else F32 -- the operands are already rounded to bf16 by
 * the caller, so the operand rounding that keeps plain bf16 out of AUTO for fp64 / fp32 operands does not arise; what remains
 * is the bf16 rounding of the softmax weights P (<= 2e-3 on N(0,1) inputs).  Pure host function; usable without a GPU. */
int sdpa_precision_supported_for(int dtype, int precision, int dk, int dv, int* resolved);

/* ---------------------------------------------------------------------------
 * 1. The reference entry point (replaces mpi.c:191-192; the serial flavour
 *    ser.c:20-21 is the same call with mpi_rank=0, mpi_size=1).
 *
 *    Q [m x dk], K [n x dk], V [n x dv], result [m x dv]: dense row-major fp64
 *    host arrays, valid on rank 0 only (mpi.c:508-517); m,n,dk,dv are taken from
 *    rank 0 (mpi.c:193-197).  Blocking; result is complete on return on rank 0.
 *    The caller keeps ownership of all four buffers; inputs are not modified.
 *
 *    mpi_size == 1 : one process drives SDPA_NGPUS GPUs (env, default 1); K/V rows
 *                    are sharded over them with owner_count/owner_disp.
 *    mpi_size  > 1 : one process per GPU.  The NCCL communicator is bootstrapped
 *                    from sdpa_set_bootstrap_id() (a launcher with MPI broadcasts
 *                    the id, see INTEGRATION.md) or, failing that, from the file
 *                    named by env SDPA_NCCL_ID_FILE.  Rank 0 scatters the shards.
 *    Precision / batch come from env SDPA_PRECISION (auto|f32|bf16|bf16x3), SDPA_Q_BATCH.
 *    Fatal errors: message on stderr, exit(1).
 * ------------------------------------------------------------------------- */
void attention(double* Q, double* K, double* V, double* result,
               int m, int n, int dk, int dv, int mpi_rank, int mpi_size);

/* Creates the context attention() will use (CUDA contexts, streams, NCCL communicator)
 * ahead of the first call: the analogue of MPI_Init (mpi.c:504), which the reference also
 * keeps outside its timed region (mpi.c:519-522).  Optional. */
sdpa_status sdpa_runtime_init(int mpi_rank, int mpi_size);
void sdpa_runtime_shutdown(void);
/* MAX over all ranks of *value, in place on every rank: the reference reports the slowest rank's elapsed time
 * (MPI_Reduce(MAX), mpi.c:524).  Uses the communicator of the runtime context; identity when mpi_size == 1. */
sdpa_status sdpa_runtime_max(double* value);

/* ---------------------------------------------------------------------------
 * 2. Shard map (replaces owner_count / owner_disp, mpi.c:19-27): balanced
 *    contiguous partition of n rows; the first n % size ranks own one more.
 *    Pure host functions; usable without a GPU.
 * ------------------------------------------------------------------------- */
int sdpa_owner_count(int n, int size, int rank);
int sdpa_owner_disp(int n, int size, int rank);

/* ---------------------------------------------------------------------------
 * 3. Context API: what attention() is built from, for callers that keep K/V
 *    resident, feed pre-sharded inputs, or time the path without file I/O.
 * ------------------------------------------------------------------------- */
void sdpa_config_init(sdpa_config* cfg);
/* nccl_id: 128-byte ncclUniqueId shared by all processes, or NULL when
 * world_size == num_local (single process).  */
sdpa_status sdpa_ctx_create(sdpa_ctx** out, const sdpa_config* cfg, const void* nccl_id);
sdpa_status sdpa_ctx_destroy(sdpa_ctx* ctx);
/* Writes a fresh 128-byte ncclUniqueId (rank 0 calls it, the launcher broadcasts it). */
sdpa_status sdpa_get_unique_id(void* out128);
/* Registers the id used by attention() when mpi_size > 1. */
sdpa_status sdpa_set_bootstrap_id(const void* id128);

/* K/V shard upload + cast (mpi.c:213-266: cvt_d2f of K,V then Bcast/Scatterv).
 * K_shards[i] / V_shards[i] are the rows owned by local GPU i
 * (n_local[i] x dk, n_local[i] x dv, fp64 row-major).  *_host: host memory
 * (pinned or pageable), blocking; *_device: already resident on that GPU, and stream-ordered: the
 * casts are queued and the arrays must stay untouched until the next sdpa_attention_* call returns. */
sdpa_status sdpa_load_kv_host(sdpa_ctx* ctx, const double* const* K_shards,
                              const double* const* V_shards, const int* n_local, int dk, int dv);
sdpa_status sdpa_load_kv_device(sdpa_ctx* ctx, const double* const* K_shards,
                                const double* const* V_shards, const int* n_local, int dk, int dv);
/* Convenience for a single process: full K [n x dk], V [n x dv] on the host, sharded
 * over the local GPUs with sdpa_owner_count / sdpa_owner_disp. */
sdpa_status sdpa_load_kv_host_full(sdpa_ctx* ctx, const double* K, const double* V, int n, int dk, int dv);

/* Attention of m query rows against the resident K/V (mpi.c:268-399: the
 * ping-pong Q-batch loop).  Q is replicated: the host variant reads one host
 * array; the device variant takes one fp64 device pointer per local GPU.
 * The result (m x dv fp64) is delivered on the process that owns global shard 0
 * (host array, or device pointer on its first GPU); other processes pass NULL. */
sdpa_status sdpa_attention_host(sdpa_ctx* ctx, const double* Q, double* result, int m);
sdpa_status sdpa_attention_device(sdpa_ctx* ctx, const double* const* Q_dev, double* result_dev, int m);

/* Pinned host memory for callers that choose their allocator (the harness does; replaces read_matrix's malloc,
 * attention-mpi.c:417-423).  Arrays from malloc work too: pageable sources are staged through a pinned ring by a small
 * pool of copy threads (SDPA_STAGING_THREADS, default cores/8 capped at 8; SDPA_HOST_STAGING=0 leaves it to the driver). */
void* sdpa_host_alloc(size_t bytes);
void sdpa_host_free(void* p);
/* The staging pool's multi-threaded memcpy by itself (no CUDA): returns the number of threads that took part. */
int sdpa_host_copy(void* dst, const void* src, size_t bytes);

/* load_kv_device + attention_device in one call (the whole attention() path on device-resident fp64). */
sdpa_status sdpa_attention_device_full(sdpa_ctx* ctx, const double* const* K_shards, const double* const* V_shards,
                                       const int* n_local, int dk, int dv, const double* const* Q_dev,
                                       double* result_dev, int m);

/* The same pass, queued instead of blocking: returns once the work is enqueued on the context's streams.  Consecutive
 * passes run back to back in stream order (they share the context's buffers), which removes the host round trip
 * between passes; every array must be complete when the call is made and stay valid and unmodified until
 * sdpa_synchronize() returns -- the K/V/Q of a queued pass may be read (cast to compute precision on a side stream) while
 * the PREVIOUS pass is still computing, and its result may not be read by the caller before sdpa_synchronize().  This is the form
 * bench.py times for the HBM-resident metric -- the blocking calls above keep the reference's semantics
 * (attention() returns with the result complete, attention-mpi.c:521-523). */
sdpa_status sdpa_enqueue_device_full(sdpa_ctx* ctx, const double* const* K_shards, const double* const* V_shards,
                                     const int* n_local, int dk, int dv, const double* const* Q_dev,
                                     double* result_dev, int m);
/* Waits for every queued pass.  It is also where a queued pass whose overflow guard fired is repaired (re-run with the exact
 * kernel variant; blocking calls carry that variant in the stream instead), so results are final on return -- which is why the
 * arrays of queued passes must stay valid until then.  On a context that spans several processes the call is collective. */
sdpa_status sdpa_synchronize(sdpa_ctx* ctx);

/* sdpa_attention_device_full / sdpa_enqueue_device_full on device arrays of element type `dtype` (sdpa_dtype): K/V shards,
 * Q and the result are dense row-major arrays of that type, the result (m x dv, root process only) too.  SDPA_DTYPE_F64 is
 * exactly the fp64 call.  The kernel follows sdpa_precision_supported_for(dtype, cfg.precision, dk, dv).  No fp64 copy is
 * made: the casts into compute precision read the caller's arrays, and where the arrays already are in compute precision
 * (bf16 operands at BF16, fp32 operands at F32) the fused kernel reads them in place and no cast runs at all -- which for the
 * tensor-core kernels needs K, V and Q 16-byte aligned (else SDPA_ERR_INVALID; nothing is copied to make up for it).  The
 * result is merged in fp64 and rounded once (round to nearest even) into `dtype`.  The queued form has the contract of
 * sdpa_enqueue_device_full: arrays valid and unmodified until sdpa_synchronize(), which also repairs its passes.  Typed
 * passes never cast ahead. */
sdpa_status sdpa_attention_device_typed(sdpa_ctx* ctx, int dtype, const void* const* K_shards, const void* const* V_shards,
                                        const int* n_local, int dk, int dv, const void* const* Q_dev, void* result_dev, int m);
sdpa_status sdpa_enqueue_device_typed(sdpa_ctx* ctx, int dtype, const void* const* K_shards, const void* const* V_shards,
                                      const int* n_local, int dk, int dv, const void* const* Q_dev, void* result_dev, int m);

/* The reference's calling convention on a one-GPU-per-process context (world_size > 1):
 * dimensions and Q/K/V/result are valid on the process that owns shard 0 only; that process
 * scatters the K/V shards and broadcasts the Q batches over NCCL (mpi.c:196,213-266,305,327). */
sdpa_status sdpa_scatter_attention(sdpa_ctx* ctx, const double* Q, const double* K, const double* V,
                                   double* result, int m, int n, int dk, int dv);

/* Per-shard partial softmax state, the contract of online_softmax_attention
 * (mpi.c:168-189) over a batch of rows: contrib [m x dv] un-normalised, lmax [m],
 * lsum [m], all fp32 device pointers on local GPU `local`; Qf is fp32 [m x dk] on
 * that GPU.  Uses the resident K/V shard.  Synchronous. */
sdpa_status sdpa_online_softmax_partials(sdpa_ctx* ctx, int local, const float* Qf_dev, int m,
                                         float* contrib_dev, float* lmax_dev, float* lsum_dev);

/* Device time (ms) of the stages of the last sdpa_attention_* call, max over
 * local GPUs: [0] total, [1] casts, [2] fused attention kernel(s),
 * [3] merge + collectives, [4] fused-kernel launches, [5] all kernel launches. */
sdpa_status sdpa_last_timings(sdpa_ctx* ctx, float* out6);
/* The same stage times summed over every sdpa_attention_* call since the last reset; the event queries happen
 * here, not inside the calls.  out6: [0] total, [1] casts, [2] fused, [3] merge (ms), [4] fused launches, [5] calls. */
sdpa_status sdpa_accumulated_timings(sdpa_ctx* ctx, double* out6, int reset);
/* Which kernel the last call used: "f32_simt" | "bf16_umma" | "bf16_umma_v8" | "bf16_umma_general" | "bf16x3_umma". */
const char* sdpa_last_kernel(sdpa_ctx* ctx);

/* ---------------------------------------------------------------------------
 * 4. The casts as standalone device operations (replace cvt_d2f_avx512
 *    mpi.c:31-64 and cvt_f2d_avx512 mpi.c:68-101).  Device pointers on the
 *    current device; `stream` is a cudaStream_t (NULL = default).  Asynchronous.
 * ------------------------------------------------------------------------- */
sdpa_status sdpa_cvt_d2f(float* dst_dev, const double* src_dev, size_t count, void* stream);
sdpa_status sdpa_cvt_f2d(double* dst_dev, const float* src_dev, size_t count, void* stream);
sdpa_status sdpa_cvt_d2bf16(uint16_t* dst_dev, const double* src_dev, size_t count, void* stream);
/* The operand split of SDPA_PREC_BF16X3: hi = bf16(fp32(x)), lo = bf16(fp32(x) - hi), both round-to-nearest-even. */
sdpa_status sdpa_cvt_d2bf16x2(uint16_t* hi_dev, uint16_t* lo_dev, const double* src_dev, size_t count, void* stream);

/* ---------------------------------------------------------------------------
 * 5. Diagnostics.
 * ------------------------------------------------------------------------- */
const char* sdpa_last_error(void);
const char* sdpa_version(void);
int sdpa_device_count(void);
/* Kernels launched by this library in this process so far (all GPUs). */
unsigned long long sdpa_launch_count(void); /* CUDA devices visible; 0 when there is none (never falls back to CPU) */

#ifdef __cplusplus
}
#endif
#endif /* SDPA_B200_H */
