// attn_umma_bf16.cu -- fused QK^T -> online softmax -> .V on the 5th-generation tensor cores (tcgen05.mma, accumulators in
// TMEM, operands staged by TMA) for the headline shape dk = dv = 128, bf16 operands / fp32 accumulate.
//
// The B200 counterpart of online_softmax_attention (attention-mpi.c:168-189): where the reference does one AVX-512 dot
// (dot_avx512, :103-121) and one axpy (axpy_avx512, :123-140) per (query, key) pair, these kernels do two 256x128x128
// tensor-core GEMMs per (256-query block, 128-key tile) pair; the running max / running sum of mpi.c:177-180 live in
// registers, one (query row, 64-key half) per thread.
//
// Two kernels behind one launcher (launch_attn_umma); both produce the same partial softmax state:
//   attn_umma_kernel_v8  the PERSISTENT kernel: one cluster per SM pair walks a contiguous range of (row block, key tile)
//                        units ("stream-K" over the key axis): no wave quantisation, one prologue per SM, 3-4 partial
//                        states per row block instead of 9.  Used whenever the caller merges by pieces (see its banner).
//   attn_umma_kernel_v7  the same pipeline as a plain grid (row block x split): small problems, explicit split counts.
// Common design (v7 banner): a cluster of two CTAs forms one M=256 tcgen05.mma.cta_group::2, each CTA keeps half of every
// K/V tile, S and P are double-buffered in TMEM (no MMA waits for the softmax of its own S), two softmax groups ping-pong
// over alternating key tiles.  The softmax reference is fixed by the first key tile of a range; scores that outgrow it by
// more than 2^64 raise a guard and the exact two-phase variant of the general kernel (attn_umma_general.cu) -- launched
// behind every fast launch, leaving at once unless the guard fired -- recomputes the launch.
// Every other shape (dk, dv multiples of 8 up to 256) and the fp32-accurate split precision: attn_umma_general.cu.
// History of the kernel generations (v1 ... v7, with measurements): profiles/README.md.
#include "umma_ptx.cuh"
#include "umma_general.h"

#include <type_traits>
#include <vector>
#include <stdlib.h>

namespace sdpa {

namespace {

using namespace umma;

constexpr int HEAD = 128;            // dk == dv
constexpr float kGuardThreshold = 64.0f;              // fast mode: exponents beyond 2^64 hand the launch to the safe kernel

struct KernelParams {
    int rows;            // valid Q rows
    int n;               // keys in the shard
    int tiles_total;     // ceil(n / 128)
    int splits;
    float scale_log2;    // 1/sqrt(dk) * log2(e)
    float* part_o;
    float* part_tmax;
    float* part_lsum;
    int rows_capacity;
    double* out64;       // non-null (splits == 1): normalised fp64 output
    long long* trace;    // TRACE build only: clock64 stamps of CTA (0,0), [role][iteration][event]
    unsigned int* guard; // fast mode writes `epoch` here when an exponent would overflow; the safe kernel runs iff *guard == epoch
    unsigned int epoch;
    WorkMap wm;          // v8 only: the persistent kernel's work decomposition
};

constexpr int TRACE_ITERS = 24, TRACE_EVENTS = 8, TRACE_ROLES = 6;

// (v6 -- the cluster-of-two, multicast stepping stone between v5 and v7 -- was removed in round 2: measured slower than both,
//  profiles/README.md keeps its numbers.)
constexpr uint32_t V6_S = 0, V6_O = 256, V6_P = 384;   // TMEM map of the chain-free kernels: S0 S1 | O | P0 P1

// =====================================================================================
// v7: v6 with the 2-CTA tensor-core instruction (tcgen05.mma.cta_group::2).  The two CTAs of a cluster
// form ONE M=256 MMA: each holds its own 128-row Q tile (A) and its own accumulators/P in its TMEM, and
// each keeps only HALF of every K tile (64 keys) and V tile (64 value columns) in shared memory -- the
// B operand is split across the pair -- so per SM the shared-memory traffic per key tile drops from
// 160 KB (v6) to 96 KB and no multicast is needed.  Only the leader CTA (cluster rank 0) issues MMAs;
// its barriers collect both CTAs' TMA bytes (2-SM TMA form: the mbarrier address is mapped to the
// leader) and both CTAs' softmax arrivals (remote mbarrier.arrive through mapa); tcgen05.commit
// multicasts completions to both CTAs.
// =====================================================================================
constexpr int V7_KSTAGES = 4, V7_VSTAGES = 3;
constexpr uint32_t HALF_TILE_BYTES = TILE_BYTES / 2;   // 64 keys x 128 (K half) or 128 keys x 64 columns (V half)

struct __align__(1024) SharedV7 {
    uint8_t q[TILE_BYTES];
    uint8_t k[V7_KSTAGES][HALF_TILE_BYTES];
    uint8_t v[V7_VSTAGES][HALF_TILE_BYTES];
    uint64_t q_full;
    uint64_t k_full[V7_KSTAGES], k_empty[V7_KSTAGES];
    uint64_t v_full[V7_VSTAGES], v_empty[V7_VSTAGES];
    uint64_t s_full[2], p_ready[2], s_free[2], pv_done[2], o_done;
    uint32_t tmem_base;
    float xchg[2][4][TILE];   // [first-tile max | final sum][group*NPARTS + part][row]
    float mref[TILE];         // the agreed reference, handed from softmax group 0 to the others
};


// Two softmax groups ping-pong over alternating key tiles (group g owns tiles j = g mod GROUPS and the
// S/P buffers g): with the reference fixed by the first tile the tiles are independent, so while one
// group sits in its fixed latencies (barrier wake-up, TMEM store drain, remote arrive) the other keeps the
// MUFU / FMA pipes busy.  The groups' row sums are added in the epilogue.
template <bool TRACE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(640, 1)
attn_umma_kernel_v7(const __grid_constant__ CUtensorMap map_khalf, const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const KernelParams prm)
{
    constexpr int NPARTS = 2, GROUPS = 2;   // (row, 64-key half) threads; two softmax groups
    extern __shared__ uint8_t smem_raw[];
    SharedV7& sm = *reinterpret_cast<SharedV7*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    const int row_block = blockIdx.x;             // 128 rows; blockIdx.x = 2*cluster + rank
    const int split = blockIdx.y;
    const uint32_t rank = cluster_cta_rank();      // 0 = leader (issues the MMAs); rank r keeps keys [64r,64r+64) of K and columns [64r,64r+64) of V
    const bool leader = rank == 0;

    const int tq = prm.tiles_total / prm.splits, tr = prm.tiles_total % prm.splits;
    const int tile_begin = split * tq + min(split, tr);
    const int num_tiles = tq + (split < tr ? 1 : 0);   // identical in both CTAs of the cluster

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&map_khalf);
        prefetch_tensormap(&map_q);
        prefetch_tensormap(&map_k);
        prefetch_tensormap(&map_v);
        mbar_init(&sm.q_full, 2);          // leader's copy is the one used: one arrival per CTA's producer + all bytes
        mbar_init(&sm.o_done, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&sm.s_full[i], 1);
            mbar_init(&sm.p_ready[i], 2 * 4 * NPARTS);   // leader's copy: one arrival per softmax warp of BOTH CTAs
            mbar_init(&sm.s_free[i], 2 * 4 * NPARTS);    // leader's copy: S buffer i has been read into registers
            mbar_init(&sm.pv_done[i], 1);                // both CTAs: P buffer i may be overwritten
        }
        for (int i = 0; i < V7_KSTAGES; ++i) {
            mbar_init(&sm.k_full[i], 2);
            mbar_init(&sm.k_empty[i], 1);  // the leader's commit, multicast to both CTAs
        }
        for (int i = 0; i < V7_VSTAGES; ++i) {
            mbar_init(&sm.v_full[i], 2);
            mbar_init(&sm.v_empty[i], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc_2cta(&sm.tmem_base, 512);   // the same warp in both CTAs
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();   // the peer's barriers are initialised before anything is multicast to them
    tcgen05_fence_after();
    const uint32_t tmem = sm.tmem_base;
    auto stamp = [&](int role, int j, int ev) {
        if constexpr (TRACE) {
            if (blockIdx.x == 0 && blockIdx.y == 0 && lane == 0 && j < TRACE_ITERS)
                prm.trace[(role * TRACE_ITERS + j) * TRACE_EVENTS + ev] = clock64();
        }
    };

    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
        if (num_tiles > 0) {
            if (warp == 0) {
                // ================================ TMA producer ================================
                // every load lands in this CTA's shared memory and reports its bytes to the LEADER's barrier;
                // the leader arms the barrier with the bytes of both CTAs, the peer adds its plain arrival.
                const int qrow = row_block * TILE;
                const uint32_t leader_qfull = map_to_cta(&sm.q_full, 0);
                for (int j = 0; j < num_tiles; ++j) {
                    const int ks = j % V7_KSTAGES, vs = j % V7_VSTAGES;
                    const uint32_t kph = (uint32_t)(j / V7_KSTAGES) & 1u, vph = (uint32_t)(j / V7_VSTAGES) & 1u;
                    const int key0 = (tile_begin + j) * TILE;
                    if (j == 0 && elect_one_sync()) {
                        if (leader) mbar_arrive_expect_tx(&sm.q_full, 2 * TILE_BYTES);
                        else mbar_arrive_cluster(leader_qfull);
                        tma_load_2d_2sm(sm.q, &map_q, &sm.q_full, 0, qrow);
                        tma_load_2d_2sm(sm.q + HALF_BYTES, &map_q, &sm.q_full, 64, qrow);
                    }
                    mbar_wait(&sm.k_empty[ks], kph ^ 1u, 100 + ks);
                    stamp(5, j, 0);
                    if (elect_one_sync()) {
                        if (leader) mbar_arrive_expect_tx(&sm.k_full[ks], TILE_BYTES);
                        else mbar_arrive_cluster(map_to_cta(&sm.k_full[ks], 0));
                        // my 64 keys of the tile: two boxes of 64 columns x 64 rows (8 KiB each)
                        tma_load_2d_2sm(sm.k[ks], &map_khalf, &sm.k_full[ks], 0, key0 + 64 * (int)rank);
                        tma_load_2d_2sm(sm.k[ks] + HALF_TILE_BYTES / 2, &map_khalf, &sm.k_full[ks], 64, key0 + 64 * (int)rank);
                    }
                    mbar_wait(&sm.v_empty[vs], vph ^ 1u, 110 + vs);
                    stamp(5, j, 1);
                    if (elect_one_sync()) {
                        if (leader) mbar_arrive_expect_tx(&sm.v_full[vs], TILE_BYTES);
                        else mbar_arrive_cluster(map_to_cta(&sm.v_full[vs], 0));
                        // my 64 value columns of the tile: one box of 64 columns x 128 keys (16 KiB)
                        tma_load_2d_2sm(sm.v[vs], &map_v, &sm.v_full[vs], 64 * (int)rank, key0);
                    }
                    __syncwarp();
                }
            } else if (warp == 1) {
                // ================================ MMA issuer (leader CTA only) ==================
                if (leader) {
                constexpr uint32_t idesc_qk = make_idesc(2 * TILE, TILE, 0);   // M = 256 over the CTA pair
                constexpr uint32_t idesc_pv = make_idesc(2 * TILE, HEAD, 1);
                const uint64_t dq = desc_kmajor(smem_u32(sm.q), 0);
                // stage s of a ring: base descriptor + s * stage bytes (>> 4 in the address field); no indexed local arrays on the issue path
                const uint64_t dk0 = make_desc(smem_u32(sm.k[0]), 16u, 1024u), dv0 = make_desc(smem_u32(sm.v[0]), HALF_TILE_BYTES, 1024u);
                const uint16_t both = 0x3;

                auto issue_s = [&](int j) {
                    const int sb = j & 1, ks = j % V7_KSTAGES;
                    mbar_wait(&sm.k_full[ks], (uint32_t)(j / V7_KSTAGES) & 1u, 200 + ks);   // (already tested by the scheduler below)
                    tcgen05_fence_after();
                    if (elect_one_sync()) {
                        const uint64_t b0 = dk0 + (uint64_t)((uint32_t)ks * (HALF_TILE_BYTES >> 4));
                        const uint32_t d = tmem + V6_S + 128u * sb;
#pragma unroll
                        for (int kk = 0; kk < HEAD / 16; ++kk) {
                            const uint64_t offa = (uint64_t)(((kk >> 2) * HALF_BYTES + (kk & 3) * 32u) >> 4);            // Q: boxes of 128 rows
                            const uint64_t offb = (uint64_t)(((kk >> 2) * (HALF_TILE_BYTES / 2) + (kk & 3) * 32u) >> 4);   // K half: boxes of 64 rows
                            umma_ss_2cta(d, dq + offa, b0 + offb, idesc_qk, kk > 0 ? 1u : 0u);
                        }
                        umma_commit_2cta(&sm.s_full[sb], both);
                        umma_commit_2cta(&sm.k_empty[ks], both);
                    }
                    __syncwarp();
                };
                auto issue_pv = [&](int j, bool last) {
                    const int pb = j & 1, vs = j % V7_VSTAGES;
                    mbar_wait(&sm.v_full[vs], (uint32_t)(j / V7_VSTAGES) & 1u, 210 + vs);
                    mbar_wait(&sm.p_ready[pb], (uint32_t)(j >> 1) & 1u, 212 + pb);
                    stamp(4, j, 1);
                    tcgen05_fence_after();
                    if (elect_one_sync()) {
                        const uint64_t b0 = dv0 + (uint64_t)((uint32_t)vs * (HALF_TILE_BYTES >> 4));
                        const uint32_t d = tmem + V6_O;
                        const uint32_t a = tmem + V6_P + 64u * pb;
#pragma unroll
                        for (int kk = 0; kk < TILE / 16; ++kk)
                            umma_ts_2cta(d, a + 8u * kk, b0 + (uint64_t)((kk * 2048u) >> 4), idesc_pv, (j > 0 || kk > 0) ? 1u : 0u);
                        umma_commit_2cta(&sm.pv_done[pb], both);
                        umma_commit_2cta(&sm.v_empty[vs], both);
                        if (last) umma_commit_2cta(&sm.o_done, both);
                    }
                    __syncwarp();
                };

                mbar_wait(&sm.q_full, 0, 201);
                issue_s(0);
                if (num_tiles > 1) issue_s(1);
                // Fixed order per tile: S(j+2) as soon as S(j) sits in the softmax registers (s_free), then PV(j) once
                // P(j) is ready.  (A scheduler issuing "whichever stream is ready" was measured slower -- polling two
                // barriers costs more than the occasional head-of-line wait: profiles/r01/sweep_v7_3_testwait_scheduler.txt.)
                for (int j = 0; j < num_tiles; ++j) {
                    stamp(4, j, 0);
                    if (j + 2 < num_tiles) {
                        mbar_wait(&sm.s_free[j & 1], (uint32_t)(j >> 1) & 1u, 214 + (j & 1));
                        issue_s(j + 2);
                    }
                    stamp(4, j, 2);
                    issue_pv(j, j + 1 == num_tiles);
                    stamp(4, j, 3);
                }
                }
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
        constexpr int COLS = TILE / NPARTS;            // keys (S columns) per thread: 64 or 32
        constexpr int OCOLS = HEAD / (NPARTS * GROUPS); // output columns per thread in the epilogue
        const int sw = warp - 4;
        const int group = sw / (4 * NPARTS);           // which softmax group (owns tiles j = group mod GROUPS)
        const int half = (sw % (4 * NPARTS)) >> 2;     // which COLS-wide part of the row (0..NPARTS-1)
        const int gp = group * NPARTS + half;          // 0 .. NPARTS*GROUPS-1
        const int quad = warp & 3;                     // TMEM lane quadrant of this warp
        const int row_in_tile = quad * 32 + lane;
        const int grow = row_block * TILE + row_in_tile;
        if (num_tiles > 0) {
            // ================================ softmax + epilogue ==========================
            const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
            const uint32_t o_addr = tmem + lane_base + V6_O + (uint32_t)OCOLS * gp;
            const float scale = prm.scale_log2;
            const uint64_t scale2 = pack_f32x2(scale, scale);
            const int bar_id = 1 + quad;               // the warps of ONE group that share these 32 rows
            const int bar_all = 5 + quad;              // the warps of ALL groups that share these 32 rows
            const uint32_t leader_pready0 = map_to_cta(&sm.p_ready[0], 0), leader_sfree0 = map_to_cta(&sm.s_free[0], 0);   // [1] is 8 bytes further

            float m_ref = -CUDART_INF_F;
            float lsum = 0.f;

            auto exp_chunk = [&](const uint32_t* sv, uint64_t neg_ref2, uint64_t& acc0, uint64_t& acc1, uint32_t* pr) {
#pragma unroll
                for (int c = 0; c < 16; c += 2) {
                    const uint64_t x2 = pack_f32x2(__uint_as_float(sv[c]), __uint_as_float(sv[c + 1]));
                    const uint64_t t2 = fma_f32x2(x2, scale2, neg_ref2);
                    float t0, t1;
                    unpack_f32x2(t2, t0, t1);
                    const float p0 = fast_exp2(t0), p1 = fast_exp2(t1);
                    const uint64_t p2 = pack_f32x2(p0, p1);
                    if (c & 4) acc1 = add_f32x2(acc1, p2);
                    else acc0 = add_f32x2(acc0, p2);
                    pr[c / 2] = pack_bf16x2(p0, p1);
                }
            };

            auto tile_step = [&](int j, auto masked_tag, auto first_tag) {
                constexpr bool MASKED = decltype(masked_tag)::value;
                constexpr bool FIRST = decltype(first_tag)::value;
                const int sb = j & 1;
                const uint32_t s_addr = tmem + lane_base + V6_S + 128u * sb + (uint32_t)COLS * half;
                const uint32_t p_addr = tmem + lane_base + V6_P + 64u * sb + (uint32_t)(COLS / 2) * half;
                mbar_wait(&sm.s_full[sb], (uint32_t)(j >> 1) & 1u, 300 + sb);
                if (quad == 0 && half == 0) stamp(group, j, 0);
                tcgen05_fence_after();

                uint32_t sr[COLS];
                SDPA_TMEM_LD32(s_addr, sr);
                if constexpr (COLS == 64) SDPA_TMEM_LD32(s_addr + 32, (sr + 32));
                tmem_wait_ld();
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(leader_sfree0 + 8u * (uint32_t)sb);   // S buffer sb may be overwritten by S(j+2)
                if (quad == 0 && half == 0) stamp(group, j, 1);
                if constexpr (MASKED) {
                    const int keys_left = prm.n - (tile_begin + j) * TILE - COLS * half;
#pragma unroll
                    for (int c = 0; c < COLS; ++c)
                        if (c >= keys_left) sr[c] = 0xff800000u;  // -inf
                }
                float mx0 = -CUDART_INF_F, mx1 = -CUDART_INF_F, mx2 = -CUDART_INF_F, mx3 = -CUDART_INF_F;
#pragma unroll
                for (int c = 0; c < COLS; c += 8) {
                    mx0 = fmaxf(mx0, fmaxf(__uint_as_float(sr[c + 0]), __uint_as_float(sr[c + 1])));
                    mx1 = fmaxf(mx1, fmaxf(__uint_as_float(sr[c + 2]), __uint_as_float(sr[c + 3])));
                    mx2 = fmaxf(mx2, fmaxf(__uint_as_float(sr[c + 4]), __uint_as_float(sr[c + 5])));
                    mx3 = fmaxf(mx3, fmaxf(__uint_as_float(sr[c + 6]), __uint_as_float(sr[c + 7])));
                }
                const float my_max = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
                if constexpr (FIRST) {
                    // the reference of the whole key range: the first tile's row max, agreed by the two halves
                    sm.xchg[0][half][row_in_tile] = my_max;
                    named_barrier_sync(bar_id, 32 * NPARTS);
                    m_ref = my_max;
#pragma unroll
                    for (int p = 0; p < NPARTS; ++p) m_ref = fmaxf(m_ref, sm.xchg[0][p][row_in_tile]);
                    if constexpr (GROUPS > 1) {
                        if (half == 0) sm.mref[row_in_tile] = m_ref;
                        named_barrier_sync(bar_all, 32 * NPARTS * GROUPS);   // the other groups pick the reference up
                    }
                }
                // No wait is needed before overwriting P buffer sb: PV(j-2), its last reader, was issued before
                // S(j), and the commit behind s_full(j) covers every MMA issued before it.
                if (quad == 0 && half == 0) stamp(group, j, 2);

                const uint64_t neg_ref2 = pack_f32x2(-m_ref * scale, -m_ref * scale);
                uint64_t acc0 = pack_f32x2(0.f, 0.f), acc1 = acc0;
                uint32_t pr[COLS / 2];   // the packed bf16 P of the whole part; stored at the end, once PV(j-2) has left the buffer
#pragma unroll
                for (int ch = 0; ch < COLS / 16; ++ch) exp_chunk(sr + 16 * ch, neg_ref2, acc0, acc1, pr + 8 * ch);
                if (j >= 2) mbar_wait(&sm.pv_done[sb], (uint32_t)((j >> 1) - 1) & 1u, 310 + sb);
                tcgen05_fence_after();
#pragma unroll
                for (int ch = 0; ch < COLS / 16; ++ch) SDPA_TMEM_ST8(p_addr + 8 * ch, (pr + 8 * ch));
                float a0, a1, a2, a3;
                unpack_f32x2(acc0, a0, a1);
                unpack_f32x2(acc1, a2, a3);
                lsum += (a0 + a1) + (a2 + a3);
                if constexpr (!FIRST) {
                    // overflow guard, off the critical path (the max chain overlaps the exponentials)
                    if (__any_sync(0xffffffffu, (my_max - m_ref) * scale > kGuardThreshold)) {
                        if (lane == 0) atomicExch(prm.guard, prm.epoch);   // hand the launch to the SAFE kernel
                    }
                }
                if (quad == 0 && half == 0) stamp(group, j, 4);
                tmem_wait_st();
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(leader_pready0 + 8u * (uint32_t)sb);   // one arrival per warp, on the leader's barrier
                if (quad == 0 && half == 0) stamp(group, j, 5);
            };

            const bool ragged = (prm.n % TILE) != 0 && (tile_begin + num_tiles) == prm.tiles_total;
            if (group == 0) {
                if (ragged && num_tiles == 1) tile_step(0, std::true_type{}, std::true_type{});
                else tile_step(0, std::false_type{}, std::true_type{});
            } else {
                named_barrier_sync(bar_all, 32 * NPARTS * GROUPS);   // wait for group 0's reference
                m_ref = sm.mref[row_in_tile];
            }
            for (int j = (group == 0 ? GROUPS : group); j < num_tiles; j += GROUPS) {
                if (ragged && j == num_tiles - 1) tile_step(j, std::true_type{}, std::false_type{});
                else tile_step(j, std::false_type{}, std::false_type{});
            }

            // ---------------- epilogue ----------------
            sm.xchg[1][gp][row_in_tile] = lsum;
            named_barrier_sync(bar_all, 32 * NPARTS * GROUPS);
            lsum = 0.f;
#pragma unroll
            for (int p = 0; p < NPARTS * GROUPS; ++p) lsum += sm.xchg[1][p][row_in_tile];
            mbar_wait(&sm.o_done, 0, 320);
            tcgen05_fence_after();
            const bool valid = grow < prm.rows;
            const float inv = (lsum == 0.f) ? 0.f : 1.f / lsum;
#pragma unroll
            for (int c0 = 0; c0 < OCOLS; c0 += 32) {
                uint32_t orr[32];
                SDPA_TMEM_LD32(o_addr + c0, orr);
                tmem_wait_ld();
                if (valid) {
                    const int col = OCOLS * gp + c0;
                    if (prm.out64 != nullptr) {
                        double2* dst = reinterpret_cast<double2*>(prm.out64 + (size_t)grow * HEAD + col);
#pragma unroll
                        for (int c = 0; c < 32; c += 2)
                            dst[c / 2] = make_double2((double)(__uint_as_float(orr[c]) * inv),
                                                      (double)(__uint_as_float(orr[c + 1]) * inv));
                    } else {
                        float4* dst = reinterpret_cast<float4*>(prm.part_o + ((size_t)split * prm.rows_capacity + grow) * HEAD + col);
#pragma unroll
                        for (int c = 0; c < 32; c += 4)
                            dst[c / 4] = make_float4(__uint_as_float(orr[c]), __uint_as_float(orr[c + 1]),
                                                     __uint_as_float(orr[c + 2]), __uint_as_float(orr[c + 3]));
                    }
                }
            }
            if (valid && gp == 0 && prm.out64 == nullptr) {
                prm.part_tmax[(size_t)split * prm.rows_capacity + grow] = m_ref * scale;
                prm.part_lsum[(size_t)split * prm.rows_capacity + grow] = lsum;
            }
        } else if (grow < prm.rows) {
            // empty key range: the neutral state (0, -inf, 0), mpi.c:172,188
            if (prm.out64 != nullptr) {
                for (int c = 0; c < OCOLS; ++c) prm.out64[(size_t)grow * HEAD + OCOLS * gp + c] = 0.0;
            } else {
                float* dst = prm.part_o + ((size_t)split * prm.rows_capacity + grow) * HEAD + OCOLS * gp;
                for (int c = 0; c < OCOLS; ++c) dst[c] = 0.f;
                if (gp == 0) {
                    prm.part_tmax[(size_t)split * prm.rows_capacity + grow] = -CUDART_INF_F;
                    prm.part_lsum[(size_t)split * prm.rows_capacity + grow] = 0.f;
                }
            }
        }
    }

    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();   // neither CTA leaves while the other may still multicast into it or arrive on its barriers
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc_2cta(tmem, 512);
    }
}

// =====================================================================================
// v8 (SDPA_UMMA_V8=1, EXPERIMENTAL: written after the round's GPU budget was spent, not yet run on hardware).
// v7's pipeline made PERSISTENT: one cluster per SM pair walks a contiguous range of the linear work space
// (row block of 256 rows, key tile) -- "stream-K" over the key axis.  With 74 clusters every cluster gets
// RB*T/74 key tiles (+-1): no wave quantisation (v7 on c3: 288 equal units on 74 slots = 97.3 %), the prologue
// (barrier init, TMEM alloc, cluster sync, first loads) runs once per SM instead of once per 57-tile unit, and a
// row block is cut into ~T*74/(RB*T) + 1 pieces instead of 9 splits, so the split merge reads a third of the partials.
// A cluster's range crosses row-block boundaries: it is processed as SEGMENTS (row block, first tile, tile count).
// What v7 keeps per launch is carried across segments here:
//   * K/V rings and the S/P double buffers run on ONE tile counter g over all segments of the cluster, so the
//     S MMAs of the next segment's first tiles are issued while the current segment drains (no pipeline refill);
//   * Q has two shared-memory slots (segment parity); q_free (a commit behind the segment's last S MMA) lets the
//     producer overwrite a slot two segments later;
//   * the single O accumulator is handed back by o_free: every softmax warp of both CTAs arrives after it has read
//     its share of O in the segment's epilogue; the first PV of the next segment waits for it;
//   * the softmax reference is per segment: the group owning the segment's first tile (g & 1) fixes and publishes it.
// The partial state of segment (rb, piece) goes to partial slot `piece` = cluster - first cluster touching rb; the
// merge reads pieces(rb) states per row (merge_pieces_kernel), or all max_pieces after the SAFE twin ran.
// =====================================================================================
struct __align__(1024) SharedV8 {
    uint8_t q[2][TILE_BYTES];
    uint8_t k[V7_KSTAGES][HALF_TILE_BYTES];
    uint8_t v[V7_VSTAGES][HALF_TILE_BYTES];
    uint64_t q_full[2], q_free[2];
    uint64_t k_full[V7_KSTAGES], k_empty[V7_KSTAGES];
    uint64_t v_full[V7_VSTAGES], v_empty[V7_VSTAGES];
    uint64_t s_full[2], p_ready[2], s_free[2], pv_done[2], o_done, o_free;
    uint32_t tmem_base;
    float xchg[2][4][TILE];   // [first-tile max | final sum][group*2 + part][row]
    float mref[TILE];
};

// Walks the segments of the unit range [begin, end) of one cluster.
struct SegCursor {
    int u, uend, T;
    int seg, rb, t0, nt;
    __device__ __forceinline__ void init(int begin, int end, int tiles_per_row_block)
    {
        u = begin;
        uend = end;
        T = tiles_per_row_block;
        seg = -1;
        nt = 0;
        rb = t0 = 0;
    }
    __device__ __forceinline__ bool next()
    {
        u += nt;
        if (u >= uend) {
            nt = 0;
            return false;
        }
        rb = u / T;
        t0 = u - rb * T;
        nt = min(T - t0, uend - u);
        ++seg;
        return true;
    }
};

// (Measured and rejected in round 2, profiles/README.md: a separate V producer warp, P stored chunk by chunk, part of the
// exponentials as a polynomial on the FMA pipe.)
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(640, 1)
attn_umma_kernel_v8(const __grid_constant__ CUtensorMap map_khalf, const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const KernelParams prm)
{
    constexpr int NPARTS = 2, GROUPS = 2;
    extern __shared__ uint8_t smem_raw[];
    SharedV8& sm = *reinterpret_cast<SharedV8*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    const int cluster = blockIdx.x >> 1;
    const uint32_t rank = cluster_cta_rank();      // 0 = leader (issues the MMAs); rank r keeps keys [64r,64r+64) of K and columns [64r,64r+64) of V
    const bool leader = rank == 0;
    const WorkMap wm = prm.wm;
    const int T = wm.T;
    const int unit_begin = (int)wm_begin(wm, cluster), unit_end = (int)wm_begin(wm, cluster + 1);
    const int total_tiles = unit_end - unit_begin;   // identical in both CTAs of the cluster

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&map_khalf);
        prefetch_tensormap(&map_q);
        prefetch_tensormap(&map_k);
        prefetch_tensormap(&map_v);
        mbar_init(&sm.o_done, 1);
        mbar_init(&sm.o_free, 2 * 4 * NPARTS * GROUPS);   // leader's copy: every softmax warp of BOTH CTAs has read its share of O
        for (int i = 0; i < 2; ++i) {
            mbar_init(&sm.q_full[i], 2);       // leader's copy: one arrival per CTA's producer + all bytes
            mbar_init(&sm.q_free[i], 1);       // both CTAs: the commit behind the last S MMA that read the slot
            mbar_init(&sm.s_full[i], 1);
            mbar_init(&sm.p_ready[i], 2 * 4 * NPARTS);
            mbar_init(&sm.s_free[i], 2 * 4 * NPARTS);
            mbar_init(&sm.pv_done[i], 1);
        }
        for (int i = 0; i < V7_KSTAGES; ++i) {
            mbar_init(&sm.k_full[i], 2);
            mbar_init(&sm.k_empty[i], 1);
        }
        for (int i = 0; i < V7_VSTAGES; ++i) {
            mbar_init(&sm.v_full[i], 2);
            mbar_init(&sm.v_empty[i], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc_2cta(&sm.tmem_base, 512);
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();
    tcgen05_fence_after();
    const uint32_t tmem = sm.tmem_base;

    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
        if (total_tiles > 0) {
            if (warp == 0) {
                // ================================ TMA producer ================================
                SegCursor cur;
                cur.init(unit_begin, unit_end, T);
                int g = 0;
                while (cur.next()) {
                    const int qs = cur.seg & 1;
                    if (cur.seg >= 2) mbar_wait(&sm.q_free[qs], (uint32_t)((cur.seg >> 1) - 1) & 1u, 120 + qs);
                    if (elect_one_sync()) {
                        const int qrow = (2 * cur.rb + (int)rank) * TILE;
                        if (leader) mbar_arrive_expect_tx(&sm.q_full[qs], 2 * TILE_BYTES);
                        else mbar_arrive_cluster(map_to_cta(&sm.q_full[qs], 0));
                        tma_load_2d_2sm(sm.q[qs], &map_q, &sm.q_full[qs], 0, qrow);
                        tma_load_2d_2sm(sm.q[qs] + HALF_BYTES, &map_q, &sm.q_full[qs], 64, qrow);
                    }
                    __syncwarp();
                    for (int j = 0; j < cur.nt; ++j, ++g) {
                        const int ks = g % V7_KSTAGES, vs = g % V7_VSTAGES;
                        const uint32_t kph = (uint32_t)(g / V7_KSTAGES) & 1u, vph = (uint32_t)(g / V7_VSTAGES) & 1u;
                        const int key0 = (cur.t0 + j) * TILE;
                        mbar_wait(&sm.k_empty[ks], kph ^ 1u, 100 + ks);
                        if (elect_one_sync()) {
                            if (leader) mbar_arrive_expect_tx(&sm.k_full[ks], TILE_BYTES);
                            else mbar_arrive_cluster(map_to_cta(&sm.k_full[ks], 0));
                            tma_load_2d_2sm(sm.k[ks], &map_khalf, &sm.k_full[ks], 0, key0 + 64 * (int)rank);
                            tma_load_2d_2sm(sm.k[ks] + HALF_TILE_BYTES / 2, &map_khalf, &sm.k_full[ks], 64, key0 + 64 * (int)rank);
                        }
                        mbar_wait(&sm.v_empty[vs], vph ^ 1u, 110 + vs);
                        if (elect_one_sync()) {
                            if (leader) mbar_arrive_expect_tx(&sm.v_full[vs], TILE_BYTES);
                            else mbar_arrive_cluster(map_to_cta(&sm.v_full[vs], 0));
                            tma_load_2d_2sm(sm.v[vs], &map_v, &sm.v_full[vs], 64 * (int)rank, key0);
                        }
                        __syncwarp();
                    }
                }
            } else if (warp == 1) {
                // ================================ MMA issuer (leader CTA only) ==================
                if (leader) {
                constexpr uint32_t idesc_qk = make_idesc(2 * TILE, TILE, 0);
                constexpr uint32_t idesc_pv = make_idesc(2 * TILE, HEAD, 1);
                const uint64_t dq0 = desc_kmajor(smem_u32(sm.q[0]), 0);
                // stage s of a ring: base descriptor + s * stage bytes (>> 4 in the address field); no indexed local arrays on the issue path
                const uint64_t dk0 = make_desc(smem_u32(sm.k[0]), 16u, 1024u), dv0 = make_desc(smem_u32(sm.v[0]), HALF_TILE_BYTES, 1024u);
                const uint16_t both = 0x3;

                SegCursor cs, cp;   // the S stream runs two tiles ahead of the PV stream, possibly in the next segment
                cs.init(unit_begin, unit_end, T);
                cp.init(unit_begin, unit_end, T);
                cs.next();
                cp.next();
                int js = 0, jp = 0;

                auto issue_s = [&](int g) {
                    const int sb = g & 1, ks = g % V7_KSTAGES, qs = cs.seg & 1;
                    if (js == 0) mbar_wait(&sm.q_full[qs], (uint32_t)(cs.seg >> 1) & 1u, 201 + qs);
                    mbar_wait(&sm.k_full[ks], (uint32_t)(g / V7_KSTAGES) & 1u, 204 + ks);
                    tcgen05_fence_after();
                    const bool last_of_segment = (js == cs.nt - 1);
                    if (elect_one_sync()) {
                        const uint64_t a0 = dq0 + (uint64_t)((uint32_t)qs * (TILE_BYTES >> 4)), b0 = dk0 + (uint64_t)((uint32_t)ks * (HALF_TILE_BYTES >> 4));
                        const uint32_t d = tmem + V6_S + 128u * sb;
#pragma unroll
                        for (int kk = 0; kk < HEAD / 16; ++kk) {
                            const uint64_t offa = (uint64_t)(((kk >> 2) * HALF_BYTES + (kk & 3) * 32u) >> 4);
                            const uint64_t offb = (uint64_t)(((kk >> 2) * (HALF_TILE_BYTES / 2) + (kk & 3) * 32u) >> 4);
                            umma_ss_2cta(d, a0 + offa, b0 + offb, idesc_qk, kk > 0 ? 1u : 0u);
                        }
                        umma_commit_2cta(&sm.s_full[sb], both);
                        umma_commit_2cta(&sm.k_empty[ks], both);
                        if (last_of_segment) umma_commit_2cta(&sm.q_free[qs], both);   // no later MMA reads this Q slot
                    }
                    __syncwarp();
                    if (++js == cs.nt) {
                        cs.next();
                        js = 0;
                    }
                };
                auto issue_pv = [&](int g) {
                    const int pb = g & 1, vs = g % V7_VSTAGES;
                    const bool first = (jp == 0), last = (jp == cp.nt - 1);
                    // the accumulator still holds the previous segment until all of its epilogue reads are done
                    if (first && cp.seg >= 1) mbar_wait(&sm.o_free, (uint32_t)(cp.seg - 1) & 1u, 220);
                    mbar_wait(&sm.v_full[vs], (uint32_t)(g / V7_VSTAGES) & 1u, 210 + vs);
                    mbar_wait(&sm.p_ready[pb], (uint32_t)(g >> 1) & 1u, 214 + pb);
                    tcgen05_fence_after();
                    if (elect_one_sync()) {
                        const uint64_t b0 = dv0 + (uint64_t)((uint32_t)vs * (HALF_TILE_BYTES >> 4));
                        const uint32_t d = tmem + V6_O;
                        const uint32_t a = tmem + V6_P + 64u * pb;
#pragma unroll
                        for (int kk = 0; kk < TILE / 16; ++kk)
                            umma_ts_2cta(d, a + 8u * kk, b0 + (uint64_t)((kk * 2048u) >> 4), idesc_pv, (!first || kk > 0) ? 1u : 0u);
                        umma_commit_2cta(&sm.pv_done[pb], both);
                        umma_commit_2cta(&sm.v_empty[vs], both);
                        if (last) umma_commit_2cta(&sm.o_done, both);
                    }
                    __syncwarp();
                    if (++jp == cp.nt) {
                        cp.next();
                        jp = 0;
                    }
                };

                issue_s(0);
                if (total_tiles > 1) issue_s(1);
                for (int g = 0; g < total_tiles; ++g) {
                    if (g + 2 < total_tiles) {
                        mbar_wait(&sm.s_free[g & 1], (uint32_t)(g >> 1) & 1u, 216 + (g & 1));
                        issue_s(g + 2);
                    }
                    issue_pv(g);
                }
                }
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
        constexpr int COLS = TILE / NPARTS;             // 64 keys (S columns) per thread
        constexpr int OCOLS = HEAD / (NPARTS * GROUPS);  // 32 output columns per thread in the epilogue
        const int sw = warp - 4;
        const int group = sw / (4 * NPARTS);
        const int half = (sw % (4 * NPARTS)) >> 2;
        const int gp = group * NPARTS + half;
        const int quad = warp & 3;
        const int row_in_tile = quad * 32 + lane;
        if (total_tiles > 0) {
            const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
            const uint32_t o_addr = tmem + lane_base + V6_O + (uint32_t)OCOLS * gp;
            const float scale = prm.scale_log2;
            const uint64_t scale2 = pack_f32x2(scale, scale);
            const int bar_id = 1 + quad;
            const int bar_all = 5 + quad;
            const uint32_t leader_pready0 = map_to_cta(&sm.p_ready[0], 0), leader_sfree0 = map_to_cta(&sm.s_free[0], 0);   // [1] is 8 bytes further
            const uint32_t leader_ofree = map_to_cta(&sm.o_free, 0);

            float m_ref = -CUDART_INF_F;
            float lsum = 0.f;

            auto exp_chunk = [&](const uint32_t* sv, uint64_t neg_ref2, uint64_t& acc0, uint64_t& acc1, uint32_t* pr) {
#pragma unroll
                for (int c = 0; c < 16; c += 2) {
                    const uint64_t x2 = pack_f32x2(__uint_as_float(sv[c]), __uint_as_float(sv[c + 1]));
                    const uint64_t t2 = fma_f32x2(x2, scale2, neg_ref2);
                    float t0, t1;
                    unpack_f32x2(t2, t0, t1);
                    const float p0 = fast_exp2(t0), p1 = fast_exp2(t1);
                    const uint64_t p2 = pack_f32x2(p0, p1);
                    if (c & 4) acc1 = add_f32x2(acc1, p2);
                    else acc0 = add_f32x2(acc0, p2);
                    pr[c / 2] = pack_bf16x2(p0, p1);
                }
            };

            // g: tile counter of the cluster (buffers and barrier phases), key_tile: index of the tile in the shard
            auto tile_step = [&](int g, int key_tile, auto masked_tag, auto first_tag) {
                constexpr bool MASKED = decltype(masked_tag)::value;
                constexpr bool FIRST = decltype(first_tag)::value;
                const int sb = g & 1;
                const uint32_t s_addr = tmem + lane_base + V6_S + 128u * sb + (uint32_t)COLS * half;
                const uint32_t p_addr = tmem + lane_base + V6_P + 64u * sb + (uint32_t)(COLS / 2) * half;
                mbar_wait(&sm.s_full[sb], (uint32_t)(g >> 1) & 1u, 300 + sb);
                tcgen05_fence_after();

                uint32_t sr[COLS];
                SDPA_TMEM_LD32(s_addr, sr);
                SDPA_TMEM_LD32(s_addr + 32, (sr + 32));
                tmem_wait_ld();
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(leader_sfree0 + 8u * (uint32_t)sb);
                if constexpr (MASKED) {
                    const int keys_left = prm.n - key_tile * TILE - COLS * half;
#pragma unroll
                    for (int c = 0; c < COLS; ++c)
                        if (c >= keys_left) sr[c] = 0xff800000u;  // -inf
                }
                float mx0 = -CUDART_INF_F, mx1 = -CUDART_INF_F, mx2 = -CUDART_INF_F, mx3 = -CUDART_INF_F;
#pragma unroll
                for (int c = 0; c < COLS; c += 8) {
                    mx0 = fmaxf(mx0, fmaxf(__uint_as_float(sr[c + 0]), __uint_as_float(sr[c + 1])));
                    mx1 = fmaxf(mx1, fmaxf(__uint_as_float(sr[c + 2]), __uint_as_float(sr[c + 3])));
                    mx2 = fmaxf(mx2, fmaxf(__uint_as_float(sr[c + 4]), __uint_as_float(sr[c + 5])));
                    mx3 = fmaxf(mx3, fmaxf(__uint_as_float(sr[c + 6]), __uint_as_float(sr[c + 7])));
                }
                const float my_max = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
                if constexpr (FIRST) {
                    // the reference of the segment: its first tile's row max, agreed by the two halves, published to the other group
                    sm.xchg[0][half][row_in_tile] = my_max;
                    named_barrier_sync(bar_id, 32 * NPARTS);
                    m_ref = fmaxf(sm.xchg[0][0][row_in_tile], sm.xchg[0][1][row_in_tile]);
                    if (half == 0) sm.mref[row_in_tile] = m_ref;
                    named_barrier_sync(bar_all, 32 * NPARTS * GROUPS);
                }
                const uint64_t neg_ref2 = pack_f32x2(-m_ref * scale, -m_ref * scale);
                uint64_t acc0 = pack_f32x2(0.f, 0.f), acc1 = acc0;
                uint32_t pr[COLS / 2];
#pragma unroll
                for (int ch = 0; ch < COLS / 16; ++ch) exp_chunk(sr + 16 * ch, neg_ref2, acc0, acc1, pr + 8 * ch);
                if (g >= 2) mbar_wait(&sm.pv_done[sb], (uint32_t)((g >> 1) - 1) & 1u, 310 + sb);
                tcgen05_fence_after();
#pragma unroll
                for (int ch = 0; ch < COLS / 16; ++ch) SDPA_TMEM_ST8(p_addr + 8 * ch, (pr + 8 * ch));
                float a0, a1, a2, a3;
                unpack_f32x2(acc0, a0, a1);
                unpack_f32x2(acc1, a2, a3);
                lsum += (a0 + a1) + (a2 + a3);
                if constexpr (!FIRST) {
                    if (__any_sync(0xffffffffu, (my_max - m_ref) * scale > kGuardThreshold)) {
                        if (lane == 0) atomicExch(prm.guard, prm.epoch);
                    }
                }
                tmem_wait_st();
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(leader_pready0 + 8u * (uint32_t)sb);
            };

            SegCursor cur;
            cur.init(unit_begin, unit_end, T);
            int g0 = 0;   // tile counter at the start of the segment
            while (cur.next()) {
                const bool ragged = (prm.n % TILE) != 0 && (cur.t0 + cur.nt) == T;   // the segment ends with the shard's partial tile
                m_ref = -CUDART_INF_F;
                lsum = 0.f;
                int g;
                if (group == (g0 & 1)) {   // this group owns the segment's first tile: it fixes the reference
                    if (ragged && cur.nt == 1) tile_step(g0, cur.t0, std::true_type{}, std::true_type{});
                    else tile_step(g0, cur.t0, std::false_type{}, std::true_type{});
                    g = g0 + 2;
                } else {
                    named_barrier_sync(bar_all, 32 * NPARTS * GROUPS);
                    m_ref = sm.mref[row_in_tile];
                    g = g0 + 1;
                }
                for (; g < g0 + cur.nt; g += 2) {
                    if (ragged && g == g0 + cur.nt - 1) tile_step(g, cur.t0 + (g - g0), std::true_type{}, std::false_type{});
                    else tile_step(g, cur.t0 + (g - g0), std::false_type{}, std::false_type{});
                }

                // ---------------- epilogue of the segment ----------------
                sm.xchg[1][gp][row_in_tile] = lsum;
                named_barrier_sync(bar_all, 32 * NPARTS * GROUPS);
                lsum = 0.f;
#pragma unroll
                for (int p = 0; p < NPARTS * GROUPS; ++p) lsum += sm.xchg[1][p][row_in_tile];
                mbar_wait(&sm.o_done, (uint32_t)cur.seg & 1u, 320);
                tcgen05_fence_after();
                const int grow = (2 * cur.rb + (int)rank) * TILE + row_in_tile;
                const int piece = cluster - wm_cluster_of(wm, (long long)cur.rb * T);
                const bool valid = grow < prm.rows;
                {
                    uint32_t orr[32];
                    SDPA_TMEM_LD32(o_addr, orr);
                    tmem_wait_ld();
                    tcgen05_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cluster(leader_ofree);   // my share of O is in registers: the accumulator may be reused
                    if (valid) {
                        float4* dst = reinterpret_cast<float4*>(prm.part_o + ((size_t)piece * prm.rows_capacity + grow) * HEAD + OCOLS * gp);
#pragma unroll
                        for (int c = 0; c < 32; c += 4)
                            dst[c / 4] = make_float4(__uint_as_float(orr[c]), __uint_as_float(orr[c + 1]),
                                                     __uint_as_float(orr[c + 2]), __uint_as_float(orr[c + 3]));
                    }
                }
                if (valid && gp == 0) {
                    prm.part_tmax[(size_t)piece * prm.rows_capacity + grow] = m_ref * scale;
                    prm.part_lsum[(size_t)piece * prm.rows_capacity + grow] = lsum;
                }
                g0 += cur.nt;
            }
        }
    }

    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc_2cta(tmem, 512);
    }
}

// ---------------------------------------------------------------- host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode()
{
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

// 2-D bf16 row-major [rows][cols] tensor, box = 64 columns x box_rows rows, 128-byte swizzle; rows and columns of a box that
// lie outside the tensor are filled with zeros (this is what replaces the reference's masked vector tails, mpi.c:115-119).
sdpa_status encode_map(CUtensorMap* map, const void* base, int rows, int box_rows = TILE, int cols = HEAD)
{
    PFN_encodeTiled enc = get_encode();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
        return SDPA_ERR_CUDA;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)(rows > 0 ? rows : 1)};
    const cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (base=%p rows=%d cols=%d)", (int)r, base, rows, cols);
        return SDPA_ERR_CUDA;
    }
    return SDPA_OK;
}

}  // namespace

struct UmmaPlan {
    int dk = 0, dv = 0, hl = 1;      // operand widths; hl = 2: hi/lo split operands (lo arrays lo_off elements behind hi)
    bool general = false;            // the shape goes to attn_umma_general_kernel (anything but dk = dv = 128 bf16)
    CUtensorMap gmaps[2][6];         // general kernel, per Q slot: q_hi q_lo k_hi k_lo v_hi v_lo
    CUtensorMap map_k, map_v, map_q[2];
    CUtensorMap map_khalf;   // K with 64-row boxes (v7: each CTA of a pair keeps 64 keys of a tile)
    int n = 0;
    bool kv_bound = false, q_bound[2] = {false, false};
    const void* q_base[2] = {nullptr, nullptr};
    const void* k_base = nullptr;
    const void* v_base = nullptr;
    int q_rows[2] = {0, 0};
    size_t q_lo[2] = {0, 0};
    bool attr_set[64] = {};
    // Overflow guard: a ring of kGuardRing device words; the launch with epoch e uses word e % kGuardRing and a fast kernel writes
    // e into it when an exponent would overflow.  A word equals a launch's epoch only if THAT launch raised it, so the words are
    // never cleared and the host can inspect a whole queue of launches after the fact (deferred repair, engine.cu).
    unsigned int* guard = nullptr;
    unsigned int epoch = 0;
    bool force_exact = false;        // run the exact variant alone (the host-side repair of a launch whose guard fired)
    unsigned int twin_epoch = 0;     // epoch the twin of the last fast launch must see in the guard word to run
    bool allow_v8 = false;           // set per call by the engine: the caller merges with launch_merge_pieces
    bool last_v8 = false;            // the last launch used the persistent kernel; last_wm / last_pieces describe its partials
    WorkMap last_wm{0, 0, 0};
    int last_pieces = 0;
    bool attr8_set[64] = {};
};

__global__ void set_word_kernel(unsigned int* p, unsigned int v) { *p = v; }

static sdpa_status plan_guard_ring(UmmaPlan* plan)
{
    if (plan->guard) return SDPA_OK;
    SDPA_CUDA_TRY(cudaMalloc(&plan->guard, kGuardRing * sizeof(unsigned int)));
    SDPA_CUDA_TRY(cudaMemset(plan->guard, 0, kGuardRing * sizeof(unsigned int)));
    return SDPA_OK;
}
static unsigned int plan_next_epoch(UmmaPlan* plan)
{
    if (++plan->epoch == 0) ++plan->epoch;   // 0 is the "never raised" value of a fresh ring
    return plan->epoch;
}

sdpa_status umma_plan_create(UmmaPlan** plan)
{
    *plan = new UmmaPlan();
    return SDPA_OK;
}
void umma_plan_destroy(UmmaPlan* plan)
{
    if (plan && plan->guard) cudaFree(plan->guard);
    delete plan;
}

bool attn_umma_supported(int dk, int dv, int hl) { return attn_umma_general_shape(dk, dv, hl, nullptr); }

static bool force_general()
{
    const char* e = getenv("SDPA_UMMA_GENERAL");   // developer knob: run dk = dv = 128 bf16 on the general kernel too
    return e && *e == '1';
}

sdpa_status umma_plan_bind_kv(UmmaPlan* plan, const __nv_bfloat16* K, const __nv_bfloat16* V, int n, int dk, int dv, int hl,
                              size_t k_lo_off, size_t v_lo_off)
{
    if (!attn_umma_supported(dk, dv, hl)) {
        set_error("tensor-core kernel: dk, dv must be multiples of 8 up to 256 (split precision: up to 128); got dk=%d dv=%d", dk, dv);
        return SDPA_ERR_UNSUPPORTED;
    }
    if (plan->kv_bound && plan->k_base == K && plan->v_base == V && plan->n == n && plan->dk == dk && plan->dv == dv && plan->hl == hl)
        return SDPA_OK;   // descriptors still valid
    if (plan->dk != dk || plan->hl != hl) plan->q_bound[0] = plan->q_bound[1] = false;
    plan->dk = dk;
    plan->dv = dv;
    plan->hl = hl;
    plan->general = !(dk == HEAD && dv == HEAD && hl == 1) || force_general();
    {   // the general kernel's maps are bound for every shape: its exact variant is the repair twin of v7 / v8 too
        for (int slot = 0; slot < 2; ++slot) {
            SDPA_TRY(encode_map(&plan->gmaps[slot][2], K, n, 64, dk));
            SDPA_TRY(encode_map(&plan->gmaps[slot][3], K + (hl == 2 ? k_lo_off : 0), n, 64, dk));
            SDPA_TRY(encode_map(&plan->gmaps[slot][4], V, n, TILE, dv));
            SDPA_TRY(encode_map(&plan->gmaps[slot][5], V + (hl == 2 ? v_lo_off : 0), n, TILE, dv));
        }
    }
    if (dk == HEAD && dv == HEAD && hl == 1) {
        SDPA_TRY(encode_map(&plan->map_k, K, n));
        SDPA_TRY(encode_map(&plan->map_v, V, n));
        SDPA_TRY(encode_map(&plan->map_khalf, K, n, 64));
    }
    plan->k_base = K;
    plan->v_base = V;
    plan->n = n;
    plan->kv_bound = true;
    return SDPA_OK;
}

sdpa_status umma_plan_bind_q(UmmaPlan* plan, int slot, const __nv_bfloat16* Q, int rows_capacity, int dk, int hl, size_t q_lo_off)
{
    if (slot < 0 || slot > 1 || dk != plan->dk || hl != plan->hl) {
        set_error("umma_plan_bind_q: bad slot, or dk / precision differ from the bound K/V shard");
        return SDPA_ERR_INVALID;
    }
    if (plan->q_bound[slot] && plan->q_base[slot] == Q && plan->q_rows[slot] == rows_capacity && plan->q_lo[slot] == q_lo_off) return SDPA_OK;
    {
        SDPA_TRY(encode_map(&plan->gmaps[slot][0], Q, rows_capacity, TILE, dk));
        SDPA_TRY(encode_map(&plan->gmaps[slot][1], Q + (hl == 2 ? q_lo_off : 0), rows_capacity, TILE, dk));
    }
    if (dk == HEAD && plan->dv == HEAD && hl == 1) SDPA_TRY(encode_map(&plan->map_q[slot], Q, rows_capacity));
    plan->q_bound[slot] = true;
    plan->q_base[slot] = Q;
    plan->q_rows[slot] = rows_capacity;
    plan->q_lo[slot] = q_lo_off;
    return SDPA_OK;
}

static bool trace_env_set()
{
    const char* t = getenv("SDPA_UMMA_TRACE");
    return t && *t;
}

// Kernel generation: v7 (cluster of two 128-row CTAs, 2-CTA MMA) unless SDPA_UMMA_V7=0 asks for v5.

// Persistent kernel: its work map for (rows, n) on sm_count SMs, or false when the shape
// does not suit it (too little work per cluster, or more pieces per row block than the merge takes).
static bool v8_work_map(int rows, int n, int sm_count, WorkMap* wm, int* max_pieces)
{
    const char* e = getenv("SDPA_UMMA_V8");   // SDPA_UMMA_V8=0: always the plain-grid kernel (v7)
    if ((e && *e == '0') || rows <= 0 || n <= 0) return false;
    WorkMap w;
    w.T = ceil_div(n, TILE);
    w.RB = ceil_div(rows, 2 * TILE);
    w.C = std::max(1, sm_count / 2);
    if (wm_total(w) < 4LL * w.C || wm_total(w) > 0x3fffffffLL) return false;
    int mp = 0;
    for (int rb = 0; rb < w.RB; ++rb) mp = std::max(mp, wm_pieces(w, rb));
    if (mp < 1 || mp > 64) return false;
    *wm = w;
    *max_pieces = mp;
    return true;
}

int attn_umma_v8_pieces(int rows, int n, int sm_count)
{
    WorkMap w;
    int mp = 0;
    return v8_work_map(rows, n, sm_count, &w, &mp) ? mp : 0;
}

void umma_plan_allow_v8(UmmaPlan* plan, bool allow)
{
    if (plan) plan->allow_v8 = allow;
}

bool umma_plan_last_v8(const UmmaPlan* plan, WorkMap* wm, int* max_pieces, const unsigned int** guard, unsigned int* epoch)
{
    if (!plan || !plan->last_v8) return false;
    *wm = plan->last_wm;
    *max_pieces = plan->last_pieces;
    *guard = plan->guard + (plan->twin_epoch % kGuardRing);
    *epoch = plan->twin_epoch;
    return true;
}

// The guard word and epoch of the fast launch that just went out (for the engine's deferred repair), and the ring itself.
void umma_plan_last_guard(const UmmaPlan* plan, unsigned int* slot, unsigned int* epoch)
{
    *slot = plan->twin_epoch % kGuardRing;
    *epoch = plan->twin_epoch;
}
const unsigned int* umma_plan_guard_ring(const UmmaPlan* plan) { return plan ? plan->guard : nullptr; }
void umma_plan_force_exact(UmmaPlan* plan, bool on)
{
    if (plan) plan->force_exact = on;
}

int attn_umma_pick_splits(int rows, int n, int sm_count)
{
    const int row_blocks = 2 * ceil_div(ceil_div(rows, TILE), 2);   // 128-row CTAs in clusters of two
    const int tiles = ceil_div(n, TILE);
    if (row_blocks <= 0 || tiles <= 1) return 1;
    // choose the split count (<= 64, >= 4 key tiles each) with the best wave efficiency of the
    // grid row_blocks x splits over sm_count CTAs-at-a-time; prefer fewer splits on ties.
    const int max_splits = std::min(64, std::max(1, tiles / 4));
    auto efficiency = [&](int s) {
        const int ctas = row_blocks * s;
        const int waves = ceil_div(ctas, sm_count);
        const int tiles_per = ceil_div(tiles, s);  // the slowest CTA of a wave sets its length
        return (double)row_blocks * tiles / ((double)waves * sm_count * tiles_per);
    };
    double best_eff = 0.0;
    for (int s = 1; s <= max_splits; ++s) best_eff = std::max(best_eff, efficiency(s));
    // fewest splits within 4% of the best: every extra split costs rows*dv*8 bytes of partial traffic
    int best = 1;
    for (int s = 1; s <= max_splits; ++s)
        if (efficiency(s) >= 0.96 * best_eff) {
            best = s;
            break;
        }
    return best;
}

void preload_attn_umma_general_kernels();
void preload_attn_umma_kernels()
{
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, attn_umma_kernel_v7<false>);
    cudaFuncGetAttributes(&a, attn_umma_kernel_v8);
    cudaGetLastError();
    preload_attn_umma_general_kernels();
}

// The exact variant behind the fast launch that just went out (same epoch): leaves at once unless the guard was raised.
sdpa_status launch_attn_umma_twin(UmmaPlan* plan, int q_slot, int rows, int splits, Partials part, double* out64, cudaStream_t stream)
{
    if (!plan || rows <= 0) return SDPA_OK;
    if (splits < 1) splits = 1;
    GeneralLaunch L;
    L.rows = rows;
    L.n = plan->n;
    L.dk = plan->dk;
    L.dv = plan->dv;
    L.hl = plan->hl;
    L.splits = splits;
    L.exact = true;
    L.part = part;
    L.out64 = out64;
    L.guard = plan->guard + (plan->twin_epoch % kGuardRing);
    L.epoch = plan->twin_epoch;
    L.maps = plan->gmaps[q_slot];
    return launch_attn_umma_general(L, stream);
}

// The fast fused kernel only; the caller launches launch_attn_umma_twin behind it (separately, so that the stage timing of the
// fused kernel does not include the twin's launch).
sdpa_status launch_attn_umma(UmmaPlan* plan, int q_slot, int rows, int splits, Partials part, double* out64,
                             int sm_count, cudaStream_t stream)
{
    if (!plan || !plan->kv_bound || q_slot < 0 || q_slot > 1 || !plan->q_bound[q_slot]) {
        set_error("launch_attn_umma: plan is not bound");
        return SDPA_ERR_INVALID;
    }
    if (rows <= 0) return SDPA_OK;
    if (splits < 1) splits = 1;
    if (out64 != nullptr && splits != 1) {
        set_error("direct fp64 output requires splits == 1");
        return SDPA_ERR_INVALID;
    }
    if (plan->general) {
        // every shape but dk = dv = 128 bf16: the general kernel, then its exact twin (leaves at once unless the guard fired)
        SDPA_TRY(plan_guard_ring(plan));
        GeneralLaunch L;
        L.rows = rows;
        L.n = plan->n;
        L.dk = plan->dk;
        L.dv = plan->dv;
        L.hl = plan->hl;
        L.splits = splits;
        L.part = part;
        L.out64 = out64;
        L.epoch = plan_next_epoch(plan);
        L.guard = plan->guard + (L.epoch % kGuardRing);
        L.maps = plan->gmaps[q_slot];
        plan->last_v8 = false;
        plan->twin_epoch = L.epoch;
        const char* env_safe = getenv("SDPA_UMMA_SAFE");
        if (plan->force_exact || (env_safe && *env_safe == '1')) {
            // only the exact variant (the twin, launched by the caller): this launch's guard word is made to carry its epoch
            set_word_kernel<<<1, 1, 0, stream>>>(L.guard, L.epoch);
            count_launch();
            return SDPA_OK;
        }
        L.exact = false;
        return launch_attn_umma_general(L, stream);
    }
    int dev = 0;
    SDPA_CUDA_TRY(cudaGetDevice(&dev));
    // developer knob: SDPA_UMMA_SAFE=1 runs the exact variant alone
    const char* env_safe = getenv("SDPA_UMMA_SAFE");
    const bool force_safe = plan->force_exact || (env_safe && *env_safe == '1');
    if (dev < 64 && !plan->attr_set[dev]) {
        const int sb7 = (int)(sizeof(SharedV7) + 1024);
        SDPA_CUDA_TRY(cudaFuncSetAttribute(attn_umma_kernel_v7<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, sb7));
        SDPA_CUDA_TRY(cudaFuncSetAttribute(attn_umma_kernel_v7<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sb7));
        plan->attr_set[dev] = true;
    }
    SDPA_TRY(plan_guard_ring(plan));
    KernelParams prm;
    prm.rows = rows;
    prm.n = plan->n;
    prm.tiles_total = ceil_div(plan->n, TILE);
    prm.splits = splits;
    prm.scale_log2 = (1.0f / sqrtf((float)HEAD)) * 1.4426950408889634f;
    prm.part_o = part.o;
    prm.part_tmax = part.tmax;
    prm.part_lsum = part.lsum;
    prm.rows_capacity = part.rows_capacity;
    prm.out64 = out64;
    prm.trace = nullptr;
    prm.epoch = plan_next_epoch(plan);
    prm.guard = plan->guard + (prm.epoch % kGuardRing);
    const size_t smem7 = sizeof(SharedV7) + 1024;
    dim3 grid6(2 * ceil_div(ceil_div(rows, TILE), 2), splits);          // v7: 128 rows per CTA, clusters of two along x
    // persistent kernel: only when the engine announced that it merges by pieces, no direct fp64 output, and the caller's
    // split count is the map's piece count (the exact twin behind it then fills every partial slot the merge may read)
    WorkMap wm8{0, 0, 0};
    int pieces8 = 0;
    const bool use_v8 = plan->allow_v8 && out64 == nullptr && !force_safe && !(trace_env_set()) &&
                        v8_work_map(rows, plan->n, sm_count, &wm8, &pieces8) && pieces8 == splits;
    plan->last_v8 = false;
    const char* trace_path = getenv("SDPA_UMMA_TRACE");   // developer aid: dump a clock64 timeline of CTA (0,0)
    if (trace_path && *trace_path) {
        const size_t count = (size_t)TRACE_ROLES * TRACE_ITERS * TRACE_EVENTS;
        long long* dtrace = nullptr;
        SDPA_CUDA_TRY(cudaMalloc(&dtrace, count * sizeof(long long)));
        SDPA_CUDA_TRY(cudaMemsetAsync(dtrace, 0, count * sizeof(long long), stream));
        prm.trace = dtrace;
        attn_umma_kernel_v7<true><<<grid6, 640, smem7, stream>>>(plan->map_khalf, plan->map_q[q_slot], plan->map_k, plan->map_v, prm);
        count_launch();
        std::vector<long long> host(count);
        SDPA_CUDA_TRY(cudaMemcpyAsync(host.data(), dtrace, count * sizeof(long long), cudaMemcpyDeviceToHost, stream));
        SDPA_CUDA_TRY(cudaStreamSynchronize(stream));
        SDPA_CUDA_TRY(cudaFree(dtrace));
        if (FILE* f = fopen(trace_path, "w")) {
            fprintf(f, "role iteration event clock\n");
            for (int r = 0; r < TRACE_ROLES; ++r)
                for (int j = 0; j < TRACE_ITERS; ++j)
                    for (int e = 0; e < TRACE_EVENTS; ++e)
                        if (host[(r * TRACE_ITERS + j) * TRACE_EVENTS + e])
                            fprintf(f, "%d %d %d %lld\n", r, j, e, host[(r * TRACE_ITERS + j) * TRACE_EVENTS + e]);
            fclose(f);
        }
        prm.trace = nullptr;
    } else if (force_safe) {
        // only the exact variant (launched by the caller): make this launch's guard word carry its epoch
        set_word_kernel<<<1, 1, 0, stream>>>(prm.guard, prm.epoch);
        count_launch();
    } else if (use_v8) {
        const int dev8 = dev;
        const size_t smem8 = sizeof(SharedV8) + 1024;
        prm.wm = wm8;
        const dim3 grid8(2 * wm8.C, 1);
        static bool attr8_done[64] = {};
        if (dev8 < 64 && !attr8_done[dev8]) {
            SDPA_CUDA_TRY(cudaFuncSetAttribute(attn_umma_kernel_v8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem8));
            // the SM's shared-memory carveout at its maximum (228 KB), not the smallest step that holds this CTA (196 KB): the
            // rest is what the small-footprint side kernels (cast-ahead, background merge) run in beside a resident CTA
            SDPA_CUDA_TRY(cudaFuncSetAttribute(attn_umma_kernel_v8, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
            attr8_done[dev8] = true;
        }
        attn_umma_kernel_v8<<<grid8, 640, smem8, stream>>>(plan->map_khalf, plan->map_q[q_slot], plan->map_k, plan->map_v, prm);
        count_launch();
        plan->last_v8 = true;
        plan->last_wm = wm8;
        plan->last_pieces = pieces8;
    } else {
        attn_umma_kernel_v7<false><<<grid6, 640, smem7, stream>>>(plan->map_khalf, plan->map_q[q_slot], plan->map_k, plan->map_v, prm);
        count_launch();
    }
    plan->twin_epoch = prm.epoch;
    SDPA_CUDA_TRY(cudaGetLastError());
    return SDPA_OK;
}

}  // namespace sdpa
