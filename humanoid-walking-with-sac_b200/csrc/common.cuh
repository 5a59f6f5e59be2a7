// Shared device/host definitions of the SAC update "program": a static list of tile tasks grouped into
// dependency stages.  The same task code runs (a) as one kernel per stage inside a CUDA graph and
// (b) inside ONE persistent cooperative launch with grid barriers between stages.
//
// Operand storage ("pair matrix", PM): every matrix a GEMM reads -- minibatch inputs, activations, activation
// gradients and a shadow of every hidden/head weight -- is kept in HBM/L2 as two bf16 planes, hi = bf16(x) and
// lo = bf16(x - hi), each row-major [rows, ld] with ld a multiple of 8 (16 B).  x ~= hi + lo to 2^-17 relative.
// TMA moves 128-byte-swizzled boxes of both planes straight into shared memory; the tensor core then forms
// a*b as  a_lo*b_hi + a_hi*b_lo + a_hi*b_hi  (three kind::f16 MMAs, fp32 accumulate in TMEM).  The fp32
// master weights, Adam moments and all scalars/vectors stay fp32.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sacb {

// ---- reference constants (SURVEY 3.6) ------------------------------------------------------------------
constexpr float kLogStdMin = -20.f, kLogStdMax = 2.f;     // networks_model1.py:74, networks_model2.py:95
constexpr float kSquashEps = 1e-6f;                        // networks_model1.py:96
constexpr float kLogSqrt2Pi = 0.91893853320467274178f;     // torch Normal.log_prob
constexpr float kBeta1 = 0.9f, kBeta2 = 0.999f, kAdamEps = 1e-8f;  // torch.optim.Adam defaults (sac_imp.py:39-41)

// ---- a pointer that is valid for every agent of a population: region base + offset ----------------------
// region 0 = arena (params, targets, Adam state, weight shadows, scalars), region 1 = workspace
struct Ref {
    int64_t v;   // -1 = null ; bit 62 = region ; low bits = float offset
};
__host__ __device__ inline Ref make_ref(int region, int64_t off) { Ref r; r.v = ((int64_t)region << 62) | off; return r; }
__host__ __device__ inline Ref null_ref() { Ref r; r.v = -1; return r; }
__host__ __device__ inline bool is_null(Ref r) { return r.v < 0; }

struct AgentBases {
    float *arena;      // base of agent 0
    float *ws;
    int64_t arena_stride, ws_stride;   // floats between consecutive agents
};
__device__ __forceinline__ float *resolve(Ref r, const AgentBases &b, int agent) {
    if (r.v < 0) return nullptr;
    const int64_t off = r.v & ((1ll << 62) - 1);
    return ((r.v >> 62) & 1) ? b.ws + agent * b.ws_stride + off : b.arena + agent * b.arena_stride + off;
}

// ---- pair-matrix view: rows [row0, row0+R) of a PM; `base` points at element (0,0) of the view's hi plane ----
struct PmRef {
    Ref base;            // float-unit offset of the first hi element of the view (16 B aligned)
    int32_t ld;          // bf16 elements between rows (multiple of 8)
    int32_t pad;
    int64_t plane;       // bf16 elements from a hi element to its lo element
};
struct Pm {              // resolved for one agent
    __nv_bfloat16 *hi;
    int ld;
    int64_t plane;
};
__device__ __forceinline__ Pm resolve_pm(const PmRef &r, const AgentBases &b, int agent) {
    Pm p; p.hi = reinterpret_cast<__nv_bfloat16 *>(resolve(r.base, b, agent)); p.ld = r.ld; p.plane = r.plane; return p;
}
__host__ __device__ inline PmRef null_pm() { PmRef r; r.base = null_ref(); r.ld = 0; r.pad = 0; r.plane = 0; return r; }

// ---- scalars kept per agent in the arena (offsets in floats from the scalar block) ----------------------
enum ScalarSlot {
    SC_LOG_ALPHA = 0, SC_LOG_ALPHA_M, SC_LOG_ALPHA_V,
    SC_ALPHA0, SC_ALPHA1,            // alpha used by step t = SC_ALPHA0 + (n_updates & 1); written for t+1 into the other
    SC_STEP_POLICY, SC_STEP_Q1, SC_STEP_Q2, SC_STEP_ALPHA, SC_N_UPDATES,   // stored as int32 bit patterns
    SC_LOSS_Q1, SC_LOSS_Q2, SC_LOSS_PI, SC_LOSS_ALPHA,
    SC_ERROR_FLAG,                   // copy of the device error flag made by T_FINISH: losses + flag come back in ONE D2H copy
    SC_COUNT = 16,
    SC_HIST_POS = 24,                // int32 bit pattern: completed updates since create, never reset: loss_hist[(pos % kLossHist)] = losses of that update
    // Adam bias-correction factors of the NEXT step of each optimizer, refreshed whenever a step counter changes
    // (T_FINISH, sacb_set_scalars, the data-parallel apply): [SC_FAC0 + 2*(step_slot - SC_STEP_POLICY)] = step_size, +1 = sqrt(bc2)
    SC_FAC0 = 16
};

// ---- GEMM operand: logical X[R, K] (R = M for A, N for B) held in a PM -----------------------------------
// mn_major = 0: the PM stores [R, K] (K contiguous);  mn_major = 1: the PM stores [K, R] (R contiguous) and the
// tensor core reads it transposed (UMMA MN-major descriptor) -- nothing is ever transposed in memory.
struct Operand {
    PmRef pm;
    int32_t mn_major;
    int32_t r0;          // the operand is rows [r0, r0+R) of the view along its M/N dimension.  TMA needs the byte offset of
                         // a box along the contiguous dimension to be a multiple of 16: r0 % 8 == 0 when mn_major = 1
};

enum TaskType : int32_t {
    T_GEMM = 0,
    T_SHADOW,        // fp32 master weights -> bf16 hi/lo shadow PMs (start of every step)
    T_GATHER,        // replay ring rows -> minibatch PMs
    T_SAMPLE,        // policy head outputs -> tanh-Gaussian sample + log-prob     (networks_model1.py:78-99)
    T_TARGET_LOSS,   // Bellman target + twin critic MSE + dL/dq + dL/dh_last      (sac_imp.py:92-105)
    T_ACTOR_LOSS,    // policy loss, min-Q routing + dL/dh_last                    (sac_imp.py:117-121)
    T_SAMPLE_BWD,    // dL/da -> dL/dmean, dL/dlog_std                             (SURVEY 3.3)
    T_OUT_ADAM,      // Q output layer: dW=dq^T h, db=sum dq, Adam, Polyak
    T_BIAS_ADAM,     // hidden-layer bias: db = colsum(dh), Adam, Polyak
    T_FINISH,        // loss scalars, temperature step (sac_imp.py:128-135), step counters
    T_LN_FWD,        // opt-in LayerNorm variant: z (fp32) -> relu(LN(z) * gamma + beta) as a PM, row statistics kept
    T_LN_BWD         // gradient of that: dpre (PM, ReLU mask applied) -> dz (PM) and the per-row terms of dgamma
};

enum Epilogue : int32_t {
    EPI_F32 = 0,         // C[fp32] = acc (+ bias[n])
    EPI_BIAS_RELU,       // PM  = relu(acc + bias[n])
    EPI_MASK,            // PM  = acc * (mask_hi[m,n] > 0)
    EPI_ADAM,            // acc = dW tile: Adam on W (+ Polyak into Wt, + shadow PM refresh, + optional grad export)
    EPI_SAMPLE           // policy heads: C[fp32] = acc + bias (mean | log_std_raw), then the tanh-Gaussian sample + log-prob of
                         // the tile's rows (the T_SAMPLE task fused into the heads GEMM; its arguments sit in the generic slots)
};

struct AdamArgs {
    Ref w, m, v;        // same shape as the GEMM output, ld = N
    Ref wt;             // Polyak target (null for the policy)
    Ref gexp;           // gradient export (null unless SACB_EXPORT_GRADS / data-parallel mode)
    PmRef shadow;       // bf16 pair shadow of w refreshed in place (null: not needed before the next step)
    PmRef shadow2;      // second shadow holding only columns >= shadow2_col0 of w (the action block of a critic's fc1)
    PmRef shadow_t;     // throughput programs only (stream.cuh): bf16 pair shadow of the Polyak target wt, refreshed in the epilogue too
    int32_t shadow2_col0, pad0;
    int32_t step_slot;  // ScalarSlot of the optimizer step counter (value BEFORE this step's increment)
    int32_t apply;      // 0 = only export the gradient (data-parallel backward), 1 = apply Adam
    float lr, tau;
};

struct alignas(64) Task {
    // TMA descriptors of the two GEMM operands: dims {cols, rows, plane(2), agent}, SWIZZLE_128B, bf16
    CUtensorMap tmA, tmB;
    int32_t type;
    int32_t tile_begin;       // first tile of this task inside its stage
    int32_t n_tiles;
    int32_t tiles_m, tiles_n;
    int32_t bm, bn;           // output tile of this GEMM task: 128 or 64 rows x 64 or 32 columns (chosen per stage by the builder)
    // --- GEMM
    Operand A, B;
    int32_t M, N, K;
    int32_t epi;
    Ref C; int32_t ldc;       // EPI_F32
    PmRef Cpm;                // EPI_BIAS_RELU / EPI_MASK
    Ref bias;
    PmRef mask;
    AdamArgs adam;
    // --- elementwise tasks: generic slots (meaning depends on type, see tasks.cuh)
    Ref p[24];
    PmRef pm[6];
    int32_t i[8];
    float f[6];
};

// Specialised builds of the stage kernel (staged mode): a launch only carries the code its stage can reach -- the task types and
// GEMM epilogues in its masks -- which keeps the register allocation of the hot paths free of the other paths' pressure (no
// spills in the forward / element-wise stages) and the instruction footprint of a 3-10 us kernel small.  X(index, task types, epilogues);
// the host picks the smallest variant that covers a stage, variant 0 (everything) runs the persistent single-launch mode.
constexpr uint32_t tb(int t) { return 1u << t; }
constexpr uint32_t kAllTypes = (1u << (T_LN_BWD + 1)) - 1, kAllEpis = (1u << (EPI_SAMPLE + 1)) - 1;
// everything the reference architecture needs: the single persistent launch of a handle without LayerNorm does not carry the
// LayerNorm tasks (their code alone cost the everything-build 0.265 -> 0.302 ms per update)
constexpr uint32_t kBaseTypes = kAllTypes & ~((1u << T_LN_FWD) | (1u << T_LN_BWD));
constexpr uint32_t kPlainEpis = tb(EPI_F32) | tb(EPI_BIAS_RELU) | tb(EPI_MASK);
constexpr uint32_t kElemTypes = tb(T_SHADOW) | tb(T_GATHER) | tb(T_SAMPLE) | tb(T_TARGET_LOSS) | tb(T_ACTOR_LOSS) | tb(T_SAMPLE_BWD) | tb(T_FINISH) | tb(T_LN_FWD) | tb(T_LN_BWD);
#define SACB_KERNEL_VARIANTS(X)                                                                     \
    X(0, kBaseTypes, kAllEpis)                                                                      \
    X(1, tb(T_GEMM), tb(EPI_BIAS_RELU))                                                         \
    X(2, tb(T_GEMM), tb(EPI_MASK))                                                                  \
    X(3, tb(T_GEMM), tb(EPI_F32))                                                                   \
    X(4, tb(T_GEMM), kPlainEpis)                                                                    \
    X(5, tb(T_GEMM) | tb(T_OUT_ADAM), tb(EPI_MASK))                                                 \
    X(6, tb(T_GEMM) | tb(T_BIAS_ADAM) | tb(T_SHADOW), tb(EPI_ADAM))                                 \
    X(7, tb(T_GEMM) | tb(T_BIAS_ADAM) | tb(T_SHADOW), tb(EPI_ADAM) | tb(EPI_MASK))                               \
    X(8, tb(T_GEMM) | tb(T_BIAS_ADAM) | tb(T_OUT_ADAM), kPlainEpis | tb(EPI_ADAM))                  \
    X(9, tb(T_SHADOW) | tb(T_GATHER), 0u)                                                           \
    X(10, tb(T_SAMPLE), 0u)                                                                         \
    X(11, tb(T_TARGET_LOSS), 0u)                                                                    \
    X(12, tb(T_ACTOR_LOSS), 0u)                                                                     \
    X(13, tb(T_SAMPLE_BWD), 0u)                                                                     \
    X(14, tb(T_FINISH), 0u)                                                                                    \
    X(15, kElemTypes, 0u)                                                                           \
    X(16, tb(T_GEMM) | tb(T_SHADOW), tb(EPI_BIAS_RELU))                                             \
    X(17, tb(T_OUT_ADAM) | tb(T_BIAS_ADAM), 0u)                                                     \
    X(18, tb(T_LN_FWD), 0u)                                                                         \
    X(19, tb(T_LN_BWD), 0u)                                                                         \
    X(20, kAllTypes, kAllEpis)
constexpr int kNumKernelVariants = 21;
constexpr int kVariantEverything = 0, kVariantEverythingLn = 20;      // the build a persistent launch runs (without / with LayerNorm)
// "Light" builds: column-sum / sample-backward stages only.  A tile of theirs is one batch of loads, two barriers and a 64-element
// Adam step: a throughput program walks thousands of them (population: 2304 per stage) and one 512-thread CTA per SM leaves the
// memory system idle between its two dependent round trips.  They are compiled for TWO resident CTAs per SM (<= 64 registers).
constexpr uint32_t kLightTypes = tb(T_OUT_ADAM) | tb(T_BIAS_ADAM) | tb(T_SAMPLE_BWD);
constexpr int variant_min_blocks(uint32_t types, uint32_t epis) { return (types != 0 && (types & ~kLightTypes) == 0 && epis == 0) ? 2 : 1; }

// builds that carry the chained form of a launch (Stage::chain_map): tensor-core GEMMs with the plain epilogues, T_SHADOW riders.  The
// others keep ONE call site of their task bodies (a second one makes the compiler outline them: stack frame, 4 us more per Adam stage)
constexpr bool variant_chains(int math, uint32_t types, uint32_t epis) {
    return math != SACB_MATH_FP32 && (types & tb(T_GEMM)) != 0 && (types & ~(tb(T_GEMM) | tb(T_SHADOW))) == 0 && (epis & ~kPlainEpis) == 0;
}
constexpr int kMaxStageTasks = 28;
constexpr int kMaxChainClusters = 32;
struct Stage {
    int32_t task_begin, task_end;
    int32_t n_tiles;          // per agent
    int32_t tile_begin[kMaxStageTasks];   // first tile of each task of the stage (copy of Task::tile_begin: one load finds the task)
    // Chained launch (program.cu: find_chains): consecutive row-local GEMM stages in ONE launch of thread-block clusters, cluster c
    // owns one row block in every stage of the chain, CTA rank r its column tile r.  The chain's first stage holds the number of
    // stages and of row clusters (further clusters of the launch walk the T_SHADOW riders of the chain's stages); every stage of the
    // chain holds, per row cluster, (stage tile of the row block's first column tile) | (column tiles << 16), or -1: no tile.
    int32_t chain_len, chain_clusters;
    int32_t chain_map[kMaxChainClusters];
};

struct Program {
    const Task *tasks;
    const Stage *stages;
    int32_t n_stages;
    int32_t n_agents;
    AgentBases bases;
    Ref scalars;              // arena ref of the scalar block
    unsigned int *barrier;    // grid barrier counter (persistent mode)
    // replay ring (T_GATHER)
    const float *ring; int64_t ring_agent_stride; int32_t ring_row; int32_t pad0;
    const int64_t *ring_meta; // [n_agents][2] = (stored transitions, slot of the oldest one): the uniform ring as the device sees it (device index draws)
    const int32_t *slots;     // physical ring slots of the minibatch rows [n_agents, B]
    int32_t slots_stride; int32_t pad1;
    int32_t *error_flag;      // set by watchdogs (mbarrier / grid barrier timeouts)
    const float2 *adam_table;     // [kAdamTable] (step_size, sqrt(bc2)) of Adam step t+1 for t = index, computed on the host in float64
    unsigned long long *timeline; // optional [n_stages][4]: earliest CTA start, earliest dependency release, latest CTA end (profiling aid)
    unsigned long long *trace; // optional [grid][kTraceSlots] globaltimer stamps of each CTA's first tile (profiling aid), or null
    float *host_losses;       // pinned HOST memory (addressable from the device), or null: T_FINISH of agent 0 stores the three losses, the
                              // alpha loss and the error flag there as well, so that the caller's read-back needs no copy behind the step
};

// ---- tile geometry ----------------------------------------------------------------------------------------
constexpr int kThreads = 512;
constexpr int kAdamTable = 32768;   // beyond ~17.3 k steps both bias corrections round to exactly 1.0f: the last entry serves every later step
constexpr int kLossHist = 64;     // per-agent ring of the last updates' (q1, q2, policy, alpha) losses: K updates per call, ONE read-back
constexpr int kTraceSlots = 64;   // 0..5 kernel phases, 6 accumulator ready, 16+kb TMA issue of k-block kb, 32+kb its arrival (kb < 16)
// FFMA path (checker / strict mode)
constexpr int kSM = 64, kSN = 64, kSK = 16;
// tcgen05 path: output tile up to 128 x 64 (a task may use 64 rows and / or 32 columns: Task::bm, bn), K blocks of 64 bf16
// (= 128 B, one SWIZZLE_128B row), both planes per stage
constexpr int kTM = 128, kTN = 64, kTK = 64, kTStages = 4;
constexpr int kTcABytes = kTM * kTK * 2 * 2;                      // hi + lo planes of the A tile: 32 KB
constexpr int kTcBBytes = kTN * kTK * 2 * 2;                      // 16 KB
constexpr int kTcStageBytes = kTcABytes + kTcBBytes;              // 48 KB
constexpr int kTcSmemBytes = kTStages * kTcStageBytes + 1024;     // + slack for the 1024 B alignment of the ring
constexpr int kSimtSmemBytes = 2 * kSK * (kSM + 4) * 4;

__host__ __device__ inline int cdiv(int a, int b) { return (a + b - 1) / b; }

}  // namespace sacb
