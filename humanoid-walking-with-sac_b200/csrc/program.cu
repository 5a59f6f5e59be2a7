// The SAC update as a static tile program: layout, kernel, host-side program builder, launch / CUDA graph.
//
// Reference semantics: sac_imp.SAC.update_parameters (sac_imp.py:74-144), in its order of operations
// (SURVEY 3.2): target with pre-step policy/targets -> twin critic MSE + Adam -> actor through the UPDATED
// critics + Adam -> temperature + Adam -> Polyak.
#include <algorithm>
#include <string>
#include <map>
#include <tuple>
#include <cstring>
#include <cstdio>
#include <cstdlib>

#include "handle.h"
#include "tasks.cuh"
#include "stream.cuh"

#ifndef SACB_NO_OUTLINE
#define SACB_NO_OUTLINE 1   // outlining measured SLOWER on B200 (persistent 0.265 -> 0.278 ms, one-kernel staged 0.242 -> 0.250): kept as an experiment switch
#endif

namespace sacb {

// ================================================================================================================
// layout
// ================================================================================================================
void NetLayout::tensor(int t, int64_t &off, int64_t &rows, int64_t &cols) const {
    const int pl = per_layer(), nh2 = pl * n_hidden;
    if (t < nh2) {
        const int l = t / pl, j = t % pl;
        if (j == 0) { off = w[l]; rows = hidden; cols = in_of(l); }
        else { off = j == 1 ? b[l] : (j == 2 ? g[l] : be[l]); rows = hidden; cols = 1; }
        return;
    }
    const int k = t - nh2;
    if (!is_policy) {   // fc_out.weight [1,H], fc_out.bias [1]
        if (k == 0) { off = w_out; rows = 1; cols = hidden; } else { off = b_out; rows = 1; cols = 1; }
    } else {            // mean.weight, mean.bias, log_std.weight, log_std.bias
        const int A = out_dim / 2;
        if (k == 0) { off = w_out; rows = A; cols = hidden; }
        else if (k == 1) { off = b_out; rows = A; cols = 1; }
        else if (k == 2) { off = w_out + (int64_t)A * hidden; rows = A; cols = hidden; }
        else { off = b_out + A; rows = A; cols = 1; }
    }
}

static void build_net(NetLayout &n, bool is_policy, int in_dim, int hidden, int n_hidden, int out_dim, int act_cols, bool layer_norm) {
    n.is_policy = is_policy; n.in_dim = in_dim; n.hidden = hidden; n.n_hidden = n_hidden; n.out_dim = out_dim; n.layer_norm = layer_norm;
    int64_t o = 0;
    for (int l = 0; l < n_hidden; l++) {
        n.w[l] = o; o = align_up(o + (int64_t)hidden * n.in_of(l), 4);
        n.b[l] = o; o = align_up(o + hidden, 4);
        if (layer_norm) { n.g[l] = o; o = align_up(o + hidden, 4); n.be[l] = o; o = align_up(o + hidden, 4); }
    }
    n.w_out = o; o = align_up(o + (int64_t)out_dim * hidden, 4);
    n.b_out = o; o = align_up(o + out_dim, 4);
    n.size = align_up(o, 32);
    // shadows: a PM of R rows and row stride ld (bf16) takes R*ld floats (two planes of R*ld bf16)
    o = 0;
    for (int l = 0; l < n_hidden; l++) {
        n.sh_ld[l] = (int)align_up(n.in_of(l), 8);
        n.sh_w[l] = o; o = align_up(o + (int64_t)hidden * n.sh_ld[l], 32);
    }
    n.sh_out = o;
    if (is_policy) o = align_up(o + (int64_t)out_dim * hidden, 32);
    n.sh_act = o; n.sh_act_ld = (int)align_up(std::max(act_cols, 1), 8);
    if (!is_policy) o = align_up(o + (int64_t)hidden * n.sh_act_ld, 32);
    n.sh_size = align_up(o, 32);
}

void Layout::build(int obs_, int act_, int hidden_, int n_hidden_, int maxB_, bool layer_norm_) {
    obs = obs_; act = act_; hidden = hidden_; n_hidden = n_hidden_; maxB = maxB_; layer_norm = layer_norm_;
    ldx = (int)align_up(obs + act, 8);
    ldg = (int)align_up(2 * act, 8);
    build_net(pol, true, obs, hidden, n_hidden, 2 * act, 0, layer_norm);
    build_net(q, false, obs + act, hidden, n_hidden, 1, act, layer_norm);
    int64_t o = 0;
    scalars = o; o += 32;
    loss_hist = o; o += 4 * kLossHist;
    param[0] = o; o += pol.size;
    for (int k = 1; k < 5; k++) { param[k] = o; o += q.size; }
    const int64_t sz[3] = {pol.size, q.size, q.size};
    for (int k = 0; k < 3; k++) { adam_m[k] = o; o += sz[k]; }
    for (int k = 0; k < 3; k++) { adam_v[k] = o; o += sz[k]; }
    for (int k = 0; k < 3; k++) { grad[k] = o; o += sz[k]; }
    grad_scalars = o; o += 32;
    dp_flags = o; o += 32;
    shadow[0] = o; o += pol.sh_size;
    for (int k = 1; k < 5; k++) { shadow[k] = o; o += q.sh_size; }
    arena_size = align_up(o, 64);
    // workspace
    const int64_t B = maxB, H = hidden, A = act;
    auto take = [&](int64_t n) { int64_t r = o; o = align_up(o + n, 32); return r; };
    o = 0;
    X = take(3 * B * ldx);
    r = take(B); d = take(B); isw = take(B); y = take(B); td = take(B);
    dq[0] = take(B); dq[1] = take(B);
    logp = take(2 * B); eps = take(2 * B * A);
    head_raw = take(2 * B * 2 * A); g_head = take(B * ldg);
    da[0] = take(B * A); da[1] = take(B * A);
    loss_part = take(2 * ((B + kLossRows - 1) / kLossRows) + 8); aloss_part = take(2 * ((B + kLossRows - 1) / kLossRows) + 8);
    for (int l = 0; l < n_hidden; l++) { hp[l] = take(2 * B * H); dhp[l] = take(B * H); }
    for (int k = 0; k < 2; k++)
        for (int l = 0; l < n_hidden; l++) {
            ht[k][l] = take(B * H); hc[k][l] = take(B * H); ha[k][l] = take(B * H);
            dhc[k][l] = take(B * H); dha[k][l] = take(B * H);
        }
    if (layer_norm) {
        for (int l = 0; l < n_hidden; l++) { zp[l] = take(2 * B * H); sp[l] = take(4 * B); dzp[l] = take(B * H); ggp[l] = take(B * H); }
        for (int k = 0; k < 2; k++)
            for (int l = 0; l < n_hidden; l++) {
                zt[k][l] = take(B * H); zc[k][l] = take(B * H); za[k][l] = take(B * H);
                st[k][l] = take(2 * B); sc[k][l] = take(2 * B); sa[k][l] = take(2 * B);
                dzc[k][l] = take(B * H); dza[k][l] = take(B * H); ggc[k][l] = take(B * H);
            }
    }
    ws_size = align_up(o, 64);
}

// ================================================================================================================
// TMA descriptors
// ================================================================================================================
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {     // resolved through the runtime: the library does not link libcuda (it must load on GPU-less build hosts)
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

int make_pm_tensor_map(CUtensorMap *out, const void *base, int64_t cols, int64_t rows, int64_t ld, int64_t plane_elems,
                       int64_t agent_stride_bytes, int n_agents, int box_rows) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return fail(SACB_ERR_DEVICE, "cuTensorMapEncodeTiled is not available from the CUDA driver");
    if (ld % 8 || plane_elems % 8 || agent_stride_bytes % 16 || (reinterpret_cast<uintptr_t>(base) & 15))
        return fail(SACB_ERR_ARG, "pair matrix is not 16-byte aligned for TMA");
    const cuuint64_t dims[4] = {(cuuint64_t)cols, (cuuint64_t)rows, 2, (cuuint64_t)n_agents};
    const cuuint64_t strides[3] = {(cuuint64_t)ld * 2, (cuuint64_t)plane_elems * 2, (cuuint64_t)std::max<int64_t>(agent_stride_bytes, 16)};
    const cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 2, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(SACB_ERR_DEVICE, "cuTensorMapEncodeTiled failed (code " + std::to_string((int)r) + ")");
    return SACB_OK;
}

// ================================================================================================================
// kernel
// ================================================================================================================
__device__ __forceinline__ void grid_barrier(unsigned int *counter, unsigned int target, int *error_flag) {
    // writers: generic-proxy global stores of this stage must be visible to the TMA (async proxy) reads of the next
    tc::fence_proxy_async();
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        unsigned int it = 0;
        while (true) {
            unsigned int v;
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
            if (v >= target) break;
            if (++it > (1u << 24)) { atomicExch(error_flag, 2); break; }   // watchdog: never hang the box
        }
        __threadfence();
    }
    __syncthreads();
    tc::fence_proxy_async();
}

// The build that carries every code path (variant 0: the single persistent launch) calls its task bodies through NON-inlined
// functions, one per task type / GEMM epilogue: each body then gets its own register allocation and schedule (as in the per-stage
// builds) instead of sharing the union of everybody's live ranges, which put spills into the MMA issue loop and the Adam epilogue.
template <uint32_t kEpi>
__device__ __noinline__ void gemm_tile_tc_outlined(const Task &t, const Task *tg, int tile, const AgentBases &bases, int agent, const float *scalars,
                                                   tc::TcState &st, int *error_flag, bool first_tile, uint64_t seed) {
    gemm_tile_tc<kEpi>(t, tg, tile, bases, agent, scalars, st, error_flag, first_tile, seed);
}
__device__ __noinline__ void task_shadow_outlined(const Task &t, int tile, const Program &P, int agent) { task_shadow(t, tile, P, agent); }
__device__ __noinline__ void task_gather_outlined(const Task &t, int tile, const Program &P, int agent, const float *scalars, uint64_t seed) { task_gather(t, tile, P, agent, scalars, seed); }
__device__ __noinline__ void task_sample_outlined(const Task &t, int tile, const Program &P, int agent, const float *scalars, uint64_t seed) { task_sample(t, tile, P, agent, scalars, seed); }
__device__ __noinline__ void task_target_loss_outlined(const Task &t, int tile, const Program &P, int agent, const float *scalars, float *smem) { task_target_loss(t, tile, P, agent, scalars, smem); }
__device__ __noinline__ void task_actor_loss_outlined(const Task &t, int tile, const Program &P, int agent, const float *scalars, float *smem) { task_actor_loss(t, tile, P, agent, scalars, smem); }
__device__ __noinline__ void task_sample_bwd_outlined(const Task &t, int tile, const Program &P, int agent, const float *scalars) { task_sample_bwd(t, tile, P, agent, scalars); }
__device__ __noinline__ void task_out_adam_outlined(const Task &t, int tile, const Program &P, int agent, const float *scalars, float *smem) { task_out_adam(t, tile, P, agent, scalars, smem); }
__device__ __noinline__ void task_bias_adam_outlined(const Task &t, int tile, const Program &P, int agent, const float *scalars, float *smem) { task_bias_adam(t, tile, P, agent, scalars, smem); }
__device__ __noinline__ void task_finish_outlined(const Task &t, const Program &P, int agent, float *scalars, float *smem) { task_finish(t, P, agent, scalars, smem); }

// Between two layers of a chained launch: the epilogue's global stores (generic proxy) become visible to the TMA reads (async proxy)
// of the other CTAs of the cluster, which own the rest of the row block.  A chain of one-CTA clusters only orders its own CTA.
__device__ __forceinline__ void chain_barrier(uint32_t cluster_size) {
    asm volatile("fence.proxy.async.global;" ::: "memory");
    if (cluster_size > 1) { tc::cluster_arrive(); tc::cluster_wait(); }
    else __syncthreads();
    asm volatile("fence.proxy.async.global;" ::: "memory");
}

template <int kMath, uint32_t kTypes, uint32_t kEpis>
__global__ void __launch_bounds__(kThreads, variant_min_blocks(kTypes, kEpis))
sac_update_kernel(const __grid_constant__ Program P, const __grid_constant__ Stage single, const int stage_begin, const int stage_end, const int tc_setup,
                  const int chained, const uint64_t seed) {
    // `single` = the stage table entry when the launch covers exactly one stage (staged mode): no global load before the first task.
    // chained != 0: the launch covers the stages of one chain (Stage::chain_map), as thread-block clusters.
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ uint64_t s_bars[2 * kTStages + 1];
    __shared__ uint32_t s_tmem;
    __shared__ float s_red[kColsumSmem];      // >= kThreads floats
    __shared__ Stage s_stage;
    __shared__ Task s_task;            // fields of the current task (the TMA descriptors are used from global memory)

    auto stamp = [&](int slot) {
        if (P.trace && threadIdx.x == 0) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            P.trace[(size_t)blockIdx.x * kTraceSlots + slot] = t;
        }
    };
    stamp(0);
    auto timeline = [&](int slot, bool is_max) {      // one entry per launch, under its first stage
        if (P.timeline && threadIdx.x == 0 && (stage_end - stage_begin == 1 || chained)) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (is_max) atomicMax(&P.timeline[stage_begin * 4 + slot], t); else atomicMin(&P.timeline[stage_begin * 4 + slot], t);
        }
    };
    timeline(0, false);
    tc::TcState st;
    st.g = 0; st.accum_uses = 0; st.tmem_base = 0; st.b_pre = 0;
    st.full_bar = s_bars; st.empty_bar = s_bars + kTStages; st.accum_bar = s_bars + 2 * kTStages; st.trace = P.trace;
    constexpr bool kTc = kMath != SACB_MATH_FP32;
    st.tiles = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    if (kTc && (kTypes & tb(T_GEMM)) != 0 && tc_setup) {
        if (threadIdx.x == 32) {      // warp 1 initialises the barriers while warp 0 allocates tensor memory
            for (int i = 0; i <= 2 * kTStages; i++) tc::mbar_init(&s_bars[i], 1);
            tc::fence_barrier_init();
        }
        if (threadIdx.x < 32) tc::tmem_alloc(&s_tmem, kTN);
        tc::tc_fence_before();
        __syncthreads();
        tc::tc_fence_after();
        st.tmem_base = s_tmem;
    }

    stamp(1);
    bool dep_synced = false;
    const Task *cached_task = nullptr;
    auto load_stage = [&](int s) {
        __syncthreads();      // the previous stage's readers of s_stage are done
        if (threadIdx.x < sizeof(Stage) / 4) {
            const int32_t *src = (stage_end - stage_begin == 1) ? reinterpret_cast<const int32_t *>(&single) : reinterpret_cast<const int32_t *>(&P.stages[s]);
            reinterpret_cast<int32_t *>(&s_stage)[threadIdx.x] = src[threadIdx.x];
        }
        __syncthreads();
        stamp(9);
    };
    // task of stage tile `tile_in_stage` (s_stage) -> global record, tile index inside the task; its fields -> s_task
    auto fetch_task = [&](int tile_in_stage, int &tile, bool first) -> const Task * {
        int k = 0;
        while (k + 1 < s_stage.task_end - s_stage.task_begin && tile_in_stage >= s_stage.tile_begin[k + 1]) k++;
        const Task *tg = &P.tasks[s_stage.task_begin + k];
        tile = tile_in_stage - s_stage.tile_begin[k];
        if (tg != cached_task) {   // one parallel fetch of the task's fields instead of a chain of dependent global loads; a CTA that walks
                                   // many tiles of the same task (population / large batch) keeps its copy
            cached_task = tg;
            constexpr int kSkip = 2 * sizeof(CUtensorMap) / 4, kWords = sizeof(Task) / 4 - kSkip;
            static_assert(kWords <= kThreads, "task copy");
            if (kTc && threadIdx.x == kThreads - 1) { tc::tma_prefetch_desc(&tg->tmA); tc::tma_prefetch_desc(&tg->tmB); }
            __syncthreads();     // the previous tile's readers of s_task are done
            if (first) stamp(10);
            if ((int)threadIdx.x < kWords)
                reinterpret_cast<int32_t *>(&s_task)[kSkip + threadIdx.x] = __ldcg(reinterpret_cast<const int32_t *>(tg) + kSkip + threadIdx.x);
            __syncthreads();
            if (first) stamp(11);
        }
        return tg;
    };
    auto dep_sync = [&]() {      // everything before only read launch parameters and the static task tables
        if (dep_synced) return;
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        dep_synced = true;
        timeline(1, false);
    };
    auto run_task = [&](const Task *tg, int tile, int agent, bool first) {
        const Task &t = s_task;
        float *scalars = resolve(P.scalars, P.bases, agent);
        constexpr bool kOutlined = kTc && (kTypes & kBaseTypes) == kBaseTypes && kEpis == kAllEpis && !SACB_NO_OUTLINE;
        if constexpr (kOutlined) {
            switch (t.type) {
                case T_GEMM:
                    switch (t.epi) {
                        case EPI_F32: gemm_tile_tc_outlined<tb(EPI_F32)>(t, tg, tile, P.bases, agent, scalars, st, P.error_flag, first, seed); break;
                        case EPI_BIAS_RELU: gemm_tile_tc_outlined<tb(EPI_BIAS_RELU)>(t, tg, tile, P.bases, agent, scalars, st, P.error_flag, first, seed); break;
                        case EPI_MASK: gemm_tile_tc_outlined<tb(EPI_MASK)>(t, tg, tile, P.bases, agent, scalars, st, P.error_flag, first, seed); break;
                        case EPI_SAMPLE: gemm_tile_tc_outlined<tb(EPI_SAMPLE)>(t, tg, tile, P.bases, agent, scalars, st, P.error_flag, first, seed); break;
                        default: gemm_tile_tc_outlined<tb(EPI_ADAM)>(t, tg, tile, P.bases, agent, scalars, st, P.error_flag, first, seed); break;
                    }
                    break;
                case T_SHADOW: task_shadow_outlined(t, tile, P, agent); break;
                case T_GATHER: task_gather_outlined(t, tile, P, agent, scalars, seed); break;
                case T_SAMPLE: task_sample_outlined(t, tile, P, agent, scalars, seed); break;
                case T_TARGET_LOSS: task_target_loss_outlined(t, tile, P, agent, scalars, s_red); break;
                case T_ACTOR_LOSS: task_actor_loss_outlined(t, tile, P, agent, scalars, s_red); break;
                case T_SAMPLE_BWD: task_sample_bwd_outlined(t, tile, P, agent, scalars); break;
                case T_OUT_ADAM: task_out_adam_outlined(t, tile, P, agent, scalars, s_red); break;
                case T_BIAS_ADAM: task_bias_adam_outlined(t, tile, P, agent, scalars, s_red); break;
                case T_FINISH: task_finish_outlined(t, P, agent, scalars, s_red); break;
                case T_LN_FWD: task_ln_fwd(t, tile, P, agent); break;
                case T_LN_BWD: task_ln_bwd(t, tile, P, agent); break;
            }
        } else
        switch (t.type) {      // only the task types of this build's mask are compiled in
            case T_GEMM:
                if constexpr ((kTypes & tb(T_GEMM)) != 0) {
                    if (kTc) gemm_tile_tc<kEpis>(t, tg, tile, P.bases, agent, scalars, st, P.error_flag, first, seed);
                    else gemm_tile_ffma(t, tile, P.bases, agent, scalars, reinterpret_cast<float *>(smem_raw));
                }
                break;
            case T_SHADOW: if constexpr ((kTypes & tb(T_SHADOW)) != 0) task_shadow(t, tile, P, agent); break;
            case T_GATHER: if constexpr ((kTypes & tb(T_GATHER)) != 0) task_gather(t, tile, P, agent, scalars, seed); break;
            case T_SAMPLE: if constexpr ((kTypes & tb(T_SAMPLE)) != 0) task_sample(t, tile, P, agent, scalars, seed); break;
            case T_TARGET_LOSS: if constexpr ((kTypes & tb(T_TARGET_LOSS)) != 0) task_target_loss(t, tile, P, agent, scalars, s_red); break;
            case T_ACTOR_LOSS: if constexpr ((kTypes & tb(T_ACTOR_LOSS)) != 0) task_actor_loss(t, tile, P, agent, scalars, s_red); break;
            case T_SAMPLE_BWD: if constexpr ((kTypes & tb(T_SAMPLE_BWD)) != 0) task_sample_bwd(t, tile, P, agent, scalars); break;
            case T_OUT_ADAM: if constexpr ((kTypes & tb(T_OUT_ADAM)) != 0) task_out_adam<variant_min_blocks(kTypes, kEpis) == 1>(t, tile, P, agent, scalars, s_red); break;
            case T_BIAS_ADAM: if constexpr ((kTypes & tb(T_BIAS_ADAM)) != 0) task_bias_adam<variant_min_blocks(kTypes, kEpis) == 1>(t, tile, P, agent, scalars, s_red); break;
            case T_FINISH: if constexpr ((kTypes & tb(T_FINISH)) != 0) task_finish(t, P, agent, scalars, s_red); break;
            case T_LN_FWD: if constexpr ((kTypes & tb(T_LN_FWD)) != 0) task_ln_fwd(t, tile, P, agent); break;
            case T_LN_BWD: if constexpr ((kTypes & tb(T_LN_BWD)) != 0) task_ln_bwd(t, tile, P, agent); break;
        }
        if (first) stamp(4);
    };

    if (!chained) {
        unsigned int bar_target = 0;
        for (int s = stage_begin; s < stage_end; s++) {
            load_stage(s);
            const int n_stage_tiles = s_stage.n_tiles, total = n_stage_tiles * P.n_agents;
            for (int wi = blockIdx.x; wi < total; wi += gridDim.x) {
                const int agent = wi / n_stage_tiles;
                int tile;
                const Task *tg = fetch_task(wi % n_stage_tiles, tile, wi == (int)blockIdx.x);
                if (!dep_synced) {
                    if constexpr (kTc && (kTypes & tb(T_GEMM)) != 0) {
                        if (s_task.type == T_GEMM && s_task.i[6] && tc_setup && stage_end - stage_begin == 1) tc::tc_prefetch_b(s_task, tg, tile, agent, st, P.error_flag);
                    }
                    dep_sync();
                }
                run_task(tg, tile, agent, wi == (int)blockIdx.x);
            }
            if (s + 1 < stage_end) {
                bar_target += gridDim.x;
                grid_barrier(P.barrier, bar_target, P.error_flag);
            }
        }
    } else if constexpr (variant_chains(kMath, kTypes, kEpis)) {
        // chained launch (one agent): cluster c < chain_clusters owns its row block in every stage of the chain, rank r its column tile r;
        // a cluster stops behind the last stage that has a tile for it (a uniform decision: the map is per cluster).  The other clusters
        // walk the riders (T_SHADOW tasks of the chain's stages, independent of the chain) without barriers.
        const uint32_t cw = tc::cluster_nctarank(), r = tc::cluster_ctarank();
        const int c = (int)(blockIdx.x / cw);
        load_stage(stage_begin);
        const int n_row = s_stage.chain_clusters;
        if (c < n_row) {
            int e = s_stage.chain_map[c], tile = 0;
            bool have = e >= 0 && (int)r < (e >> 16);
            const Task *tg = have ? fetch_task((e & 0xffff) + (int)r, tile, true) : nullptr;
            dep_sync();
            for (int s = stage_begin;; s++) {
                if (have) run_task(tg, tile, 0, s == stage_begin);
                if (s + 1 == stage_end) break;
                load_stage(s + 1);
                e = s_stage.chain_map[c];
                if (e < 0) break;
                have = (int)r < (e >> 16);
                if (have) {      // the next layer's weights do not depend on this layer: request their first K blocks now
                    tg = fetch_task((e & 0xffff) + (int)r, tile, false);
                    tc::tc_prefetch_b(s_task, tg, tile, 0, st, P.error_flag);
                }
                chain_barrier(cw);
            }
        } else {
            const int rider = (int)blockIdx.x - n_row * (int)cw, n_riders = (int)gridDim.x - n_row * (int)cw;
            dep_sync();
            int base = 0;      // riders of all stages of the chain as one list, dealt round-robin
            for (int s = stage_begin; s < stage_end; s++) {
                if (s != stage_begin) load_stage(s);
                for (int k = 0; k < s_stage.task_end - s_stage.task_begin; k++) {
                    const int tb0 = s_stage.tile_begin[k];
                    int tile;
                    const Task *tg = fetch_task(tb0, tile, false);
                    if (s_task.type == T_GEMM) continue;
                    for (int i = ((rider - base) % n_riders + n_riders) % n_riders; i < s_task.n_tiles; i += n_riders) run_task(tg, i, 0, false);
                    base += s_task.n_tiles;
                }
            }
        }
    }

    if (!dep_synced) {           // a CTA without a tile still has to release its dependents
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    }
    if (kTc && (kTypes & tb(T_GEMM)) != 0 && tc_setup) {
        tc::tc_fence_before();
        __syncthreads();
        if (threadIdx.x < 32) tc::tmem_dealloc(st.tmem_base, kTN);
    }
    stamp(5);
    timeline(2, true);
}

// throughput form of a stage that holds only GEMM tasks (stream.cuh): one resident CTA per SM, roles decoupled across tiles
__global__ void __launch_bounds__(stream::kThreads, 1)
sac_stream_kernel(const __grid_constant__ Program P, const __grid_constant__ Stage stage, const uint64_t seed) {
    extern __shared__ __align__(1024) uint8_t smem_stream[];
    if ((tc::smem_u32(smem_stream) & 1023u) != 0) {      // SWIZZLE_128B operand tiles need 1024-byte alignment; the kernel owns all 227 KB
        if (threadIdx.x == 0) atomicExch(P.error_flag, 3);
        return;
    }
    stream::gemm_stage(P, stage, smem_stream, seed);
}

// ================================================================================================================
// program builder
// ================================================================================================================
namespace {

// a pair-matrix view together with its logical extent (what the TMA descriptor is built from)
struct PmView {
    PmRef ref;
    int rows, cols;     // stored extent of the view: rows x cols valid elements
};

struct Builder {
    sacb_handle h;
    const Layout &L;
    ProgramKey key;
    std::vector<Task> tasks;
    std::vector<Stage> stages;
    std::vector<int> has_gemm;
    int tm, tn;   // default GEMM tile dims of the math mode
    int rc = SACB_OK;
    // tensor-core tile shape per task index (bm, bn), decided by choose_tile_shapes() from a dry first pass; empty = defaults
    std::vector<std::pair<int, int>> shapes;
    std::map<int64_t, int> shadow_writer;      // arena offset of a weight shadow PM -> last stage of THIS program that writes it
    bool dry = false;      // first pass: count tiles only, no TMA descriptors
    bool stream = false;   // throughput program: GEMM stages run on the stream kernel (it alone understands split-K tasks)

    Builder(sacb_handle h_, const ProgramKey &k) : h(h_), L(h_->L), key(k) {
        if (math_is_tc(h->cfg.math_mode)) { tm = kTM; tn = kTN; } else { tm = kSM; tn = kSN; }
    }
    static Ref A(int64_t off) { return make_ref(0, off); }
    static Ref W(int64_t off) { return make_ref(1, off); }

    // view of rows [row0, row0+rows) x cols of a PM whose hi plane starts at float offset `off` of `region`,
    // has row stride ld and `plane_rows` rows per plane
    static PmView view(int region, int64_t off, int ld, int64_t plane_rows, int row0, int rows, int cols) {
        PmView v;
        v.ref.base = make_ref(region, off + (int64_t)row0 * ld / 2);
        v.ref.ld = ld; v.ref.pad = 0; v.ref.plane = plane_rows * ld;
        v.rows = rows; v.cols = cols;
        return v;
    }
    // activations / gradients [B,H] in the workspace (planes sized for maxB rows)
    PmView hview(int64_t off, int rows, int row0 = 0, int plane_mult = 1) const {
        return view(1, off, L.hidden, (int64_t)plane_mult * L.maxB, row0, rows, L.hidden);
    }
    PmView xrows(int row0, int rows, int cols) const { return view(1, L.X, L.ldx, 3 * (int64_t)L.maxB, row0, rows, cols); }
    PmView ghead(int rows) const { return view(1, L.g_head, L.ldg, L.maxB, 0, rows, 2 * L.act); }
    // weight shadows in the arena
    PmView wsh(int net, int l) const {
        const NetLayout &n = net == 0 ? L.pol : L.q;
        return view(0, L.shadow[net] + n.sh_w[l], n.sh_ld[l], L.hidden, 0, L.hidden, n.in_of(l));
    }
    PmView wsh_act(int net) const { return view(0, L.shadow[net] + L.q.sh_act, L.q.sh_act_ld, L.hidden, 0, L.hidden, L.act); }
    PmView wsh_head() const { return view(0, L.shadow[0] + L.pol.sh_out, L.hidden, 2 * L.act, 0, 2 * L.act, L.hidden); }

    void begin_stage() {
        Stage s{}; s.task_begin = (int)tasks.size(); s.task_end = s.task_begin; s.n_tiles = 0;
        stages.push_back(s); has_gemm.push_back(0);
    }
    Task blank(int type) {
        Task t; memset(&t, 0, sizeof(t));
        t.type = type;
        t.C = t.bias = null_ref();
        t.Cpm = t.mask = t.A.pm = t.B.pm = null_pm();
        t.adam.w = t.adam.m = t.adam.v = t.adam.wt = t.adam.gexp = null_ref();
        t.adam.shadow = t.adam.shadow2 = t.adam.shadow_t = null_pm();
        for (auto &p : t.p) p = null_ref();
        for (auto &p : t.pm) p = null_pm();
        return t;
    }
    void add(Task t, int n_tiles) {
        Stage &s = stages.back();
        if (s.task_end - s.task_begin >= kMaxStageTasks) { rc = fail(SACB_ERR_ARG, "too many tasks in one stage"); return; }
        s.tile_begin[s.task_end - s.task_begin] = s.n_tiles;
        t.tile_begin = s.n_tiles; t.n_tiles = n_tiles;
        s.n_tiles += n_tiles; s.task_end++;
        if (t.type == T_GEMM) has_gemm.back() = 1;
        tasks.push_back(t);
    }
    void *dev_ptr(Ref r) const {
        const int64_t off = r.v & ((1ll << 62) - 1);
        return ((r.v >> 62) & 1) ? (void *)(h->ws + off) : (void *)(h->arena + off);
    }
    int64_t agent_stride_bytes(Ref r) const { return (((r.v >> 62) & 1) ? L.ws_size : L.arena_size) * (int64_t)sizeof(float); }

    // C[M,N] = A[M,K] . B[N,K]^T with A, B taken from PM views.  mn_major = 0: the view stores [R, K]; 1: it stores [K, R].
    // b_r0: the B operand is rows/columns [b_r0, b_r0+N) of the view along its N dimension (TMA boxes need no alignment).
    void gemm(const PmView &a, int a_mn, const PmView &b, int b_mn, int M, int N, int K, Task t, int b_r0 = 0) {
        t.type = T_GEMM; t.M = M; t.N = N; t.K = K;
        t.A.pm = a.ref; t.A.mn_major = a_mn; t.A.r0 = 0; t.B.pm = b.ref; t.B.mn_major = b_mn; t.B.r0 = b_r0;
        const size_t idx = tasks.size();
        {   // B = a weight shadow (arena PM) that no stage later than two back has written: may be requested before the grid-dependency
            // wait (gemm.cuh: tc_prefetch_b).  Writers: T_SHADOW tasks and Adam epilogues; the stage right before may still be running
            const int cur = (int)stages.size() - 1;
            const bool in_arena = ((b.ref.base.v >> 62) & 1) == 0;
            const auto w = shadow_writer.find(b.ref.base.v);
            // (opt-in, SACB_EARLY_B=1: measured no gain on B200 -- 0.1990 vs 0.1984 ms -- because with one 193 KB CTA per SM only the
            //  ~20 CTAs of a stage that land on SMs the previous stage left idle are resident before the release at all)
            t.i[6] = (in_arena && !stream && (w == shadow_writer.end() || w->second <= cur - 2) && getenv("SACB_EARLY_B")) ? 1 : 0;
            for (const PmRef *r : {&t.adam.shadow, &t.adam.shadow2}) if (!is_null(r->base)) shadow_writer[r->base.v] = cur;
        }
        t.bm = idx < shapes.size() && shapes[idx].first ? shapes[idx].first : tm;
        t.bn = idx < shapes.size() && shapes[idx].second ? shapes[idx].second : tn;
        t.tiles_m = cdiv(M, t.bm); t.tiles_n = cdiv(N, t.bn);
        if (math_is_tc(h->cfg.math_mode) && rc == SACB_OK && !dry) {
            // stored extents: K-major [R, K] -> cols = K ; MN-major [K, R] -> cols = R.  TMA zero-fills beyond them.
            const int a_cols = a_mn ? M : K, a_rows = a_mn ? K : M, b_cols = b_mn ? b_r0 + N : K, b_rows = b_mn ? K : b_r0 + N;
            rc = make_pm_tensor_map(&t.tmA, dev_ptr(a.ref.base), a_cols, a_rows, a.ref.ld, a.ref.plane, agent_stride_bytes(a.ref.base),
                                    h->cfg.n_agents, a_mn ? 64 : t.bm);
            if (rc == SACB_OK)
                rc = make_pm_tensor_map(&t.tmB, dev_ptr(b.ref.base), b_cols, b_rows, b.ref.ld, b.ref.plane, agent_stride_bytes(b.ref.base),
                                        h->cfg.n_agents, b_mn ? 64 : t.bn);
        }
        int n_chunks = 1;
        if (stream && t.epi == EPI_ADAM && !apply()) {      // gradient export over a long batch dimension: split K, accumulate with atomics
            const int nkb = cdiv(K, stream::kBK);
            n_chunks = std::max(1, std::min(16, nkb / 16));
            if (n_chunks > 1) t.i[7] = cdiv(nkb, n_chunks);
        }
        add(t, t.tiles_m * t.tiles_n * n_chunks);
    }
    Task epi_bias_relu(const PmView &C, Ref bias) { Task t = blank(T_GEMM); t.epi = EPI_BIAS_RELU; t.Cpm = C.ref; t.bias = bias; return t; }
    Task epi_mask(const PmView &C, const PmView &mask) { Task t = blank(T_GEMM); t.epi = EPI_MASK; t.Cpm = C.ref; t.mask = mask.ref; return t; }
    Task epi_f32(Ref C, int ldc, Ref bias) { Task t = blank(T_GEMM); t.epi = EPI_F32; t.C = C; t.ldc = ldc; t.bias = bias; return t; }

    // rows per tile of a column-sum task (bias / output-layer gradients).  A program that only EXPORTS gradients (data-parallel
    // backward: the slab is zeroed at the start of the step) cuts large batches into chunks of 1024 rows accumulated with atomics,
    // so that the reduction over the batch spreads over the SMs; a program that applies Adam keeps one (deterministic) chunk
    int colsum_rows(int Bn) const { return (!apply() && Bn > 2048) ? 1024 : std::max(Bn, 1); }
    // which optimizer a trainable net (0 policy, 1 q1, 2 q2) uses
    static int step_slot(int net) { return net == 0 ? SC_STEP_POLICY : (net == 1 ? SC_STEP_Q1 : SC_STEP_Q2); }
    bool apply() const { return key.dp_phase < 0; }
    // A step that applies Adam leaves every shadow current, so that the next step runs without the shadow stage: the critics'
    // shadows are refreshed by their Adam epilogues (the actor phase of the SAME step reads them), the Polyak targets' and the
    // policy's by T_SHADOW tasks riding in later stages of the step that leave most SMs idle (actor-phase critic forward, policy
    // backward, finish) -- in the epilogue the two extra planes cost 1.2-1.8 us per Adam stage, there they cost nothing.
    bool keep_resident() const { return apply(); }
    // Throughput programs are bound by HBM traffic, not by stage latency: there every Adam epilogue writes the shadows of what it
    // steps (policy and Polyak targets included) straight from its registers -- no extra pass over the fp32 weights, no extra stages.
    bool epilogue_shadows() const { return stream && keep_resident(); }
    int loss_rows() const { return stream ? kLossRowsMax : kLossRows; }      // batch rows per tile of the two loss tasks (tasks.cuh)
    bool task_shadows() const { return !stream && keep_resident(); }
    bool exporting() const { return key.export_grads || key.dp_phase >= 0; }

    AdamArgs adam_args(int net, int64_t off_in_net) {
        AdamArgs a;
        a.w = A(L.param[net] + off_in_net); a.m = A(L.adam_m[net] + off_in_net); a.v = A(L.adam_v[net] + off_in_net);
        a.wt = net == 0 ? null_ref() : A(L.param[net + 2] + off_in_net);     // q1 -> q1_target, q2 -> q2_target
        a.gexp = exporting() ? A(L.grad[net] + off_in_net) : null_ref();
        a.shadow = a.shadow2 = a.shadow_t = null_pm(); a.shadow2_col0 = 0; a.pad0 = 0;
        a.step_slot = step_slot(net); a.apply = apply() ? 1 : 0;
        a.lr = h->cfg.lr; a.tau = h->cfg.tau;
        return a;
    }
    // dW epilogue of hidden layer `layer`: the critics are read again (post-step) by the actor phase of the SAME update,
    // so their shadows are refreshed in the epilogue; policy / target shadows are refreshed at the start of the next step
    Task epi_adam(int net, int layer) {
        const NetLayout &n = net == 0 ? L.pol : L.q;
        Task t = blank(T_GEMM); t.epi = EPI_ADAM; t.adam = adam_args(net, n.w[layer]);
        // (latency programs: the two policy layers stepped by the LAST backward stage refresh their shadows in the epilogue as well:
        //  +1.2 us on that stage, against +3 us for shadow tasks next to the single-CTA finish stage)
        if (net != 0 || epilogue_shadows() || (task_shadows() && layer <= 1)) t.adam.shadow = wsh(net, layer).ref;
        if (net != 0 && layer == 0) { t.adam.shadow2 = wsh_act(net).ref; t.adam.shadow2_col0 = L.obs; }
        if (net != 0 && epilogue_shadows()) t.adam.shadow_t = wsh(net + 2, layer).ref;
        return t;
    }

    void bias_adam(int net, int64_t b_off, const PmView &dh, int Bn, int N) {
        Task t = blank(T_BIAS_ADAM);
        t.pm[0] = dh.ref;
        AdamArgs a = adam_args(net, b_off);
        t.p[0] = a.w; t.p[1] = a.m; t.p[2] = a.v; t.p[3] = a.wt; t.p[4] = a.gexp;
        t.i[0] = Bn; t.i[1] = N; t.i[2] = a.step_slot; t.i[3] = a.apply; t.f[0] = a.lr; t.f[1] = a.tau;
        t.i[5] = colsum_rows(Bn);
        add(t, cdiv(N, kColsumCols) * cdiv(Bn, t.i[5]));
    }
    // ---- opt-in LayerNorm variant (cfg.layer_norm): hidden layer = Linear -> LayerNorm (affine) -> ReLU.  The forward GEMM then writes the
    // Linear output z as fp32 (EPI_F32 with the bias) and a T_LN_FWD stage behind it normalises the rows into the activation PM; a
    // backward GEMM / loss task still writes the gradient at the ReLU input (mask applied) into the dh PM -- which is now the gradient at
    // the LayerNorm OUTPUT -- and a T_LN_BWD stage turns it into dz, the gradient at the Linear output, in its own PM; dgamma / dbeta
    // are column sums over the batch (T_BIAS_ADAM) of dpre * xhat and dpre.
    bool ln() const { return L.layer_norm; }
    Task fwd_epi(const PmView &hout, Ref bias, int64_t z_off) { return ln() ? epi_f32(W(z_off), L.hidden, bias) : epi_bias_relu(hout, bias); }
    void ln_fwd(int net, int l, int64_t z_off, int64_t st_off, const PmView &hout, int rows) {
        const NetLayout &n = net == 0 ? L.pol : L.q;
        Task t = blank(T_LN_FWD);
        t.p[0] = W(z_off); t.p[1] = A(L.param[net] + n.g[l]); t.p[2] = A(L.param[net] + n.be[l]); t.p[3] = W(st_off);
        t.pm[0] = hout.ref; t.i[0] = rows; t.i[1] = L.hidden; t.f[0] = 1e-5f;      // torch.nn.LayerNorm default eps
        add(t, cdiv(rows, kLnRows));
    }
    void ln_bwd(int net, int l, const PmView &dpre, int64_t z_off, int64_t st_off, const PmView &dz, const PmView *gg, int rows) {
        const NetLayout &n = net == 0 ? L.pol : L.q;
        Task t = blank(T_LN_BWD);
        t.pm[0] = dpre.ref; t.p[0] = W(z_off); t.p[1] = A(L.param[net] + n.g[l]); t.p[3] = W(st_off);
        t.pm[1] = dz.ref; t.pm[2] = gg ? gg->ref : null_pm(); t.i[0] = rows; t.i[1] = L.hidden;
        add(t, cdiv(rows, kLnRows));
    }
    // Adam on gamma / beta of hidden layer l of a trainable net: column sums of dpre * xhat (gg) and of dpre
    void ln_param_adam(int net, int l, const PmView &gg, const PmView &dpre, int Bn) {
        const NetLayout &n = net == 0 ? L.pol : L.q;
        bias_adam(net, n.g[l], gg, Bn, L.hidden);
        bias_adam(net, n.be[l], dpre, Bn, L.hidden);
    }

    // shadow of columns [col0, col0+dst.cols) of the fp32 matrix at w_off (row stride src_ld)
    void shadow_task(int net, int64_t w_off, const PmView &dst, int src_ld, int col0 = 0) {
        Task t = blank(T_SHADOW);
        t.p[0] = A(L.param[net] + w_off); t.pm[0] = dst.ref; t.i[0] = dst.rows; t.i[1] = dst.cols; t.i[2] = col0; t.i[3] = src_ld;
        shadow_writer[dst.ref.base.v] = (int)stages.size() - 1;
        add(t, cdiv(dst.rows, kShadowRows));
    }

    // Tile shapes of a latency-bound program (tensor-core math, few agents).  A stage is as slow as its slowest CTA, a CTA's
    // main loop is bound by the per-SM L2 -> shared-memory ingest (~90 GB/s, profiles/r01_summary.md) and a 128 x 64 stage
    // keeps only 32-64 of the SMs busy.  So while the stage still fits into one wave, the most expensive task is cut into
    // smaller tiles: 128 -> 64 rows (tcgen05 M = 64) first, then 64 -> 32 columns where B is K-major and the epilogue is not
    // the Adam one.  Results do not depend on the shape (the K order of every output element is unchanged).
    static double tile_cost_us(const Task &t, int bm, int bn) {
        const double ingest = (double)(bm + bn) * std::min(t.K, 1 << 20) * 4.0 / 90e3;          // both planes, 2 B each
        const double epi = (t.epi == EPI_ADAM ? 6.0 : 1.4) * (double)(bm * bn) / (kTM * kTN);  // measured per 128 x 64 tile
        return ingest + epi;
    }
    std::vector<std::pair<int, int>> choose_tile_shapes(int wave) const {
        std::vector<std::pair<int, int>> out(tasks.size(), {0, 0});
        if (!math_is_tc(h->cfg.math_mode) || getenv("SACB_FIXED_TILES")) return out;
        for (size_t si = 0; si < stages.size(); si++) {
            const Stage &sg = stages[si];
            if (!has_gemm[si]) continue;
            struct Cand { int task, bm, bn, tiles; bool frozen; };
            std::vector<Cand> c;
            int total = 0;
            for (int k = sg.task_begin; k < sg.task_end; k++) {
                total += tasks[k].n_tiles * h->cfg.n_agents;
                if (tasks[k].type == T_GEMM) c.push_back({k, kTM, kTN, tasks[k].n_tiles, false});
            }
            while (true) {
                int best = -1; double best_cost = 0;
                for (size_t i = 0; i < c.size(); i++) {
                    if (c[i].frozen) continue;
                    const double cost = tile_cost_us(tasks[c[i].task], c[i].bm, c[i].bn);
                    if (cost > best_cost) { best_cost = cost; best = (int)i; }
                }
                if (best < 0) break;
                Cand &b = c[best];
                const Task &t = tasks[b.task];
                int nbm = b.bm, nbn = b.bn;
                if (b.bm == kTM && t.M > 64) nbm = 64;
                else if (b.bn == kTN && !t.B.mn_major && t.epi != EPI_ADAM && t.epi != EPI_SAMPLE && t.N > 32) nbn = 32;
                else { b.frozen = true; continue; }
                const int ntiles = cdiv(t.M, nbm) * cdiv(t.N, nbn);
                if (total + (ntiles - b.tiles) * h->cfg.n_agents > wave) { b.frozen = true; continue; }
                total += (ntiles - b.tiles) * h->cfg.n_agents;
                b.bm = nbm; b.bn = nbn; b.tiles = ntiles;
            }
            for (const Cand &x : c) out[x.task] = {x.bm, x.bn};
        }
        return out;
    }

    // Throughput programs (stages with many more tiles than SMs): every GEMM task takes the stream kernel's tile, 128 rows x 128
    // columns (64 where the output is narrower than 96 columns: policy heads, dL/da).
    // A stage that would hold fewer than kStreamWideMin x SMs tiles of 128 x 128 keeps 64-column tiles: twice the tiles for the
    // round-robin over the resident CTAs (mid-size batches: better wave quantisation and more tiles to overlap per CTA).
    std::vector<std::pair<int, int>> stream_tile_shapes() const {
        static const int wide_min = getenv("SACB_STREAM_WIDE_MIN") ? atoi(getenv("SACB_STREAM_WIDE_MIN")) : 3;
        // 128 x 256 tiles (two 96 KB ring slots, both 256-column accumulators) where the stage still holds kStreamN256Min x SMs of them:
        // 0.75x the L2 -> SM operand traffic per flop of the 128 x 128 tile, which is what bounds a large-batch GEMM stage
        // (SACB_STREAM_N256_MIN: waves of 256-wide tiles a stage needs, 0 = never).  Not where a task of the stage has only a handful
        // of tiles (the K = batch dW GEMMs of a fused-Adam program, 8-16 tiles of a thousand K blocks each, sharing a stage with the
        // dX GEMMs): those tiles are the stage's long pole, halving their number or their ring slots costs more than the wide tiles save
        const int n256_min = getenv("SACB_STREAM_N256_MIN") ? atoi(getenv("SACB_STREAM_N256_MIN")) : 1;      // read per program build (tests A/B both forms in one process)
        // no extra padding against 128-wide tiles; a tile that steps weights keeps 128 columns (its stage gives 64 KB of the ring to the
        // optimizer-state landing zone of the Adam epilogue: two 64 KB slots are left)
        const bool applies = apply();      // (256-column weight-stepping tiles on a one-slot ring were measured: no gain, 691 -> 786 us on a mixed stage)
        auto takes_256 = [applies](const Task &t) { return t.N >= 192 && cdiv(t.N, 256) * 256 <= cdiv(t.N, 128) * 128 && !(t.epi == EPI_ADAM && applies); };
        std::vector<std::pair<int, int>> out(tasks.size(), {0, 0});
        for (size_t si = 0; si < stages.size(); si++) {
            int wide_tiles = 0, tiles_256 = 0;
            bool all_many = true;
            for (int k = stages[si].task_begin; k < stages[si].task_end; k++)
                if (tasks[k].type == T_GEMM) {
                    // split-K chunks a gradient-export dW GEMM will be cut into (gemm(): the dry pass itself does not split)
                    const int chunks = (tasks[k].epi == EPI_ADAM && !apply()) ? std::max(1, std::min(16, cdiv(tasks[k].K, stream::kBK) / 16)) : 1;
                    wide_tiles += cdiv(tasks[k].M, stream::kBM) * cdiv(tasks[k].N, tasks[k].N >= 96 ? stream::kBN : 64) * h->cfg.n_agents;
                    const int t256 = cdiv(tasks[k].M, stream::kBM) * cdiv(tasks[k].N, takes_256(tasks[k]) ? 256 : (tasks[k].N >= 96 ? stream::kBN : 64)) * chunks * h->cfg.n_agents;
                    tiles_256 += t256;
                    all_many = all_many && 2 * t256 >= h->sm_count;
                }
            const bool wide = wide_tiles >= wide_min * h->sm_count;
            const bool very_wide = n256_min > 0 && all_many && tiles_256 >= n256_min * h->sm_count;
            for (int k = stages[si].task_begin; k < stages[si].task_end; k++)
                if (tasks[k].type == T_GEMM) out[k] = {stream::kBM, (very_wide && takes_256(tasks[k])) ? 256 : ((wide && tasks[k].N >= 96) ? stream::kBN : 64)};
        }
        return out;
    }
    // ... and a stage that mixes GEMM tasks with column-sum / element-wise tasks is cut in two (the tasks of a stage are independent
    // of each other): first the non-GEMM tasks on the generic stage kernel, then the GEMM tasks on the stream kernel.
    void split_mixed_stages(std::vector<int> &stage_stream) {
        std::vector<Task> nt;
        std::vector<Stage> ns;
        std::vector<int> ng;
        stage_stream.clear();
        auto emit = [&](const std::vector<Task> &ts, bool gemm) {
            Stage sg{};
            sg.task_begin = (int)nt.size(); sg.n_tiles = 0;
            for (size_t i = 0; i < ts.size(); i++) {
                Task t = ts[i];
                sg.tile_begin[i] = sg.n_tiles; t.tile_begin = sg.n_tiles; sg.n_tiles += t.n_tiles;
                nt.push_back(t);
            }
            sg.task_end = (int)nt.size();
            ns.push_back(sg); ng.push_back(gemm ? 1 : 0); stage_stream.push_back(gemm ? 1 : 0);
        };
        for (size_t si = 0; si < stages.size(); si++) {
            std::vector<Task> g, o;
            for (int k = stages[si].task_begin; k < stages[si].task_end; k++) (tasks[k].type == T_GEMM ? g : o).push_back(tasks[k]);
            if (!o.empty()) emit(o, false);
            if (!g.empty()) emit(g, true);
        }
        tasks.swap(nt); stages.swap(ns); has_gemm.swap(ng);
    }

    void build() {
        const int B = key.B, H = L.hidden, nh = L.n_hidden, obs = L.obs, act = L.act, A2 = 2 * act;
        const NetLayout &P = L.pol, &Q = L.q;
        const bool critics = key.dp_phase != 1, actor = key.dp_phase != 0;
        // X PM rows: [0,B) = (s2, a2)   [B,2B) = (s, a)   [2B,3B) = (s, a_new)
        auto X2 = [&](int cols) { return xrows(0, B, cols); };
        auto X1 = [&](int cols) { return xrows(B, B, cols); };
        auto X3 = [&](int cols) { return xrows(2 * B, B, cols); };

        // ---- stage: weight shadows (+ minibatch gather) --------------------------------------------------------
        const bool shadow_stage = !key.resident;
        if (shadow_stage || (key.with_gather && critics)) begin_stage();
        for (int net = 0; net < 5 && shadow_stage; net++) {
            if (!critics && (net == 3 || net == 4)) continue;      // the actor phase does not read the targets
            const NetLayout &n = net == 0 ? P : Q;
            for (int l = 0; l < nh; l++) shadow_task(net, n.w[l], wsh(net, l), n.in_of(l));
            if (net == 0) shadow_task(0, P.w_out, wsh_head(), H);
            if ((net == 1 || net == 2) && actor) shadow_task(net, Q.w[0], wsh_act(net), obs + act, obs);
        }
        if (key.with_gather && critics) {
            Task t = blank(T_GATHER);
            t.pm[0] = xrows(0, 3 * B, L.ldx).ref; t.p[0] = W(L.r); t.p[1] = W(L.d);
            t.i[0] = B; t.i[1] = obs; t.i[2] = act;
            t.i[3] = key.with_gather == 3 ? 1 : 0;      // 3: positions drawn on the device (uniform ring), see draw_position
            t.i[4] = (int32_t)h->cfg.capacity;
            add(t, cdiv(B, 4));
        }
        if (critics) {
            // ---- policy forward on [s2 ; s] (M = 2B) + critic forward on (s,a), layer by layer ---------------------
            for (int l = 0; l < nh; l++) {
                begin_stage();
                const int in_p = P.in_of(l), in_q = Q.in_of(l);
                gemm(l == 0 ? xrows(0, 2 * B, obs) : hview(L.hp[l - 1], 2 * B, 0, 2), 0, wsh(0, l), 0, 2 * B, H, in_p,
                     fwd_epi(hview(L.hp[l], 2 * B, 0, 2), A(L.param[0] + P.b[l]), L.zp[l]));
                for (int k = 0; k < 2; k++)
                    gemm(l == 0 ? X1(obs + act) : hview(L.hc[k][l - 1], B), 0, wsh(1 + k, l), 0, B, H, in_q,
                         fwd_epi(hview(L.hc[k][l], B), A(L.param[1 + k] + Q.b[l]), L.zc[k][l]));
                if (ln()) {
                    begin_stage();
                    ln_fwd(0, l, L.zp[l], L.sp[l], hview(L.hp[l], 2 * B, 0, 2), 2 * B);
                    for (int k = 0; k < 2; k++) ln_fwd(1 + k, l, L.zc[k][l], L.sc[k][l], hview(L.hc[k][l], B), B);
                }
            }
            // ---- policy heads -> head_raw [2B, 2A] (fp32) ------------------------------------------------------------
            // opt-in experiment (SACB_FUSE_SAMPLE=1, tensor-core math, 2A <= 64): the tanh-Gaussian sample + log-prob of both batches
            // in the epilogue of the heads GEMM (EPI_SAMPLE, one stage less).  Correct (parity tests pass) but slower on B200: the
            // heads GEMM has only 2B / 64 = 8 tiles, so 8 SMs do the transcendental-heavy sampling of 512 rows (13.8 us) that the
            // separate stage spreads over 32 CTAs (4 us + 1 us stage boundary); profiles/r01_summary.md
            const bool fuse_sample = math_is_tc(h->cfg.math_mode) && A2 <= kTN && getenv("SACB_FUSE_SAMPLE");
            begin_stage();
            if (fuse_sample) {
                Task t = epi_f32(W(L.head_raw), A2, A(L.param[0] + P.b_out));
                t.epi = EPI_SAMPLE;
                t.p[1] = W(L.eps); t.pm[0] = xrows(0, 3 * B, L.ldx).ref; t.p[3] = W(L.logp);
                t.i[0] = B; t.i[1] = act; t.i[2] = obs; t.i[4] = key.device_eps;
                t.f[0] = h->cfg.action_scale; t.f[1] = h->cfg.action_bias;
                gemm(hview(L.hp[nh - 1], 2 * B, 0, 2), 0, wsh_head(), 0, 2 * B, A2, H, t);
            } else {
                gemm(hview(L.hp[nh - 1], 2 * B, 0, 2), 0, wsh_head(), 0, 2 * B, A2, H, epi_f32(W(L.head_raw), A2, A(L.param[0] + P.b_out)));
            }
            // ---- reparameterised sample + log-prob for both batches -------------------------------------------------
            if (!fuse_sample) {
                begin_stage();
                Task t = blank(T_SAMPLE);
                t.p[0] = W(L.head_raw); t.p[1] = W(L.eps); t.pm[0] = xrows(0, 3 * B, L.ldx).ref; t.p[3] = W(L.logp);
                t.i[0] = B; t.i[1] = act; t.i[2] = obs; t.i[4] = key.device_eps;
                t.f[0] = h->cfg.action_scale; t.f[1] = h->cfg.action_bias;
                add(t, cdiv(2 * B, kThreads / 32));
            }
            // ---- target critics on (s2, a2) ---------------------------------------------------------------------------
            for (int l = 0; l < nh; l++) {
                begin_stage();
                const int in_q = Q.in_of(l);
                for (int k = 0; k < 2; k++)
                    gemm(l == 0 ? X2(obs + act) : hview(L.ht[k][l - 1], B), 0, wsh(3 + k, l), 0, B, H, in_q,
                         fwd_epi(hview(L.ht[k][l], B), A(L.param[3 + k] + Q.b[l]), L.zt[k][l]));
                if (ln()) {
                    begin_stage();
                    for (int k = 0; k < 2; k++) ln_fwd(3 + k, l, L.zt[k][l], L.st[k][l], hview(L.ht[k][l], B), B);
                }
            }
            // ---- Bellman target, critic losses, dL/dq, dL/dh of the last hidden layer --------------------------------
            begin_stage();
            {
                Task t = blank(T_TARGET_LOSS);
                t.pm[0] = hview(L.ht[0][nh - 1], B).ref; t.pm[1] = hview(L.ht[1][nh - 1], B).ref;
                t.pm[2] = hview(L.hc[0][nh - 1], B).ref; t.pm[3] = hview(L.hc[1][nh - 1], B).ref;
                t.pm[4] = hview(L.dhc[0][nh - 1], B).ref; t.pm[5] = hview(L.dhc[1][nh - 1], B).ref;
                const int nets[4] = {3, 4, 1, 2};
                for (int k = 0; k < 4; k++) { t.p[4 + k] = A(L.param[nets[k]] + Q.w_out); t.p[8 + k] = A(L.param[nets[k]] + Q.b_out); }
                t.p[12] = W(L.r); t.p[13] = W(L.d); t.p[14] = W(L.logp); t.p[15] = key.use_isw ? W(L.isw) : null_ref();
                t.p[16] = W(L.y); t.p[17] = W(L.dq[0]); t.p[18] = W(L.dq[1]); t.p[19] = W(L.td);
                t.p[22] = W(L.loss_part);
                t.i[0] = B; t.i[1] = H; t.i[2] = loss_rows(); t.f[0] = h->cfg.gamma;
                add(t, cdiv(B, loss_rows()));
            }
            // gradient at the Linear output of critic k's hidden layer x: the dh PM itself, or (LayerNorm variant) the dz PM behind it
            auto DZC = [&](int k, int x) { return ln() ? hview(L.dzc[k][x], B) : hview(L.dhc[k][x], B); };
            auto ln_bwd_c = [&](int x) {      // own stage: dpre -> dz of layer x of both critics
                if (!ln()) return;
                begin_stage();
                for (int k = 0; k < 2; k++) {
                    const PmView gg = hview(L.ggc[k][x], B);
                    ln_bwd(1 + k, x, hview(L.dhc[k][x], B), L.zc[k][x], L.sc[k][x], hview(L.dzc[k][x], B), &gg, B);
                }
            };
            ln_bwd_c(nh - 1);
            // ---- critic backward --------------------------------------------------------------------------------------
            //   stage s (1..nh): dX of layer l = nh-s (0-based, only while l >= 1) ; dW/db of layer l+1 ; last stage: dW/db of layer 0
            for (int s = 1; s <= nh; s++) {
                begin_stage();
                const int l = nh - s;          // layer whose dX is produced now (needs dh_l, writes dh_{l-1})
                for (int k = 0; k < 2; k++) {
                    const int net = 1 + k;
                    if (l >= 1)   // dh_{l-1} = (dh_l . W_l) * relu'(h_{l-1})
                        gemm(DZC(k, l), 0, wsh(net, l), 1, B, Q.in_of(l), H, epi_mask(hview(L.dhc[k][l - 1], B), hview(L.hc[k][l - 1], B)));
                    auto dW = [&](int layer) {   // dW_layer = dh_layer^T . x_layer ; fused Adam + Polyak + shadow refresh
                        const int in = Q.in_of(layer);
                        gemm(DZC(k, layer), 1, layer == 0 ? X1(in) : hview(L.hc[k][layer - 1], B), 1, H, in, B, epi_adam(net, layer));
                        bias_adam(net, Q.b[layer], DZC(k, layer), B, H);
                        if (ln()) ln_param_adam(net, layer, hview(L.ggc[k][layer], B), hview(L.dhc[k][layer], B), B);
                    };
                    if (l + 1 <= nh - 1) dW(l + 1);
                    if (s == nh) dW(0);
                    if (s == 1) {   // output layer
                        Task t = blank(T_OUT_ADAM);
                        AdamArgs aw = adam_args(net, Q.w_out), ab = adam_args(net, Q.b_out);
                        t.pm[0] = hview(L.hc[k][nh - 1], B).ref; t.p[1] = W(L.dq[k]);
                        t.p[2] = aw.w; t.p[3] = aw.m; t.p[4] = aw.v; t.p[5] = aw.wt; t.p[6] = aw.gexp;
                        t.p[7] = ab.w; t.p[8] = ab.m; t.p[9] = ab.v; t.p[10] = ab.wt; t.p[11] = ab.gexp;
                        t.i[0] = B; t.i[1] = H; t.i[2] = aw.step_slot; t.i[3] = aw.apply; t.f[0] = aw.lr; t.f[1] = aw.tau;
                        t.i[5] = colsum_rows(B);
                        add(t, (cdiv(H, kColsumCols) + 1) * cdiv(B, t.i[5]));      // + the bias tile, per row chunk
                    }
                }
                if (l >= 1) ln_bwd_c(l - 1);
            }
        }
        if (actor) {
            // ---- actor: updated critics on (s, a_new) ----------------------------------------------------------------
            for (int l = 0; l < nh; l++) {
                begin_stage();
                const int in_q = Q.in_of(l);
                for (int k = 0; k < 2; k++)
                    gemm(l == 0 ? X3(obs + act) : hview(L.ha[k][l - 1], B), 0, wsh(1 + k, l), 0, B, H, in_q,
                         fwd_epi(hview(L.ha[k][l], B), A(L.param[1 + k] + Q.b[l]), L.za[k][l]));
                if (critics && task_shadows())      // the Polyak targets moved in the critic backward: one layer's shadows per stage
                    for (int k = 0; k < 2; k++) shadow_task(3 + k, Q.w[nh - 1 - l], wsh(3 + k, nh - 1 - l), Q.in_of(nh - 1 - l));
                if (ln()) {
                    begin_stage();
                    for (int k = 0; k < 2; k++) ln_fwd(1 + k, l, L.za[k][l], L.sa[k][l], hview(L.ha[k][l], B), B);
                }
            }
            begin_stage();
            {
                Task t = blank(T_ACTOR_LOSS);
                t.pm[0] = hview(L.ha[0][nh - 1], B).ref; t.pm[1] = hview(L.ha[1][nh - 1], B).ref;
                t.pm[2] = hview(L.dha[0][nh - 1], B).ref; t.pm[3] = hview(L.dha[1][nh - 1], B).ref;
                t.p[2] = A(L.param[1] + Q.w_out); t.p[3] = A(L.param[2] + Q.w_out);
                t.p[4] = A(L.param[1] + Q.b_out); t.p[5] = A(L.param[2] + Q.b_out);
                t.p[6] = W(L.logp + B); t.p[9] = W(L.aloss_part);
                t.i[0] = B; t.i[1] = H; t.i[2] = loss_rows(); t.f[0] = -(float)act;
                add(t, cdiv(B, loss_rows()));
            }
            // ---- dL/da through both critics (input gradients only: the Q weights are constants here, quirk Q2) -------
            auto DZA = [&](int k, int x) { return ln() ? hview(L.dza[k][x], B) : hview(L.dha[k][x], B); };
            auto ln_bwd_a = [&](int x) {
                if (!ln()) return;
                begin_stage();
                for (int k = 0; k < 2; k++) ln_bwd(1 + k, x, hview(L.dha[k][x], B), L.za[k][x], L.sa[k][x], hview(L.dza[k][x], B), nullptr, B);
            };
            ln_bwd_a(nh - 1);
            for (int s = 1; s <= nh; s++) {
                begin_stage();
                const int l = nh - s;
                for (int k = 0; k < 2; k++) {
                    const int net = 1 + k;
                    if (l >= 1)
                        gemm(DZA(k, l), 0, wsh(net, l), 1, B, H, H, epi_mask(hview(L.dha[k][l - 1], B), hview(L.ha[k][l - 1], B)));
                    else   // layer 0: only the action columns [obs, obs+act) of W_0 [H, obs+act] (their own shadow PM)
                        gemm(DZA(k, 0), 0, wsh_act(net), 1, B, act, H, epi_f32(W(L.da[k]), act, null_ref()));
                }
                if (l >= 1) ln_bwd_a(l - 1);
            }
            begin_stage();
            {
                Task t = blank(T_SAMPLE_BWD);
                t.p[0] = W(L.da[0]); t.p[1] = W(L.da[1]); t.p[2] = W(L.head_raw + (int64_t)B * A2); t.p[3] = W(L.eps + (int64_t)B * act);
                t.pm[0] = ghead(B).ref;
                t.i[0] = B; t.i[1] = act; t.f[0] = h->cfg.action_scale; t.f[1] = h->cfg.action_bias;
                add(t, cdiv(B * act, kThreads));
            }
            // ---- policy backward (current-state rows B..2B of the policy activations) --------------------------------
            //   stage 0: dh_{nh-1} from the heads ; stage s: dh_{nh-1-s}, dW of the layer above ; last: dW_0
            auto hp_cur = [&](int l) { return hview(L.hp[l], B, B, 2); };
            auto DZP = [&](int x) { return ln() ? hview(L.dzp[x], B) : hview(L.dhp[x], B); };
            auto ln_bwd_p = [&](int x) {      // the policy's current-state rows are rows B..2B of its z / statistics
                if (!ln()) return;
                begin_stage();
                const PmView gg = hview(L.ggp[x], B);
                ln_bwd(0, x, hview(L.dhp[x], B), L.zp[x] + (int64_t)B * H, L.sp[x] + 2 * (int64_t)B, hview(L.dzp[x], B), &gg, B);
            };
            for (int s = 0; s <= nh; s++) {
                begin_stage();
                if (s == 0) {
                    gemm(ghead(B), 0, wsh_head(), 1, B, H, A2, epi_mask(hview(L.dhp[nh - 1], B), hp_cur(nh - 1)));
                    ln_bwd_p(nh - 1);
                } else {
                    const int l = nh - s;      // dh_l available; produce dh_{l-1} (if l >= 1)
                    if (l >= 1)
                        gemm(DZP(l), 0, wsh(0, l), 1, B, H, H, epi_mask(hview(L.dhp[l - 1], B), hp_cur(l - 1)));
                    if (s == 1) {              // heads: dW = g^T h_{nh-1}
                        Task t = blank(T_GEMM); t.epi = EPI_ADAM; t.adam = adam_args(0, P.w_out);
                        if (epilogue_shadows()) t.adam.shadow = wsh_head().ref;
                        gemm(ghead(B), 1, hp_cur(nh - 1), 1, A2, H, B, t);
                        bias_adam(0, P.b_out, ghead(B), B, A2);
                    } else {
                        const int lw = l + 1;  // dW of the layer whose dX ran in the previous stage
                        gemm(DZP(lw), 1, hp_cur(lw - 1), 1, H, H, B, epi_adam(0, lw));
                        bias_adam(0, P.b[lw], DZP(lw), B, H);
                        if (ln()) ln_param_adam(0, lw, hview(L.ggp[lw], B), hview(L.dhp[lw], B), B);
                    }
                    if (s == nh) {
                        gemm(DZP(0), 1, X1(obs), 1, H, obs, B, epi_adam(0, 0));
                        bias_adam(0, P.b[0], DZP(0), B, H);
                        if (ln()) ln_param_adam(0, 0, hview(L.ggp[0], B), hview(L.dhp[0], B), B);
                    }
                    if (task_shadows()) {      // shadow of what the PREVIOUS stage stepped: heads (s-1 = 1) or hidden layer nh-s+2
                        if (s == 2) shadow_task(0, P.w_out, wsh_head(), H);
                        else if (s > 2) shadow_task(0, P.w[nh - s + 2], wsh(0, nh - s + 2), P.in_of(nh - s + 2));
                    }
                    if (l >= 1) ln_bwd_p(l - 1);
                }
            }
        }
        {   // own stage: the Adam epilogues of the previous stage still read the step counters
            begin_stage();
            Task t = blank(T_FINISH);
            const int ap = apply() ? 1 : 0;
            t.p[0] = critics ? W(L.loss_part) : null_ref();
            t.p[1] = actor ? W(L.aloss_part) : null_ref();
            t.p[2] = exporting() ? A(L.grad_scalars) : null_ref();
            t.p[3] = A(L.loss_hist);
            t.i[0] = ap; t.i[1] = ap; t.i[2] = ap; t.i[3] = ap && h->cfg.auto_entropy; t.i[4] = ap;
            t.i[5] = cdiv(B, loss_rows()) * (loss_rows() / kLossRows); t.i[6] = h->cfg.auto_entropy; t.i[7] = ap;
            t.f[0] = h->cfg.lr; t.f[1] = (float)B;
            add(t, 1);

        }
    }

};

// ---- chains of row-local GEMM stages (one launch of thread-block clusters each) -----------------------------------------------
// In consecutive MLP layers, row block r of layer l+1 reads only row block r of layer l, across all its columns: with 64 x 64 tiles
// and at most 8 column tiles per layer, a cluster of CTAs holds the whole row block and a cluster barrier replaces the kernel
// boundary (clusters never wait on each other).  Stage s+1 joins stage s when
//   - both hold only GEMM tasks with a bias+ReLU, mask or fp32 epilogue, plus T_SHADOW riders, and s writes pair matrices (not fp32);
//   - every GEMM of s+1 reads, as its K-major A operand, exactly the output of its own GEMM of s, with the same rows;
//   - nothing else a GEMM of the chain reads (B, ReLU-mask source) is written by a stage of the chain;
//   - every GEMM of the chain has at most kChainMaxCols 64-column tiles.
// Results do not depend on the tile shape (the K order and the three products of every element stay the same).
constexpr int kChainMaxCols = 8;
struct Chain {
    int s0, s1, cluster;
    int n_row;                                 // row clusters (row blocks of the first stage's GEMMs)
    int rider_tiles;                           // T_SHADOW tiles of the chain's stages
    int rider_clusters = 0, kind = 0;          // clusters that walk the riders; kernel variant of the launch
};

static bool same_pm(const PmRef &a, const PmRef &b) { return a.base.v == b.base.v && a.ld == b.ld && a.plane == b.plane; }

static std::vector<Chain> find_chains(const std::vector<Task> &tasks, const std::vector<Stage> &stages) {
    auto gemms = [&](int s) { std::vector<int> g; for (int k = stages[s].task_begin; k < stages[s].task_end; k++) if (tasks[k].type == T_GEMM) g.push_back(k); return g; };
    auto eligible = [&](int s) {
        bool any = false;
        for (int k = stages[s].task_begin; k < stages[s].task_end; k++) {
            const Task &t = tasks[k];
            if (t.type == T_SHADOW) continue;
            if (t.type != T_GEMM || (t.epi != EPI_F32 && t.epi != EPI_BIAS_RELU && t.epi != EPI_MASK) || cdiv(t.N, 64) > kChainMaxCols) return false;
            any = true;
        }
        return any;
    };
    auto joins = [&](int s) {      // s -> s+1
        if (!eligible(s) || !eligible(s + 1)) return false;
        const std::vector<int> prev = gemms(s), next = gemms(s + 1);
        std::vector<int> used(prev.size(), 0);
        for (int k : prev) if (tasks[k].epi == EPI_F32) return false;
        for (int h : next) {
            const Task &t = tasks[h];
            if (t.A.mn_major || t.A.r0) return false;
            int found = -1;
            for (size_t i = 0; i < prev.size(); i++)
                if (same_pm(tasks[prev[i]].Cpm, t.A.pm) && tasks[prev[i]].M == t.M && tasks[prev[i]].N == t.K) found = (int)i;
            if (found < 0 || used[found]++) return false;
        }
        return true;
    };
    auto reads_written = [&](int s0, int s1) {      // a GEMM of [s0, s1) reads as B / mask what a task of [s0, s1) writes
        std::vector<int64_t> out;
        for (int s = s0; s < s1; s++)
            for (int k = stages[s].task_begin; k < stages[s].task_end; k++)
                out.push_back(tasks[k].type == T_GEMM ? tasks[k].Cpm.base.v : tasks[k].pm[0].base.v);
        for (int s = s0; s < s1; s++)
            for (int k : gemms(s))
                for (int64_t o : out)
                    if (o == tasks[k].B.pm.base.v || (tasks[k].epi == EPI_MASK && o == tasks[k].mask.base.v)) return true;
        return false;
    };
    std::vector<Chain> out;
    for (int s = 0; s + 1 < (int)stages.size();) {
        int e = s + 1;
        while (e < (int)stages.size() && joins(e - 1) && !reads_written(s, e + 1)) e++;
        if (e - s < 2) { s++; continue; }
        Chain c{s, e, 1, 0, 0};
        for (int x = s; x < e; x++)
            for (int k = stages[x].task_begin; k < stages[x].task_end; k++) {
                if (tasks[k].type == T_GEMM) c.cluster = std::max(c.cluster, cdiv(tasks[k].N, 64));
                else c.rider_tiles += tasks[k].n_tiles;
            }
        for (int k : gemms(s)) c.n_row += cdiv(tasks[k].M, 64);
        if (c.n_row <= kMaxChainClusters) out.push_back(c);
        s = e;
    }
    return out;
}

// Stage::chain_map of every stage of a chain (tasks built with 64 x 64 tiles)
static void fill_chain_maps(const std::vector<Task> &tasks, std::vector<Stage> &stages, const Chain &c) {
    std::map<int, int> first_cluster;      // GEMM task -> cluster of its row block 0 (row blocks r -> first + r)
    int next = 0;
    for (int s = c.s0; s < c.s1; s++) {
        Stage &sg = stages[s];
        for (int i = 0; i < kMaxChainClusters; i++) sg.chain_map[i] = -1;
        sg.chain_len = s == c.s0 ? c.s1 - c.s0 : 0;
        sg.chain_clusters = c.n_row;
        for (int k = sg.task_begin; k < sg.task_end; k++) {
            const Task &t = tasks[k];
            if (t.type != T_GEMM) continue;
            int c0 = -1;
            if (s == c.s0) { c0 = next; next += t.tiles_m; }
            else
                for (int p = stages[s - 1].task_begin; p < stages[s - 1].task_end; p++)
                    if (tasks[p].type == T_GEMM && same_pm(tasks[p].Cpm, t.A.pm)) c0 = first_cluster[p];
            first_cluster[k] = c0;
            for (int rb = 0; rb < t.tiles_m; rb++) sg.chain_map[c0 + rb] = (t.tile_begin + rb * t.tiles_n) | (t.tiles_n << 16);
        }
    }
}

}  // namespace

void free_programs(sacb_handle h) {
    for (auto &kv : h->programs) {
        if (kv.second.graph) cudaGraphExecDestroy(kv.second.graph);
        for (auto g : kv.second.graph_part) if (g) cudaGraphExecDestroy(g);
        if (kv.second.step_graph) cudaGraphExecDestroy(kv.second.step_graph);
        cudaFree(kv.second.d_tasks); cudaFree(kv.second.d_stages);
    }
    h->programs.clear();
}

int check_error_flag(sacb_handle h) {
    int32_t flag = 0;
    SACB_CUDA(cudaMemcpyAsync(&flag, h->error_flag, sizeof(flag), cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    if (flag) {
        cudaMemsetAsync(h->error_flag, 0, sizeof(int32_t), h->stream);
        return fail(SACB_ERR_DEVICE, flag == 1 ? "tcgen05 pipeline watchdog: an mbarrier never completed"
                                              : "grid barrier watchdog: persistent kernel blocks were not co-resident");
    }
    return SACB_OK;
}

// one stage = one launch of the stream kernel, optional PDL
static int launch_stream_stage(sacb_handle h, ProgramInst &p, int s, bool pdl) {
    uint64_t seed = h->cfg.seed;
    Stage single = p.stages[s];
    void *args[] = {(void *)&p.prog, (void *)&single, (void *)&seed};
    cudaLaunchConfig_t cfg{};
    const int tiles = std::max(1, single.n_tiles * h->cfg.n_agents);
    cfg.gridDim = dim3(std::min(tiles, h->sm_count)); cfg.blockDim = dim3(stream::kThreads); cfg.dynamicSmemBytes = stream::kSmemBytes; cfg.stream = h->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    SACB_CUDA(cudaLaunchKernelExC(&cfg, (const void *)sac_stream_kernel, args));
    return SACB_OK;
}

// launch `li` of a staged program: one stage, or a chain of stages as thread-block clusters; optional PDL
static int launch_stage(sacb_handle h, ProgramInst &p, int li, bool pdl) {
    const StageLaunch &L = p.launches[li];
    const int s = L.s0;
    if (p.stage_stream[s]) return launch_stream_stage(h, p, s, pdl);
    const bool tc = math_is_tc(h->cfg.math_mode), chain = L.s1 - L.s0 > 1;
    const int kind = L.kind;      // index of the kernel variant
    const size_t smem = variant_has_gemm(kind) ? math_smem(h->cfg.math_mode) : 0;      // element-wise stages only use static shared memory
    uint64_t seed = h->cfg.seed;
    int s0 = L.s0, s1 = L.s1, tc_setup = tc ? p.stage_has_gemm[s] : 0, chained = chain ? 1 : 0;
    Stage single = p.stages[s];
    void *args[] = {(void *)&p.prog, (void *)&single, (void *)&s0, (void *)&s1, (void *)&tc_setup, (void *)&chained, (void *)&seed};
    cudaLaunchConfig_t cfg{};
    int ctas = chain ? L.grid : std::max(1, single.n_tiles * h->cfg.n_agents);
    // population mode: a stage of many more tiles than SMs runs as one resident CTA per SM looping over tiles (barrier /
    // TMEM setup and teardown once per SM instead of once per tile); a single agent's stage (<= ~150 tiles) keeps one CTA per tile
    static const int grid_cap = getenv("SACB_GRID_CAP") ? atoi(getenv("SACB_GRID_CAP")) : -1;     // 0 = never cap
    const int cap = grid_cap < 0 ? h->sm_count : grid_cap;
    if (!chain && cap > 0 && ctas > 2 * h->sm_count) {      // resident CTAs looping over tiles wi = blockIdx.x + i * gridDim.x
        ctas = std::min(ctas, cap * (tc ? variant_blocks_per_sm(kind) : 1));
        // a grid that is a multiple of the stage's per-agent tile count keeps every CTA on ONE tile of ONE task across the agents it
        // walks: the task record is fetched once instead of once per tile (population mode: a column-sum stage holds 2-6 tasks)
        if (single.task_end - single.task_begin > 1 && single.n_tiles <= ctas / 2) ctas = (ctas / single.n_tiles) * single.n_tiles;
    }
    cfg.gridDim = dim3(ctas); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = smem; cfg.stream = h->stream;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (pdl) {
        // programmatic dependent launch: the next stage's CTAs may become resident (on SMs this stage leaves idle) and run
        // their prologue -- barrier init, TMEM allocation, stage / task table fetch, TMA descriptor prefetch -- while this
        // stage still computes; they block in griddepcontrol.wait before touching anything a previous stage wrote
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        na++;
    }
    if (chain && L.cluster > 1) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = L.cluster; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
        na++;
    }
    cfg.attrs = attr; cfg.numAttrs = na;
    SACB_CUDA(cudaLaunchKernelExC(&cfg, update_kernel_for(h->cfg.math_mode, kind), args));
    return SACB_OK;
}

// the stages [s0, s1) as ONE cooperative launch of the build that carries every code path (persistent mode)
static int launch_range(sacb_handle h, ProgramInst &p, int s0, int s1) {
    const bool tf32 = math_is_tc(h->cfg.math_mode);
    int needs_tc = 0, max_tiles = 1;
    for (int s = s0; s < s1; s++) { needs_tc |= p.stage_has_gemm[s]; max_tiles = std::max(max_tiles, p.stages[s].n_tiles * h->cfg.n_agents); }
    const size_t smem = math_smem(h->cfg.math_mode);
    uint64_t seed = h->cfg.seed;
    int tc_setup = tf32 ? needs_tc : 0, chained = 0;
    Stage single = p.stages[s0];
    void *args[] = {(void *)&p.prog, (void *)&single, (void *)&s0, (void *)&s1, (void *)&tc_setup, (void *)&chained, (void *)&seed};
    const void *fn = update_kernel_for(h->cfg.math_mode, h->cfg.layer_norm ? kVariantEverythingLn : kVariantEverything);
    const int grid = std::min(max_tiles, h->sm_count * h->coop_blocks_per_sm);
    SACB_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kThreads), args, smem, h->stream));
    return SACB_OK;
}

static int record_step(sacb_handle h, ProgramInst &p) {
    if (h->cfg.launch_mode == SACB_LAUNCH_PERSISTENT) {
        SACB_CUDA(cudaMemsetAsync(h->barrier, 0, sizeof(unsigned int), h->stream));
        return launch_range(h, p, 0, (int)p.stages.size());
    }
    for (int li = 0; li < (int)p.launches.size(); li++) {
        int rc = launch_stage(h, p, li, h->use_pdl != 0);
        if (rc) return rc;
    }
    return SACB_OK;
}

// clusters of `cluster` CTAs of kernel variant `kind` the GPU holds at once (cached per handle); < 0: a CUDA error code
static int max_active_clusters(sacb_handle h, int kind, int cluster) {
    const auto key = std::make_pair(kind, cluster);
    const auto it = h->max_active_clusters.find(key);
    if (it != h->max_active_clusters.end()) return it->second;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(cluster); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = math_smem(h->cfg.math_mode); cfg.stream = h->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, update_kernel_for(h->cfg.math_mode, kind), &cfg) != cudaSuccess) {
        cudaGetLastError();
        return fail(SACB_ERR_DEVICE, "cudaOccupancyMaxActiveClusters failed");
    }
    h->max_active_clusters[key] = n;
    return n;
}

int get_program(sacb_handle h, const ProgramKey &key, ProgramInst **out) {
    auto it = h->programs.find(key);
    if (it != h->programs.end()) { *out = &it->second; return SACB_OK; }
    if (key.B < 1 || key.B > h->cfg.max_batch) return fail(SACB_ERR_ARG, "batch size exceeds max_batch of the handle");
    std::vector<std::pair<int, int>> shapes;
    std::vector<Chain> chains;
    bool stream_mode = false;
    {   // dry pass with the default 128 x 64 tiles: the per-stage tile counts drive the choice of tile shapes
        Builder d(h, key);
        d.dry = true;
        d.build();
        if (d.rc != SACB_OK) return d.rc;
        int widest = 0;
        for (size_t s = 0; s < d.stages.size(); s++) if (d.has_gemm[s]) widest = std::max(widest, d.stages[s].n_tiles * h->cfg.n_agents);
        // throughput form: the widest GEMM stage has more than two waves of tiles (population of agents, large batches)
        stream_mode = math_is_tc(h->cfg.math_mode) && h->cfg.launch_mode == SACB_LAUNCH_STAGED && widest > 2 * h->sm_count &&
                      !getenv("SACB_NO_STREAM") && !getenv("SACB_FUSE_SAMPLE");
        shapes = stream_mode ? d.stream_tile_shapes() : d.choose_tile_shapes(h->sm_count);
        // chained launches: latency programs of one agent (staged, tensor cores, no LayerNorm), where every cluster of the chain fits
        // on the GPU at once (its CTAs hold one SM each)
        if (math_is_tc(h->cfg.math_mode) && h->cfg.launch_mode == SACB_LAUNCH_STAGED && !stream_mode && h->cfg.n_agents == 1 && !h->cfg.layer_norm) {
            for (Chain c : find_chains(d.tasks, d.stages)) {
                uint32_t types = 0, epis = 0;
                for (int k = d.stages[c.s0].task_begin; k < d.stages[c.s1 - 1].task_end; k++) {
                    types |= tb(d.tasks[k].type);
                    if (d.tasks[k].type == T_GEMM) epis |= tb(d.tasks[k].epi);
                }
                const int kind = pick_variant(types, epis, false);
                const int fit = max_active_clusters(h, kind, c.cluster);
                if (fit < 0) return fit;
                if (!variant_can_chain(kind)) continue;
                const int riders = c.rider_tiles ? std::min(cdiv(c.rider_tiles, c.cluster), fit - c.n_row) : 0;
                if (c.n_row > fit || (c.rider_tiles && riders < 1)) continue;
                c.rider_clusters = riders; c.kind = kind;
                chains.push_back(c);
                for (int k = d.stages[c.s0].task_begin; k < d.stages[c.s1 - 1].task_end; k++)
                    if (d.tasks[k].type == T_GEMM) shapes[k] = {64, 64};
            }
        }
    }
    Builder b(h, key);
    b.shapes = shapes;
    b.stream = stream_mode;
    b.build();
    if (b.rc != SACB_OK) return b.rc;
    std::vector<int> stage_stream;
    if (stream_mode) b.split_mixed_stages(stage_stream);
    for (const Chain &c : chains) fill_chain_maps(b.tasks, b.stages, c);
    ProgramInst &p = h->programs[key];
    p.tasks = b.tasks; p.stages = b.stages; p.stage_has_gemm = b.has_gemm;
    p.stage_stream = stage_stream.empty() ? std::vector<int>(b.stages.size(), 0) : stage_stream;
    for (size_t s = 0; s < b.stages.size(); s++) {      // the smallest build of the stage kernel that covers the stage
        uint32_t types = 0, epis = 0;
        for (int k = b.stages[s].task_begin; k < b.stages[s].task_end; k++) {
            types |= tb(b.tasks[k].type);
            if (b.tasks[k].type == T_GEMM) epis |= tb(b.tasks[k].epi);
        }
        // the two-CTAs-per-SM column-sum build (4 rows in flight per thread) pays where resident CTAs walk thousands of small tiles (a
        // population); a stage of a few long tiles (one agent, large batch) keeps the one-CTA build with 8 rows in flight
        const bool many = b.stages[s].n_tiles * h->cfg.n_agents > 2 * h->sm_count;
        p.stage_kind.push_back(getenv("SACB_ONE_KERNEL") ? (h->cfg.layer_norm ? kVariantEverythingLn : kVariantEverything) : pick_variant(types, epis, many));
    }
    for (int s = 0, ci = 0; s < (int)b.stages.size();) {
        if (ci < (int)chains.size() && chains[ci].s0 == s) {
            const Chain &c = chains[ci++];
            p.launches.push_back({c.s0, c.s1, c.cluster, (c.n_row + c.rider_clusters) * c.cluster, c.kind});
            s = c.s1;
        } else {
            p.launches.push_back({s, s + 1, 1, 0, p.stage_kind[s]});
            s++;
        }
    }
    for (auto &s : p.stages) { p.n_tiles_total += s.n_tiles; p.max_stage_tiles = std::max(p.max_stage_tiles, s.n_tiles); }
    SACB_CUDA(cudaMalloc(&p.d_tasks, p.tasks.size() * sizeof(Task)));
    SACB_CUDA(cudaMalloc(&p.d_stages, p.stages.size() * sizeof(Stage)));
    SACB_CUDA(cudaMemcpyAsync(p.d_tasks, p.tasks.data(), p.tasks.size() * sizeof(Task), cudaMemcpyHostToDevice, h->stream));
    SACB_CUDA(cudaMemcpyAsync(p.d_stages, p.stages.data(), p.stages.size() * sizeof(Stage), cudaMemcpyHostToDevice, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    Program &P = p.prog;
    P.tasks = p.d_tasks; P.stages = p.d_stages; P.n_stages = (int)p.stages.size(); P.n_agents = h->cfg.n_agents;
    P.bases.arena = h->arena; P.bases.ws = h->ws; P.bases.arena_stride = h->L.arena_size; P.bases.ws_stride = h->L.ws_size;
    P.scalars = make_ref(0, h->L.scalars);
    P.barrier = h->barrier;
    if (key.with_gather == 2) {   // minibatch supplied by the caller: rows staged in upload order (sacb_update_batch)
        P.ring = h->stage_rows; P.ring_agent_stride = 0; P.slots = h->slots_identity;
    } else {
        P.ring = h->ring; P.ring_agent_stride = h->cfg.capacity * h->ring_row; P.slots = h->slots;
    }
    P.ring_row = (int32_t)h->ring_row; P.slots_stride = h->cfg.max_batch;
    P.ring_meta = h->ring_meta;
    P.error_flag = h->error_flag;
    P.trace = nullptr; P.timeline = nullptr; P.adam_table = h->adam_table;
    P.host_losses = h->cfg.n_agents == 1 ? h->pin_small : nullptr;
    p.kernels_per_step = h->cfg.launch_mode == SACB_LAUNCH_PERSISTENT ? 1 : (int)p.launches.size();

    // capture one step into a CUDA graph (stage kernels, or memset + the single cooperative launch)
    cudaGraph_t graph = nullptr;
    cudaError_t e = cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal);
    if (e == cudaSuccess) {
        int rc = record_step(h, p);
        cudaError_t e2 = cudaStreamEndCapture(h->stream, &graph);
        if (rc == SACB_OK && e2 == cudaSuccess && graph) {
            if (cudaGraphInstantiate(&p.graph, graph, 0) != cudaSuccess) p.graph = nullptr;
        }
        if (graph) cudaGraphDestroy(graph);
    }
    cudaGetLastError();   // a failed capture falls back to direct launches
    *out = &p;
    return SACB_OK;
}

ProgramKey update_key(sacb_handle h, int B, int with_gather, int export_grads, int device_eps, int use_isw) {
    ProgramKey k{B, with_gather, export_grads, device_eps, use_isw, -1};
    static const bool always = getenv("SACB_ALWAYS_SHADOW") != nullptr;      // A/B switch: re-derive every shadow every step (round-1 behaviour)
    k.resident = (h->shadows_valid && !always) ? 1 : 0;
    return k;
}
void after_update_launch(sacb_handle h, const ProgramKey &key) {
    // a full update (Adam applied) leaves every shadow current: its epilogues refreshed what they changed
    if (key.dp_phase < 0) h->shadows_valid = true;
}

int launch_program(sacb_handle h, ProgramInst &p) {
    h->kernel_launches += p.kernels_per_step;
    if (p.graph) { SACB_CUDA(cudaGraphLaunch(p.graph, h->stream)); return SACB_OK; }
    return record_step(h, p);
}

// The replay work may start anywhere behind the critic-loss stage (the TD errors exist from there on).  It is started in front
// of the actor-loss stage: the stages from there on (losses, dL/da chain, sample backward, policy backward) leave 20-140 SMs
// idle, so the sampler's kernels do not queue behind the wide critic-backward stages (step 0.2215 -> 0.2075 ms at C2).
static int compute_split(ProgramInst &p) {
    const int ns = (int)p.stages.size();
    int td_stage = -1, actor_stage = -1;
    for (int s = 0; s < ns; s++)
        for (int k = p.stages[s].task_begin; k < p.stages[s].task_end; k++) {
            if (p.tasks[k].type == T_TARGET_LOSS && td_stage < 0) td_stage = s;
            if (p.tasks[k].type == T_ACTOR_LOSS && actor_stage < 0) actor_stage = s;
        }
    if (td_stage < 0) return fail(SACB_ERR_STATE, "program has no critic-loss stage");
    int split = actor_stage > td_stage ? actor_stage : td_stage + 1;
    if (getenv("SACB_PER_SPLIT")) split = std::min(ns - 1, std::max(td_stage + 1, atoi(getenv("SACB_PER_SPLIT"))));      // experiment switch
    // the first launch from that stage on (neither the loss stages nor their neighbours are in a chain: a launch boundary)
    const int nl = (int)p.launches.size();
    p.split = nl;
    for (int li = nl - 1; li >= 0 && p.launches[li].s0 >= split; li--) p.split = li;
    return SACB_OK;
}

// sacb_per_step as one graph launch (two graph launches + two events cost ~8 us per step: 206 against 198 us with no replay work at all)
int launch_per_step_graph(sacb_handle h, ProgramInst &p, int64_t B, int64_t k) {
    static const bool off = getenv("SACB_NO_STEP_GRAPH") != nullptr;
    if (off || h->cfg.launch_mode != SACB_LAUNCH_STAGED || p.step_graph_failed) return 1;
    const int nl = (int)p.launches.size();
    const int64_t n = h->r_len[0];
    if (!p.step_graph || p.step_graph_n != n || p.step_graph_k != k) {
        if (p.step_graph) { cudaGraphExecDestroy(p.step_graph); p.step_graph = nullptr; }
        if (p.split < 0) { if (int rc = compute_split(p)) return rc; }
        if (h->per_frame_dirty) return 1;      // the first (uncaptured) sample uploads the frame counter
        // host-side bookkeeping of the launch helpers is replayed per graph launch below: undo what the capture pass does to it
        const int64_t launches0 = h->kernel_launches, frame0 = h->per_frame[0];
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); p.step_graph_failed = true; return 1; }
        int rc = SACB_OK;
        for (int li = 0; li < p.split && rc == SACB_OK; li++) rc = launch_stage(h, p, li, h->use_pdl != 0);
        if (rc == SACB_OK && (cudaEventRecord(h->ev_td, h->stream) != cudaSuccess || cudaStreamWaitEvent(h->stream2, h->ev_td, 0) != cudaSuccess)) rc = SACB_ERR_DEVICE;
        if (rc == SACB_OK) rc = per_writeback_launch(h, h->stream2, k, false);      // first kernel of the forked branch: a full dependency
        if (rc == SACB_OK) rc = per_sample_launch(h, h->stream2, nullptr, B, nullptr);
        if (rc == SACB_OK && cudaEventRecord(h->ev_sampled, h->stream2) != cudaSuccess) rc = SACB_ERR_DEVICE;
        for (int li = p.split; li < nl && rc == SACB_OK; li++) rc = launch_stage(h, p, li, h->use_pdl != 0);
        if (rc == SACB_OK && cudaStreamWaitEvent(h->stream, h->ev_sampled, 0) != cudaSuccess) rc = SACB_ERR_DEVICE;
        const cudaError_t e2 = cudaStreamEndCapture(h->stream, &graph);
        p.step_graph_launches = nl + (int)(h->kernel_launches - launches0);      // the stage kernels + what the replay helpers counted
        p.step_graph_fused = h->per_fused;
        h->kernel_launches = launches0; h->per_frame[0] = frame0;
        if (rc != SACB_OK || e2 != cudaSuccess || !graph || cudaGraphInstantiate(&p.step_graph, graph, 0) != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            p.step_graph = nullptr; p.step_graph_failed = true;
            return 1;
        }
        cudaGraphDestroy(graph);
        p.step_graph_n = n; p.step_graph_k = k;
    }
    SACB_CUDA(cudaGraphLaunch(p.step_graph, h->stream));
    h->kernel_launches += p.step_graph_launches;
    h->per_frame[0] += 1; h->sample_k = k; h->per_fused = p.step_graph_fused; h->prio_max_valid = true;
    return SACB_OK;
}

int launch_program_part(sacb_handle h, ProgramInst &p, int part) {
    if (h->cfg.launch_mode != SACB_LAUNCH_STAGED) {      // a single cooperative launch cannot be split: part 0 is the whole step
        return part == 0 ? launch_program(h, p) : SACB_OK;
    }
    const int nl = (int)p.launches.size();
    if (!p.parts_built) {
        p.parts_built = true;
        if (p.split < 0) { if (int rc = compute_split(p)) return rc; }
        for (int part_i = 0; part_i < 2; part_i++) {
            const int s0 = part_i ? p.split : 0, s1 = part_i ? nl : p.split;
            cudaGraph_t graph = nullptr;
            if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) break;
            int rc = SACB_OK;
            for (int s = s0; s < s1 && rc == SACB_OK; s++) rc = launch_stage(h, p, s, h->use_pdl != 0);
            const cudaError_t e2 = cudaStreamEndCapture(h->stream, &graph);
            if (rc == SACB_OK && e2 == cudaSuccess && graph && cudaGraphInstantiate(&p.graph_part[part_i], graph, 0) != cudaSuccess) p.graph_part[part_i] = nullptr;
            if (graph) cudaGraphDestroy(graph);
        }
        cudaGetLastError();
    }
    const int s0 = part ? p.split : 0, s1 = part ? nl : p.split;
    h->kernel_launches += s1 - s0;
    if (p.graph_part[part]) { SACB_CUDA(cudaGraphLaunch(p.graph_part[part], h->stream)); return SACB_OK; }
    for (int s = s0; s < s1; s++) { int rc = launch_stage(h, p, s, h->use_pdl != 0); if (rc) return rc; }
    return SACB_OK;
}

}  // namespace sacb

// ================================================================================================================
// instrumentation entry points that need the kernel symbol
// ================================================================================================================
using namespace sacb;

extern "C" int sacb_time_stages(sacb_handle h, int64_t B, float *us_out, int cap) {
    if (!h) return fail(SACB_ERR_ARG, "null handle");
    ProgramInst *p;
    int rc;
    if (!h->shadows_valid) {      // one step that (re)derives the shadows, then the steady-state program is profiled
        ProgramKey k0 = update_key(h, (int)B, 0, 0, 1, 0);
        if ((rc = get_program(h, k0, &p)) || (rc = launch_program(h, *p))) return rc;
        after_update_launch(h, k0);
    }
    ProgramKey key = update_key(h, (int)B, 0, 0, 1, 0);
    if (getenv("SACB_TIME_DP_PHASE")) {      // profile the backward half of a data-parallel phase instead (gradients exported, nothing applied)
        key = ProgramKey{(int)B, 0, 1, 1, 0, atoi(getenv("SACB_TIME_DP_PHASE"))};
    }
    rc = get_program(h, key, &p);
    if (rc) return rc;
    const bool trace = getenv("SACB_TRACE") != nullptr;
    unsigned long long *d_trace = nullptr;
    std::vector<unsigned long long> h_trace;
    if (trace) { SACB_CUDA(cudaMalloc(&d_trace, sizeof(unsigned long long) * kTraceSlots * 4096)); SACB_CUDA(cudaMemset(d_trace, 0, sizeof(unsigned long long) * kTraceSlots * 4096));
                 p->prog.trace = d_trace; h_trace.resize(kTraceSlots * 4096); }
    const int nl = (int)p->launches.size();      // one entry per launch (a chain of stages is one)
    const int n = std::min<int>(cap, nl);
    std::vector<cudaEvent_t> ev(nl + 1);
    for (auto &e : ev) cudaEventCreate(&e);
    std::vector<float> acc(nl, 0.f);
    const int reps = 20;
    for (int r = 0; r < reps + 3; r++) {
        cudaEventRecord(ev[0], h->stream);
        for (int li = 0; li < nl; li++) {
            // force the staged form regardless of launch_mode: this is a per-launch profile
            { int rc2 = launch_stage(h, *p, li, false); if (rc2) return rc2; }
            cudaEventRecord(ev[li + 1], h->stream);
            const StageLaunch &L = p->launches[li];
            const int s = L.s0, ks = 1;
            if (trace && r == reps + 2 && L.s1 - L.s0 > 1) {      // chain: span of the launch (per-CTA stamps cover its first tile only)
                SACB_CUDA(cudaStreamSynchronize(h->stream));
                const int g = std::min(L.grid, 4096);
                SACB_CUDA(cudaMemcpy(h_trace.data(), d_trace, sizeof(unsigned long long) * kTraceSlots * g, cudaMemcpyDeviceToHost));
                unsigned long long t0 = ~0ull, t5 = 0;
                for (int b = 0; b < g; b++) { t0 = std::min(t0, h_trace[b * kTraceSlots]); t5 = std::max(t5, h_trace[b * kTraceSlots + 5]); }
                fprintf(stderr, "[trace] stages %2d-%2d chain cluster %d grid %4d span %6.2f us\n", L.s0, L.s1 - 1, L.cluster, L.grid, (t5 - t0) * 1e-3);
                SACB_CUDA(cudaMemset(d_trace, 0, sizeof(unsigned long long) * kTraceSlots * 4096));
            } else if (trace && r == reps + 2) {
                SACB_CUDA(cudaStreamSynchronize(h->stream));
                const int grid = std::max(1, p->stages[s].n_tiles * h->cfg.n_agents);
                SACB_CUDA(cudaMemcpy(h_trace.data(), d_trace, sizeof(unsigned long long) * kTraceSlots * std::min(grid, 4096), cudaMemcpyDeviceToHost));
                double a[8] = {0}, mx_tile = 0, mx_main = 0; unsigned long long t0 = ~0ull, t0max = 0, t5 = 0;
                const int g = std::min(grid, 4096);
                for (int b = 0; b < g; b++) {
                    const unsigned long long *q = &h_trace[b * kTraceSlots];
                    t0 = std::min(t0, q[0]); t0max = std::max(t0max, q[0]); t5 = std::max(t5, q[5]);
                    a[1] += (double)(q[1] - q[0]); a[4] += (double)(q[4] - q[1]); a[5] += (double)(q[5] - q[4]);
                    mx_tile = std::max(mx_tile, (double)(q[4] - q[1]));
                    if (p->stage_has_gemm[s]) { a[2] += (double)(q[2] - q[1]); a[3] += (double)(q[3] - q[2]); mx_main = std::max(mx_main, (double)(q[2] - q[1])); }
                }
                fprintf(stderr, "[trace] stage %2d grid %4d gemm %d span %6.2f us start-skew %5.2f | per-CTA avg: setup %.2f mainloop %.2f (max %.2f) epilogue %.2f tile %.2f (max %.2f) teardown %.2f\n",
                        s, grid, p->stage_has_gemm[s], (t5 - t0) * 1e-3, (t0max - t0) * 1e-3, a[1] / g * 1e-3, a[2] / g * 1e-3, mx_main * 1e-3, a[3] / g * 1e-3,
                        a[4] / g * 1e-3, mx_tile * 1e-3, a[5] / g * 1e-3);
                {   // slowest tile of every task of the stage (which task sets the span)
                    const Stage &sg = p->stages[s];
                    fprintf(stderr, "[trace]   per-task max tile us:");
                    for (int k = 0; k < sg.task_end - sg.task_begin; k++) {
                        const Task &tk = p->tasks[sg.task_begin + k];
                        double mx = 0;
                        for (int b = tk.tile_begin * ks; b < (tk.tile_begin + tk.n_tiles) * ks && b < g; b++)
                            if (h_trace[b * kTraceSlots + 4] > h_trace[b * kTraceSlots + 1]) mx = std::max(mx, (double)(h_trace[b * kTraceSlots + 4] - h_trace[b * kTraceSlots + 1]));
                        fprintf(stderr, " [type %d epi %d %dx%dx%d n=%d] %.1f", tk.type, tk.epi, tk.M, tk.N, tk.K, tk.n_tiles, mx * 1e-3);
                    }
                    fprintf(stderr, "\n");
                }
                if (p->stage_has_gemm[s]) {      // k-block timeline of CTA 0: TMA issue / arrival times relative to the end of setup
                  for (int cta = 0; cta < 1; cta++) {
                    const unsigned long long *q = &h_trace[cta * kTraceSlots];
                    fprintf(stderr, "[trace]   cta%d issue:", cta);
                    for (int kb = 0; kb < 16 && q[16 + kb] >= q[1]; kb++) fprintf(stderr, " %.2f", (q[16 + kb] - q[1]) * 1e-3);
                    fprintf(stderr, " | arrive:");
                    for (int kb = 0; kb < 16 && q[32 + kb] >= q[1]; kb++) fprintf(stderr, " %.2f", (q[32 + kb] - q[1]) * 1e-3);
                    fprintf(stderr, " | accum %.2f staged %.2f stored %.2f epi-end %.2f\n", (q[6] - q[1]) * 1e-3, (q[7] - q[1]) * 1e-3,
                            (q[8] - q[1]) * 1e-3, (q[3] - q[1]) * 1e-3);
                  }
                    SACB_CUDA(cudaMemset(d_trace, 0, sizeof(unsigned long long) * kTraceSlots * 4096));
                }
            }
        }
        SACB_CUDA(cudaStreamSynchronize(h->stream));
        if (r >= 3)
            for (int li = 0; li < nl; li++) { float ms; cudaEventElapsedTime(&ms, ev[li], ev[li + 1]); acc[li] += ms * 1000.f / reps; }
    }
    for (int s = 0; s < n; s++) us_out[s] = acc[s];
    if (getenv("SACB_TIMELINE")) {
        // launch timeline of ONE graph replay as the update really runs (PDL, graph): per launch the earliest CTA start, the
        // earliest release from griddepcontrol.wait and the latest CTA end, from %globaltimer (stored under the launch's first stage)
        const int ns = (int)p->stages.size();
        unsigned long long *d_tl = nullptr;
        SACB_CUDA(cudaMalloc(&d_tl, sizeof(unsigned long long) * 4 * ns));
        std::vector<unsigned long long> init(4 * ns, 0ull), tl(4 * ns);
        for (int s = 0; s < ns; s++) { init[4 * s] = ~0ull; init[4 * s + 1] = ~0ull; }
        p->prog.timeline = d_tl;
        cudaGraph_t g = nullptr; cudaGraphExec_t ge = nullptr;
        SACB_CUDA(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        int rc3 = SACB_OK;
        for (int li = 0; li < nl && rc3 == SACB_OK; li++) rc3 = launch_stage(h, *p, li, h->use_pdl != 0);
        SACB_CUDA(cudaStreamEndCapture(h->stream, &g));
        p->prog.timeline = nullptr;
        if (rc3 == SACB_OK && cudaGraphInstantiate(&ge, g, 0) == cudaSuccess) {
            for (int r = 0; r < 4; r++) {
                SACB_CUDA(cudaMemcpyAsync(d_tl, init.data(), sizeof(unsigned long long) * 4 * ns, cudaMemcpyHostToDevice, h->stream));
                SACB_CUDA(cudaStreamSynchronize(h->stream));
                SACB_CUDA(cudaGraphLaunch(ge, h->stream));
                SACB_CUDA(cudaStreamSynchronize(h->stream));
            }
            SACB_CUDA(cudaMemcpy(tl.data(), d_tl, sizeof(unsigned long long) * 4 * ns, cudaMemcpyDeviceToHost));
            const unsigned long long t0 = tl[0];
            fprintf(stderr, "[timeline] stages: first-CTA-start  dependency-release  last-CTA-end | release-after-prev-end  release-to-end  (us, graph replay with PDL)\n");
            for (int li = 0; li < nl; li++) {
                const int s = p->launches[li].s0, sp = li ? p->launches[li - 1].s0 : 0;
                fprintf(stderr, "[timeline] %2d-%2d  %8.2f %8.2f %8.2f | %6.2f %6.2f\n", s, p->launches[li].s1 - 1, (tl[4 * s] - t0) * 1e-3, (tl[4 * s + 1] - t0) * 1e-3, (tl[4 * s + 2] - t0) * 1e-3,
                        li ? ((double)tl[4 * s + 1] - (double)tl[4 * sp + 2]) * 1e-3 : 0.0, (tl[4 * s + 2] - tl[4 * s + 1]) * 1e-3);
            }
            fprintf(stderr, "[timeline] update = %.2f us\n", (tl[4 * p->launches[nl - 1].s0 + 2] - t0) * 1e-3);
            cudaGraphExecDestroy(ge);
        }
        if (g) cudaGraphDestroy(g);
        cudaFree(d_tl);
    }
    if (trace && getenv("SACB_TRACE_RANGE")) {
        // warm-code experiment: stages [a, b) in ONE cooperative launch; the surviving stamps belong to stage b-1 and are
        // printed relative to its own start (slot 9, right after the grid barrier)
        int a = 1, b = 4;
        sscanf(getenv("SACB_TRACE_RANGE"), "%d,%d", &a, &b);
        int tc_setup = 1, chained = 0; uint64_t seed = h->cfg.seed; Stage single = p->stages[a];
        void *args[] = {(void *)&p->prog, (void *)&single, (void *)&a, (void *)&b, (void *)&tc_setup, (void *)&chained, (void *)&seed};
        int grid = 1;
        for (int s = a; s < b; s++) grid = std::max(grid, p->stages[s].n_tiles);
        grid = std::min(grid, h->sm_count);
        for (int r = 0; r < 3; r++) {
            SACB_CUDA(cudaMemsetAsync(h->barrier, 0, sizeof(unsigned int), h->stream));
            SACB_CUDA(cudaLaunchCooperativeKernel(update_kernel_for(h->cfg.math_mode, h->cfg.layer_norm ? kVariantEverythingLn : kVariantEverything), dim3(grid), dim3(kThreads), args, math_smem(h->cfg.math_mode), h->stream));
        }
        SACB_CUDA(cudaStreamSynchronize(h->stream));
        SACB_CUDA(cudaMemcpy(h_trace.data(), d_trace, sizeof(unsigned long long) * kTraceSlots * grid, cudaMemcpyDeviceToHost));
        for (int c = 0; c < std::min(grid, 3); c++) {
            const unsigned long long *q = &h_trace[c * kTraceSlots];
            fprintf(stderr, "[warm] stages [%d,%d) cta%d: kernel %.2f us | last stage from its start: issue", a, b, c, (q[5] - q[0]) * 1e-3);
            for (int kb = 0; kb < 16 && q[16 + kb] >= q[9]; kb++) fprintf(stderr, " %.2f", (q[16 + kb] - q[9]) * 1e-3);
            fprintf(stderr, " | arrive");
            for (int kb = 0; kb < 16 && q[32 + kb] >= q[9]; kb++) fprintf(stderr, " %.2f", (q[32 + kb] - q[9]) * 1e-3);
            fprintf(stderr, " | accum %.2f staged %.2f stored %.2f epi-end %.2f || presync %.2f taskcopy %.2f mainloop-entry %.2f | acc-lds %.2f aux-ldg %.2f\n", (q[6] - q[9]) * 1e-3, (q[7] - q[9]) * 1e-3, (q[8] - q[9]) * 1e-3, (q[3] - q[9]) * 1e-3,
                    (q[10] - q[9]) * 1e-3, (q[11] - q[9]) * 1e-3, (q[12] - q[9]) * 1e-3, (q[13] - q[9]) * 1e-3, (q[14] - q[9]) * 1e-3);
        }
    }
    if (trace) { p->prog.trace = nullptr; cudaFree(d_trace); }
    for (auto &e : ev) cudaEventDestroy(e);
    h->kernel_launches += (int64_t)(reps + 3) * nl;
    return nl;
}

namespace sacb {
struct KernelVariant { uint32_t types, epis; };
static const KernelVariant kVariants[kNumKernelVariants] = {
#define X(i, t, e) {(t), (e)},
    SACB_KERNEL_VARIANTS(X)
#undef X
};
bool variant_has_gemm(int v) { return (kVariants[v].types & tb(T_GEMM)) != 0; }
bool variant_can_chain(int v) { return variant_chains(SACB_MATH_BF16X3, kVariants[v].types, kVariants[v].epis); }
int variant_blocks_per_sm(int v) { return variant_min_blocks(kVariants[v].types, kVariants[v].epis); }
int pick_variant(uint32_t types, uint32_t epis, bool allow_light_colsum) {
    int best = 0, best_bits = 1 << 30;
    for (int v = 0; v < kNumKernelVariants; v++) {
        if ((kVariants[v].types & types) != types || (kVariants[v].epis & epis) != epis) continue;
        if (!allow_light_colsum && variant_blocks_per_sm(v) > 1 && (kVariants[v].types & (tb(T_OUT_ADAM) | tb(T_BIAS_ADAM)))) continue;
        const int bits = __builtin_popcount(kVariants[v].types) * 8 + __builtin_popcount(kVariants[v].epis);
        if (bits < best_bits) { best_bits = bits; best = v; }
    }
    return best;
}
template <int kMath>
static const void *kernel_of_variant(int v) {
    switch (v) {
#define X(i, t, e) case i: return (const void *)sac_update_kernel<kMath, (t), (e)>;
        SACB_KERNEL_VARIANTS(X)
#undef X
        default: return nullptr;
    }
}
const void *update_kernel_for(int m, int variant) {
    // the fp32 (FFMA) math mode is the checker: one build with everything (element-wise stages still launch without dynamic smem)
    if (m != SACB_MATH_BF16X3) return (const void *)sac_update_kernel<SACB_MATH_FP32, kAllTypes, kAllEpis>;
    return kernel_of_variant<SACB_MATH_BF16X3>(variant);
}
int init_kernel_attributes(sacb_handle h) {
    const int m = h->cfg.math_mode;
    if (m != SACB_MATH_FP32 && m != SACB_MATH_BF16X3) return fail(SACB_ERR_ARG, "bad math_mode");
    for (int v = 0; v < kNumKernelVariants; v++)
        if (variant_has_gemm(v))
            SACB_CUDA(cudaFuncSetAttribute(update_kernel_for(m, v), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)math_smem(m)));
    SACB_CUDA(cudaFuncSetAttribute((const void *)sac_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, stream::kSmemBytes));
    int nb = 0;
    SACB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, update_kernel_for(m, h->cfg.layer_norm ? kVariantEverythingLn : kVariantEverything), kThreads, math_smem(m)));
    h->coop_blocks_per_sm = std::max(1, std::min(nb, math_is_tc(m) ? 2 : 4));
    return SACB_OK;
}
}  // namespace sacb
