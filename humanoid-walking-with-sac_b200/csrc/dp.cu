// Large-batch data-parallel mode (BASELINE.json configs[3]): each rank runs the backward half of a phase on its
// B_local rows with gradients exported (not applied), the host all-reduces the gradient arena over NCCL
// (torch.distributed), then sacb_dp_apply runs Adam (+ Polyak) on the averaged gradients.
//   phase 0 = critics (sac_imp.py:101-113), phase 1 = actor + temperature (sac_imp.py:116-135)
#include <cstdlib>
#include <cstring>

#include "handle.h"
#include "gemm.cuh"

namespace sacb {

__global__ void dp_apply_kernel(float *w, float *m, float *v, float *wt, const float *g, int64_t n, float scale, const float *scalars, int step_slot) {
    float ss, bs;
    adam_factors_cached(scalars, step_slot, ss, bs);
    const float tau = __ldcg(scalars + SC_TAU);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        adam_element(g[i] * scale, w + i, m + i, v + i, wt ? wt + i : nullptr, nullptr, 1, ss, bs, tau);
}

__global__ void dp_finish_kernel(float *scalars, const float *g_scalars, int phase, int auto_entropy, const AdamBias *adam_table) {
    if (threadIdx.x || blockIdx.x) return;
    if (phase == 0) {
        for (int slot = SC_STEP_Q1; slot <= SC_STEP_Q2; slot++) {
            const int step = __float_as_int(scalars[slot]) + 1;
            scalars[slot] = __int_as_float(step);
            adam_factors_store(scalars, slot, step, adam_table);
        }
    } else {
        const int n_upd = __float_as_int(scalars[SC_N_UPDATES]);
        float alpha_next = scalars[SC_ALPHA0 + (n_upd & 1)];
        if (auto_entropy) {
            float ss, bs;
            adam_factors_cached(scalars, SC_STEP_ALPHA, ss, bs);
            adam_element(g_scalars[0], &scalars[SC_LOG_ALPHA], &scalars[SC_LOG_ALPHA_M], &scalars[SC_LOG_ALPHA_V], nullptr, nullptr, 1, ss, bs, 0.f);
            alpha_next = expf(scalars[SC_LOG_ALPHA]);
            const int step = __float_as_int(scalars[SC_STEP_ALPHA]) + 1;
            scalars[SC_STEP_ALPHA] = __int_as_float(step);
            adam_factors_store(scalars, SC_STEP_ALPHA, step, adam_table);
        }
        scalars[SC_ALPHA0 + ((n_upd + 1) & 1)] = alpha_next;
        const int pstep = __float_as_int(scalars[SC_STEP_POLICY]) + 1;
        scalars[SC_STEP_POLICY] = __int_as_float(pstep);
        adam_factors_store(scalars, SC_STEP_POLICY, pstep, adam_table);
        scalars[SC_N_UPDATES] = __int_as_float(n_upd + 1);
    }
}

// ---- fused exchange + optimizer step over NVLink peer memory ---------------------------------------------------------------------
// Every replica's gradient slab lives in its arena, which the peers map with CUDA IPC.  After the backward half of a phase a
// replica (1) announces "my slab of epoch e is complete" in every peer's flag array (release at system scope), (2) waits until all
// peers have announced the same, then (3) ONE kernel reads the W slabs element by element -- its own from HBM, the peers' over
// NVLink (peer loads bypass the local L2; .cg keeps them out of the non-coherent L1) --, sums them in rank order (identical on
// every replica, so the replicas stay bit-identical), and applies Adam + Polyak: the reduced gradient never touches memory.
// The next write of a slab (zero fill at the start of the same phase one step later) is ordered behind every peer's read by the
// barrier of the OTHER phase in between.
struct PeerSlabs { const float *g[8]; uint32_t *flags[8]; };

__global__ void dp_signal_kernel(PeerSlabs ps, int rank, int world, uint32_t epoch) {
    const int p = threadIdx.x;
    if (p >= world) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(ps.flags[p] + rank), "r"(epoch) : "memory");
}

// all peers have announced `epoch` (flags live in MY arena: local polls by the first `world` threads of every CTA)
__device__ __forceinline__ void dp_wait_peers(const PeerSlabs &ps, int rank, int world, uint32_t epoch, int *error_flag) {
    if (world <= 1) return;
    if (threadIdx.x < world) {
        const uint32_t *f = ps.flags[rank] + threadIdx.x;
        long long t0 = clock64();
        while (true) {
            uint32_t x;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(x) : "l"(f) : "memory");
            if ((int32_t)(x - epoch) >= 0) break;
            if (clock64() - t0 > 4000000000ll) { atomicExch(error_flag, 4); break; }      // a peer never arrived: flag it, never hang the box
        }
    }
    __syncthreads();
}

// two-shot exchange, first half (world >= 4): replica r sums slice r of the W slabs in rank order and leaves the MEAN in its own slab
// (only r itself reads slice r of its own slab in this half, so the reduction is in place).  One-shot reads (W - 1) n bytes per
// replica over NVLink, two-shot 2 (W - 1) / W n: 7x -> 1.75x the slab at 8 replicas.
__global__ void __launch_bounds__(256) dp_reduce_scatter_kernel(PeerSlabs ps, int rank, int world, uint32_t epoch, float *mine, int64_t n4, int *error_flag) {
    dp_wait_peers(ps, rank, world, epoch, error_flag);
    const int64_t per = (n4 + world - 1) / world, i0 = rank * per, i1 = min(n4, i0 + per);
    const float inv_w = 1.0f / (float)world;
    for (int64_t i = i0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < i1; i += (int64_t)gridDim.x * blockDim.x) {
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int p = 0; p < world; p++) {
            const float4 x = __ldcg(reinterpret_cast<const float4 *>(ps.g[p]) + i);
            g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
        }
        g.x *= inv_w; g.y *= inv_w; g.z *= inv_w; g.w *= inv_w;
        reinterpret_cast<float4 *>(mine)[i] = g;
    }
}

// gathered != 0: second half of the two-shot exchange -- element i is already the replica mean, held by replica i / ceil(n4 / W)
__global__ void __launch_bounds__(256) dp_reduce_apply_kernel(PeerSlabs ps, int rank, int world, uint32_t epoch, float *w, float *m, float *v, float *wt, int64_t n,
                                                              int64_t n_first, const float *scalars, int slot_first, int slot_second, int *error_flag,
                                                              int gathered) {
    dp_wait_peers(ps, rank, world, epoch, error_flag);
    const int64_t per = (n / 4 + world - 1) / world;
    float ss[2], ibs[2];
    { float a, b; adam_factors_cached(scalars, slot_first, a, b); ss[0] = a; ibs[0] = 1.0f / b; adam_factors_cached(scalars, slot_second, a, b); ss[1] = a; ibs[1] = 1.0f / b; }
    const float tau = __ldcg(scalars + SC_TAU);
    const float inv_w = 1.0f / (float)world;
    const int64_t n4 = n / 4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gathered) {
            g = __ldcg(reinterpret_cast<const float4 *>(ps.g[i / per]) + i);
        } else {
            for (int p = 0; p < world; p++) {      // rank order on every replica
                const float4 x = __ldcg(reinterpret_cast<const float4 *>(ps.g[p]) + i);
                g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
            }
            g.x *= inv_w; g.y *= inv_w; g.z *= inv_w; g.w *= inv_w;
        }
        const int h = (i * 4 >= n_first) ? 1 : 0;
        float4 W4 = reinterpret_cast<float4 *>(w)[i], M4 = reinterpret_cast<float4 *>(m)[i], V4 = reinterpret_cast<float4 *>(v)[i];
        float4 T4 = wt ? reinterpret_cast<float4 *>(wt)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        float *gw = &g.x, *pw = &W4.x, *pm = &M4.x, *pv = &V4.x, *pt = &T4.x;
#pragma unroll
        for (int j = 0; j < 4; j++) {      // adam_element's arithmetic
            const float mm = pm[j] + (1.0f - kBeta1) * (gw[j] - pm[j]);
            const float vv = pv[j] * kBeta2 + (1.0f - kBeta2) * gw[j] * gw[j];
            const float denom = sqrtf(vv) * ibs[h] + kAdamEps;
            const float ww = pw[j] - ss[h] * (mm / denom);
            pm[j] = mm; pv[j] = vv; pw[j] = ww;
            pt[j] = pt[j] * (1.0f - tau) + ww * tau;
        }
        reinterpret_cast<float4 *>(w)[i] = W4; reinterpret_cast<float4 *>(m)[i] = M4; reinterpret_cast<float4 *>(v)[i] = V4;
        if (wt) reinterpret_cast<float4 *>(wt)[i] = T4;
    }
}

// phase 1 only: mean over the replicas of the log_alpha gradient and of the three loss scalars (each replica's mean over its own
// rows), read from the peers' arenas behind the same barrier; then the temperature step and the step counters
__global__ void dp_finish_peers_kernel(float *scalars, PeerSlabs gsc, PeerSlabs lss, int world, int phase, int auto_entropy, const AdamBias *adam_table) {
    if (threadIdx.x || blockIdx.x) return;
    float g = 0.f, l[3] = {0.f, 0.f, 0.f};
    for (int p = 0; p < world; p++) {
        if (phase == 1) g += __ldcg(gsc.g[p]);
        for (int j = 0; j < 3; j++) if ((phase == 0) == (j < 2)) l[j] += __ldcg(lss.g[p] + j);
    }
    const float inv_w = 1.0f / (float)world;
    if (phase == 0) {
        scalars[SC_DP_LOSS_Q1] = l[0] * inv_w; scalars[SC_DP_LOSS_Q1 + 1] = l[1] * inv_w;      // replica means, kept apart from the local ones
        for (int slot = SC_STEP_Q1; slot <= SC_STEP_Q2; slot++) {
            const int step = __float_as_int(scalars[slot]) + 1;
            scalars[slot] = __int_as_float(step);
            adam_factors_store(scalars, slot, step, adam_table);
        }
    } else {
        scalars[SC_DP_LOSS_Q1 + 2] = l[2] * inv_w;
        g *= inv_w;
        const int n_upd = __float_as_int(scalars[SC_N_UPDATES]);
        float alpha_next = scalars[SC_ALPHA0 + (n_upd & 1)];
        if (auto_entropy) {
            float ss, bs;
            adam_factors_cached(scalars, SC_STEP_ALPHA, ss, bs);
            adam_element(g, &scalars[SC_LOG_ALPHA], &scalars[SC_LOG_ALPHA_M], &scalars[SC_LOG_ALPHA_V], nullptr, nullptr, 1, ss, bs, 0.f);
            alpha_next = expf(scalars[SC_LOG_ALPHA]);
            const int step = __float_as_int(scalars[SC_STEP_ALPHA]) + 1;
            scalars[SC_STEP_ALPHA] = __int_as_float(step);
            adam_factors_store(scalars, SC_STEP_ALPHA, step, adam_table);
        }
        scalars[SC_ALPHA0 + ((n_upd + 1) & 1)] = alpha_next;
        const int pstep = __float_as_int(scalars[SC_STEP_POLICY]) + 1;
        scalars[SC_STEP_POLICY] = __int_as_float(pstep);
        adam_factors_store(scalars, SC_STEP_POLICY, pstep, adam_table);
        scalars[SC_N_UPDATES] = __int_as_float(n_upd + 1);
    }
}

}  // namespace sacb
using namespace sacb;

extern "C" int sacb_dp_ipc_handle(sacb_handle h, void *handle_out_64_bytes) {
    if (!h || !handle_out_64_bytes) return fail(SACB_ERR_ARG, "bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
    cudaIpcMemHandle_t hd;
    SACB_CUDA(cudaIpcGetMemHandle(&hd, h->arena));
    memcpy(handle_out_64_bytes, &hd, 64);
    return SACB_OK;
}

extern "C" int sacb_dp_connect(sacb_handle h, int rank, int world, const void *handles) {
    if (!h || rank < 0 || world < 1 || world > 8 || rank >= world || (!handles && world > 1)) return fail(SACB_ERR_ARG, "data-parallel peer exchange serves 1..8 replicas on one node");
    if (h->cfg.n_agents != 1) return fail(SACB_ERR_ARG, "data-parallel mode drives a single agent");
    if (h->cfg.layer_norm) return fail(SACB_ERR_ARG, "data-parallel mode does not serve the LayerNorm variant (its gradient exchange is not validated)");
    SACB_CUDA(cudaSetDevice(h->cfg.device));
    for (int p = 0; p < world; p++) {
        if (p == rank) { h->dp_peer_arena[p] = h->arena; continue; }
        cudaIpcMemHandle_t hd;
        memcpy(&hd, (const char *)handles + 64 * p, 64);
        void *ptr = nullptr;
        SACB_CUDA(cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess));
        h->dp_peer_arena[p] = (float *)ptr;
    }
    h->dp_rank = rank; h->dp_world = world; h->dp_epoch = 0;
    SACB_CUDA(cudaMemsetAsync(h->arena + h->L.dp_flags, 0, 32 * sizeof(float), h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

extern "C" int sacb_dp_exchange_apply(sacb_handle h, int phase) {
    if (!h || phase < 0 || phase > 1) return fail(SACB_ERR_ARG, "bad argument");
    const Layout &L = h->L;
    float *ar = h->arena, *sc = ar + L.scalars;
    const int W = h->dp_world, r = h->dp_rank;
    if (!h->dp_peer_arena[r]) h->dp_peer_arena[r] = h->arena;
    const int64_t goff = phase == 0 ? L.grad[1] : L.grad[0];
    PeerSlabs ps, gsc, lss;
    for (int p = 0; p < 8; p++) {
        float *base = p < W ? h->dp_peer_arena[p] : nullptr;
        ps.g[p] = base ? base + goff : nullptr; ps.flags[p] = base ? reinterpret_cast<uint32_t *>(base + L.dp_flags) : nullptr;
        gsc.g[p] = base ? base + L.grad_scalars : nullptr; gsc.flags[p] = nullptr;
        lss.g[p] = base ? base + L.scalars + SC_LOSS_Q1 : nullptr; lss.flags[p] = nullptr;
    }
    uint32_t epoch = ++h->dp_epoch;
    if (W > 1) { dp_signal_kernel<<<1, 32, 0, h->stream>>>(ps, r, W, epoch); h->kernel_launches++; }
    h->shadows_valid = false;      // fp32 weights only: the next program re-derives the shadows
    const int grid = 2 * h->sm_count;
    const int64_t n = phase == 0 ? 2 * L.q.size : L.pol.size;
    static const int two_shot_min = getenv("SACB_DP_TWO_SHOT_MIN") ? atoi(getenv("SACB_DP_TWO_SHOT_MIN")) : 4;
    const int gathered = W >= two_shot_min ? 1 : 0;
    if (gathered) {      // reduce-scatter in place, second barrier, then the gather rides in the apply kernel
        dp_reduce_scatter_kernel<<<h->sm_count, 256, 0, h->stream>>>(ps, r, W, epoch, ar + goff, n / 4, h->error_flag);
        epoch = ++h->dp_epoch;
        dp_signal_kernel<<<1, 32, 0, h->stream>>>(ps, r, W, epoch);
        h->kernel_launches += 2;
    }
    if (phase == 0)
        dp_reduce_apply_kernel<<<grid, 256, 0, h->stream>>>(ps, r, W, epoch, ar + L.param[1], ar + L.adam_m[1], ar + L.adam_v[1], ar + L.param[3], n, L.q.size, sc,
                                                            SC_STEP_Q1, SC_STEP_Q2, h->error_flag, gathered);
    else
        dp_reduce_apply_kernel<<<grid, 256, 0, h->stream>>>(ps, r, W, epoch, ar + L.param[0], ar + L.adam_m[0], ar + L.adam_v[0], nullptr, n, L.pol.size, sc,
                                                            SC_STEP_POLICY, SC_STEP_POLICY, h->error_flag, gathered);
    dp_finish_peers_kernel<<<1, 32, 0, h->stream>>>(sc, gsc, lss, W, phase, h->cfg.auto_entropy, h->adam_table);
    h->kernel_launches += 2;
    SACB_CUDA(cudaGetLastError());
    return SACB_OK;
}

/* losses of the last data-parallel step averaged over the replicas (the local means stay in sacb_get_losses) */
extern "C" int sacb_dp_get_losses(sacb_handle h, float *losses_out) {
    if (!h || !losses_out) return fail(SACB_ERR_ARG, "bad argument");
    SACB_CUDA(cudaMemcpyAsync(losses_out, h->arena + h->L.scalars + SC_DP_LOSS_Q1, 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return check_error_flag(h);
}

// gradients of a phase are contiguous in the arena: phase 0 = grad[q1] | grad[q2], phase 1 = grad[policy] (+ log_alpha grad kept
// in the scalar-gradient block right after grad[q2]; the host reduces it as a second tiny buffer)
extern "C" int sacb_dp_grad_buffer(sacb_handle h, int phase, void **dev_ptr, int64_t *n_floats) {
    if (!h || !dev_ptr || !n_floats || phase < 0 || phase > 2) return fail(SACB_ERR_ARG, "bad argument");
    if (phase == 0) { *dev_ptr = h->arena + h->L.grad[1]; *n_floats = 2 * h->L.q.size; }
    else if (phase == 1) { *dev_ptr = h->arena + h->L.grad[0]; *n_floats = h->L.pol.size; }
    else { *dev_ptr = h->arena + h->L.grad_scalars; *n_floats = 32; }
    return SACB_OK;
}

namespace sacb { int replay_stage_slots(sacb_handle h, const int64_t *idx, int64_t B); }

extern "C" int sacb_dp_backward(sacb_handle h, int phase, int64_t B_local, const int64_t *idx, const float *eps_next, const float *eps_cur) {
    if (h && h->cfg.layer_norm) return fail(SACB_ERR_ARG, "data-parallel mode does not serve the LayerNorm variant (its gradient exchange is not validated)");
    if (!h || phase < 0 || phase > 1 || h->cfg.n_agents != 1) return fail(SACB_ERR_ARG, "bad argument");
    if (B_local < 1 || B_local > h->L.maxB) return fail(SACB_ERR_ARG, "batch size out of range");
    if ((eps_next == nullptr) != (eps_cur == nullptr)) return fail(SACB_ERR_ARG, "pass both eps arrays or neither");
    int rc;
    // every rank averages over its own B_local rows; with equal B_local the all-reduced mean of the rank means is the global mean
    if (phase == 0) {
        if (idx && (rc = replay_stage_slots(h, idx, B_local))) return rc;
        if (eps_next) {
            const int64_t n = B_local * h->cfg.act_dim;
            SACB_CUDA(cudaMemcpyAsync(h->ws + h->L.eps, eps_next, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
            SACB_CUDA(cudaMemcpyAsync(h->ws + h->L.eps + n, eps_cur, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
            h->dp_device_eps = 0;
        } else {
            h->dp_device_eps = 1;
        }
    }
    {   // large batches accumulate their gradients over K / row chunks with atomics: the phase's slab starts at zero
        const Layout &L = h->L;
        if (phase == 0) SACB_CUDA(cudaMemsetAsync(h->arena + L.grad[1], 0, sizeof(float) * 2 * L.q.size, h->stream));
        else SACB_CUDA(cudaMemsetAsync(h->arena + L.grad[0], 0, sizeof(float) * L.pol.size, h->stream));
    }
    return run_update(h, ProgramKey{(int)B_local, phase == 0 ? 1 : 0, 1, h->dp_device_eps, 0, phase});
}

extern "C" int sacb_dp_apply(sacb_handle h, int phase) {
    if (!h || phase < 0 || phase > 1) return fail(SACB_ERR_ARG, "bad argument");
    const Layout &L = h->L;
    float *ar = h->arena;
    float *sc = ar + L.scalars;
    auto run = [&](int net, int64_t size) {
        dp_apply_kernel<<<296, 256, 0, h->stream>>>(ar + L.param[net], ar + L.adam_m[net], ar + L.adam_v[net], net ? ar + L.param[net + 2] : nullptr, ar + L.grad[net], size,
                                                    1.0f, sc, net == 0 ? SC_STEP_POLICY : (net == 1 ? SC_STEP_Q1 : SC_STEP_Q2));
        h->kernel_launches++;
    };
    h->shadows_valid = false;      // the element-wise apply writes fp32 weights only: the next program re-derives the shadows
    if (phase == 0) { run(1, L.q.size); run(2, L.q.size); } else run(0, L.pol.size);
    dp_finish_kernel<<<1, 32, 0, h->stream>>>(sc, ar + L.grad_scalars, phase, h->cfg.auto_entropy, h->adam_table);
    h->kernel_launches++;
    SACB_CUDA(cudaGetLastError());
    return SACB_OK;
}
