// Row-wise network evaluation (select_action, QNetwork / GaussianPolicy callables) and the tensor-core self test.
#include <cstdlib>
#include <cstring>
#include <vector>
#include <algorithm>

#include "handle.h"
#include "tasks.cuh"
#include "stream.cuh"

namespace sacb {

struct MlpArgs {
    const float *w[4], *b[4];
    const float *g[4], *be[4];      // LayerNorm weight / bias of hidden layer l (opt-in variant, else null)
    const float *w_out, *b_out;
    int n_hidden, in_dim, hidden, out_dim;
};

// sum of v over the CTA (all threads get it); `red` = 32 floats of shared memory
__device__ __forceinline__ float block_sum(float v, float *red) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = 0.f;
    for (int w = 0; w < nw; w++) t += red[w];
    return t;
}

// one CTA per input row: y = W_out . relu(... relu(W_0 x + b_0) ...) + b_out ; warp-per-output-row dot products,
// activations in shared memory (2 x hidden floats + in_dim).  B = 1 is the select_action latency path (sac_imp.py:54-72).
__global__ void __launch_bounds__(512) mlp_rows_kernel(MlpArgs a, const float *x, int ldx, const float *x2, int n2, float *out, int ldo) {
    extern __shared__ float sm[];
    float *cur = sm, *nxt = sm + max(a.in_dim, a.hidden);
    const int row = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int n1 = a.in_dim - n2;
    for (int j = threadIdx.x; j < a.in_dim; j += blockDim.x) cur[j] = j < n1 ? x[(int64_t)row * ldx + j] : x2[(int64_t)row * n2 + (j - n1)];
    __syncthreads();
    int in = a.in_dim;
    for (int l = 0; l < a.n_hidden; l++) {
        for (int o = warp; o < a.hidden; o += nw) {
            const float *wr = a.w[l] + (int64_t)o * in;
            float s = 0.f;
            for (int j = lane; j < in; j += 32) s = fmaf(__ldg(wr + j), cur[j], s);
            s = warp_sum(s);
            if (lane == 0) nxt[o] = a.g[l] ? s + __ldg(a.b[l] + o) : fmaxf(s + __ldg(a.b[l] + o), 0.f);
        }
        __syncthreads();
        if (a.g[l]) {      // LayerNorm (biased variance, eps 1e-5) + affine + ReLU over the row
            __shared__ float red[32];
            float ps = 0.f;
            for (int o = threadIdx.x; o < a.hidden; o += blockDim.x) ps += nxt[o];
            const float mean = block_sum(ps, red) / (float)a.hidden;
            float pq = 0.f;
            for (int o = threadIdx.x; o < a.hidden; o += blockDim.x) { const float d = nxt[o] - mean; pq += d * d; }
            const float rstd = 1.0f / sqrtf(block_sum(pq, red) / (float)a.hidden + 1e-5f);
            for (int o = threadIdx.x; o < a.hidden; o += blockDim.x)
                nxt[o] = fmaxf((nxt[o] - mean) * rstd * __ldg(a.g[l] + o) + __ldg(a.be[l] + o), 0.f);
            __syncthreads();
        }
        float *t = cur; cur = nxt; nxt = t;
        in = a.hidden;
    }
    for (int o = warp; o < a.out_dim; o += nw) {
        const float *wr = a.w_out + (int64_t)o * in;
        float s = 0.f;
        for (int j = lane; j < in; j += 32) s = fmaf(__ldg(wr + j), cur[j], s);
        s = warp_sum(s);
        if (lane == 0) out[(int64_t)row * ldo + o] = s + __ldg(a.b_out + o);
    }
}

// head_raw [n, 2A] -> action [n, A]: evaluate => tanh(mean)*scale+bias (sac_imp.py:61-64), else policy.sample (:70)
__global__ void action_kernel(const float *head, const float *eps, int n, int A, int evaluate, float scale, float bias, float *act,
                              uint64_t seed, uint32_t counter) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * A) return;
    const int r = i / A, c = i % A;
    const float mean = head[(int64_t)r * 2 * A + c], ls = head[(int64_t)r * 2 * A + A + c];
    if (evaluate) { act[i] = tanhf(mean) * scale + bias; return; }
    const float e = eps ? eps[i] : philox_normal(seed, 0x5e1ec7u, counter, (uint32_t)r, (uint32_t)c);
    act[i] = sample_elem(mean, ls, e, scale, bias).action;
}

static MlpArgs mlp_args(sacb_handle h, int agent, int net) {
    const NetLayout &nl = net == SACB_NET_POLICY ? h->L.pol : h->L.q;
    const float *base = h->arena + (int64_t)agent * h->L.arena_size + h->L.param[net];
    MlpArgs a;
    memset(&a, 0, sizeof(a));
    for (int l = 0; l < nl.n_hidden; l++) {
        a.w[l] = base + nl.w[l]; a.b[l] = base + nl.b[l];
        if (nl.layer_norm) { a.g[l] = base + nl.g[l]; a.be[l] = base + nl.be[l]; }
    }
    a.w_out = base + nl.w_out; a.b_out = base + nl.b_out;
    a.n_hidden = nl.n_hidden; a.in_dim = nl.in_dim; a.hidden = nl.hidden; a.out_dim = nl.out_dim;
    return a;
}

static size_t mlp_smem(const MlpArgs &a) { return sizeof(float) * 2 * std::max(a.in_dim, a.hidden); }

}  // namespace sacb
using namespace sacb;

namespace sacb {
// ---- select_action: one launch per layer, the output rows of a layer spread over many CTAs -------------------------------------
// A single CTA reading the whole policy (2.9 MB fp32 for 3x512 on 348 inputs) is bound by one SM's L2 ingest (~30 us); 16 output
// rows per CTA put every layer on 32 SMs, and programmatic dependent launch hides the launch latency of the 5-kernel chain.
struct LayerArgs { const float *w, *b; int in, out, relu; int64_t agent_stride; };

__global__ void __launch_bounds__(512) mlp_layer_kernel(LayerArgs a, const float *x, int ldx, float *y, int ldy, int rows_per_agent) {
    extern __shared__ float sx[];
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int row = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t ao = (int64_t)(row / rows_per_agent) * a.agent_stride;
    for (int j = threadIdx.x; j < a.in; j += blockDim.x) sx[j] = __ldcg(x + (int64_t)row * ldx + j);
    __syncthreads();
    const int o = blockIdx.x * 16 + warp;
    if (o >= a.out) return;
    const float *wr = a.w + ao + (int64_t)o * a.in;
    float s = 0.f;
    if (a.in % 4 == 0 && (reinterpret_cast<uintptr_t>(wr) & 15) == 0) {
        for (int j = lane * 4; j < a.in; j += 128) {
            const float4 w4 = __ldcg(reinterpret_cast<const float4 *>(wr + j));
            s = fmaf(w4.x, sx[j], s); s = fmaf(w4.y, sx[j + 1], s); s = fmaf(w4.z, sx[j + 2], s); s = fmaf(w4.w, sx[j + 3], s);
        }
    } else {
        for (int j = lane; j < a.in; j += 32) s = fmaf(__ldcg(wr + j), sx[j], s);
    }
    s = warp_sum(s);
    if (lane == 0) {
        s += __ldcg(a.b + ao + o);
        y[(int64_t)row * ldy + o] = a.relu ? fmaxf(s, 0.f) : s;
    }
}

// LayerNorm variant: y[row, :] <- relu(LN(y[row, :]) * gamma + beta) in place, one CTA per row, behind the layer kernel in the PDL chain
__global__ void __launch_bounds__(256) ln_relu_rows_kernel(float *y, int ldy, int H, const float *g, const float *be, int64_t agent_stride, int rows_per_agent) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    __shared__ float red[32];
    const int row = blockIdx.x;
    const int64_t ao = (int64_t)(row / rows_per_agent) * agent_stride;
    float *yr = y + (int64_t)row * ldy;
    float ps = 0.f;
    for (int o = threadIdx.x; o < H; o += blockDim.x) ps += __ldcg(yr + o);
    const float mean = block_sum(ps, red) / (float)H;
    float pq = 0.f;
    for (int o = threadIdx.x; o < H; o += blockDim.x) { const float d = __ldcg(yr + o) - mean; pq += d * d; }
    const float rstd = 1.0f / sqrtf(block_sum(pq, red) / (float)H + 1e-5f);
    for (int o = threadIdx.x; o < H; o += blockDim.x) yr[o] = fmaxf((__ldcg(yr + o) - mean) * rstd * __ldcg(g + ao + o) + __ldcg(be + ao + o), 0.f);
}

__global__ void action_pdl_kernel(const float *head, const float *eps, int n, int A, int evaluate, float scale, float bias, float *act, uint64_t seed, uint32_t counter) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * A) return;
    const int r = i / A, c = i % A;
    const float mean = __ldcg(head + (int64_t)r * 2 * A + c), ls = __ldcg(head + (int64_t)r * 2 * A + A + c);
    if (evaluate) { act[i] = tanhf(mean) * scale + bias; return; }
    const float e = eps ? eps[i] : philox_normal(seed, 0x5e1ec7u, counter, (uint32_t)r, (uint32_t)c);
    act[i] = sample_elem(mean, ls, e, scale, bias).action;
}

template <typename... KArgs, typename... Args>
static cudaError_t launch_chain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// policy forward + action for `rows` observations (rows_per_agent consecutive rows belong to one agent, first agent = agent0);
// obs / eps / action travel through pinned memory, one synchronisation
static int select_action_rows(sacb_handle h, int agent0, int rows, int rows_per_agent, const float *obs, int evaluate, const float *eps, float *action_out) {
    const int O = h->cfg.obs_dim, A = h->cfg.act_dim, H = h->cfg.hidden_dim, nh = h->cfg.n_hidden;
    const int64_t per_row = align_up(O, 4) + 2 * (int64_t)H + align_up(2 * A, 4) + 2 * align_up(A, 4);
    if (h->act_rows < rows) {
        cudaFree(h->act_ws); if (h->pin_act) cudaFreeHost(h->pin_act);
        h->act_ws = nullptr; h->pin_act = nullptr; h->act_rows = 0;
        if (cudaMalloc(&h->act_ws, sizeof(float) * per_row * rows) != cudaSuccess || cudaMallocHost(&h->pin_act, sizeof(float) * (O + 2 * A) * rows) != cudaSuccess)
            return fail(SACB_ERR_NOMEM, "select_action scratch allocation failed");
        h->act_rows = rows;
    }
    float *d_obs = h->act_ws, *d_h0 = d_obs + (int64_t)align_up(O, 4) * rows, *d_h1 = d_h0 + (int64_t)H * rows;
    float *d_head = d_h1 + (int64_t)H * rows, *d_eps = d_head + (int64_t)align_up(2 * A, 4) * rows, *d_act = d_eps + (int64_t)align_up(A, 4) * rows;
    float *p_obs = h->pin_act, *p_eps = p_obs + (int64_t)O * rows, *p_act = p_eps + (int64_t)A * rows;
    const bool use_eps = eps && !evaluate;
    memcpy(p_obs, obs, sizeof(float) * O * rows);      // the previous call synchronised: the pinned block is free
    SACB_CUDA(cudaMemcpyAsync(d_obs, p_obs, sizeof(float) * O * rows, cudaMemcpyHostToDevice, h->stream));
    if (use_eps) {
        memcpy(p_eps, eps, sizeof(float) * A * rows);
        SACB_CUDA(cudaMemcpyAsync(d_eps, p_eps, sizeof(float) * A * rows, cudaMemcpyHostToDevice, h->stream));
    }
    const NetLayout &nl = h->L.pol;
    const float *base = h->arena + (int64_t)agent0 * h->L.arena_size + h->L.param[SACB_NET_POLICY];
    const float *x = d_obs; int ldx = O;
    float *bufs[2] = {d_h0, d_h1};
    for (int l = 0; l <= nh; l++) {
        LayerArgs a;
        a.w = base + (l < nh ? nl.w[l] : nl.w_out); a.b = base + (l < nh ? nl.b[l] : nl.b_out);
        a.in = l == 0 ? O : H; a.out = l < nh ? H : 2 * A; a.relu = l < nh && !nl.layer_norm; a.agent_stride = h->L.arena_size;
        float *y = l < nh ? bufs[l & 1] : d_head;
        const int ldy = l < nh ? H : 2 * A;
        SACB_CUDA(launch_chain(mlp_layer_kernel, dim3((a.out + 15) / 16, rows), dim3(512), sizeof(float) * a.in, h->stream, a, x, ldx, y, ldy, rows_per_agent));
        if (l < nh && nl.layer_norm) {
            SACB_CUDA(launch_chain(ln_relu_rows_kernel, dim3(rows), dim3(256), 0, h->stream, y, ldy, H, base + nl.g[l], base + nl.be[l], (int64_t)h->L.arena_size, rows_per_agent));
            h->kernel_launches++;
        }
        x = y; ldx = ldy;
    }
    SACB_CUDA(launch_chain(action_pdl_kernel, dim3((rows * A + 127) / 128), dim3(128), 0, h->stream, (const float *)d_head, (const float *)(use_eps ? d_eps : nullptr),
                           rows, A, evaluate, h->cfg.action_scale, h->cfg.action_bias, d_act, h->cfg.seed, h->act_counter++));
    h->kernel_launches += nh + 2;
    SACB_CUDA(cudaMemcpyAsync(p_act, d_act, sizeof(float) * A * rows, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    memcpy(action_out, p_act, sizeof(float) * A * rows);
    return SACB_OK;
}
}  // namespace sacb

// the first version (one CTA walks the whole policy, pageable copies), kept behind SACB_ACT_SINGLE_CTA=1 for A/B timing
static int select_action_single_cta(sacb_handle h, int agent, const float *obs, int evaluate, const float *eps, float *action_out) {
    const int O = h->cfg.obs_dim, A = h->cfg.act_dim;
    float *d_obs = h->stage_rows, *d_head = d_obs + align_up(O, 4), *d_eps = d_head + align_up(2 * A, 4), *d_act = d_eps + align_up(A, 4);
    SACB_CUDA(cudaMemcpyAsync(d_obs, obs, sizeof(float) * O, cudaMemcpyHostToDevice, h->stream));
    if (eps && !evaluate) SACB_CUDA(cudaMemcpyAsync(d_eps, eps, sizeof(float) * A, cudaMemcpyHostToDevice, h->stream));
    MlpArgs a = mlp_args(h, agent, SACB_NET_POLICY);
    mlp_rows_kernel<<<1, 512, mlp_smem(a), h->stream>>>(a, d_obs, O, nullptr, 0, d_head, 2 * A);
    action_kernel<<<1, std::max(32, (A + 31) / 32 * 32), 0, h->stream>>>(d_head, (eps && !evaluate) ? d_eps : nullptr, 1, A, evaluate, h->cfg.action_scale,
                                                                        h->cfg.action_bias, d_act, h->cfg.seed, h->act_counter++);
    h->kernel_launches += 2;
    SACB_CUDA(cudaGetLastError());
    SACB_CUDA(cudaMemcpyAsync(action_out, d_act, sizeof(float) * A, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

extern "C" int sacb_select_action(sacb_handle h, int agent, const float *obs, int evaluate, const float *eps, float *action_out) {
    if (!h || !obs || !action_out || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    static const bool single = getenv("SACB_ACT_SINGLE_CTA") != nullptr;
    if (single) return select_action_single_cta(h, agent, obs, evaluate, eps, action_out);
    return select_action_rows(h, agent, 1, 1, obs, evaluate, eps, action_out);
}

extern "C" int sacb_select_action_batch(sacb_handle h, const float *obs, int evaluate, const float *eps, float *action_out) {
    if (!h || !obs || !action_out) return fail(SACB_ERR_ARG, "bad argument");
    return select_action_rows(h, 0, h->cfg.n_agents, 1, obs, evaluate, eps, action_out);
}

extern "C" int sacb_q_forward(sacb_handle h, int agent, int net, const float *s, const float *a, int64_t n, float *q_out) {
    if (!h || !s || !a || !q_out || net < SACB_NET_Q1 || net > SACB_NET_Q2_TARGET || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    const int O = h->cfg.obs_dim, A = h->cfg.act_dim;
    float *d_s, *d_a, *d_q;
    SACB_CUDA(cudaMalloc(&d_s, sizeof(float) * n * O)); SACB_CUDA(cudaMalloc(&d_a, sizeof(float) * n * A)); SACB_CUDA(cudaMalloc(&d_q, sizeof(float) * n));
    SACB_CUDA(cudaMemcpyAsync(d_s, s, sizeof(float) * n * O, cudaMemcpyHostToDevice, h->stream));
    SACB_CUDA(cudaMemcpyAsync(d_a, a, sizeof(float) * n * A, cudaMemcpyHostToDevice, h->stream));
    MlpArgs m = mlp_args(h, agent, net);
    mlp_rows_kernel<<<(int)n, 512, mlp_smem(m), h->stream>>>(m, d_s, O, d_a, A, d_q, 1);
    h->kernel_launches++;
    SACB_CUDA(cudaMemcpyAsync(q_out, d_q, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(d_s); cudaFree(d_a); cudaFree(d_q);
    return SACB_OK;
}

extern "C" int sacb_policy_forward(sacb_handle h, int agent, const float *s, int64_t n, float *mean_out, float *log_std_out) {
    if (!h || !s || !mean_out || !log_std_out || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    const int O = h->cfg.obs_dim, A = h->cfg.act_dim;
    float *d_s, *d_h;
    SACB_CUDA(cudaMalloc(&d_s, sizeof(float) * n * O)); SACB_CUDA(cudaMalloc(&d_h, sizeof(float) * n * 2 * A));
    SACB_CUDA(cudaMemcpyAsync(d_s, s, sizeof(float) * n * O, cudaMemcpyHostToDevice, h->stream));
    MlpArgs m = mlp_args(h, agent, SACB_NET_POLICY);
    mlp_rows_kernel<<<(int)n, 512, mlp_smem(m), h->stream>>>(m, d_s, O, nullptr, 0, d_h, 2 * A);
    h->kernel_launches++;
    std::vector<float> head((size_t)n * 2 * A);
    SACB_CUDA(cudaMemcpyAsync(head.data(), d_h, sizeof(float) * n * 2 * A, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    for (int64_t r = 0; r < n; r++)
        for (int c = 0; c < A; c++) {
            mean_out[r * A + c] = head[r * 2 * A + c];
            log_std_out[r * A + c] = std::min(std::max(head[r * 2 * A + A + c], kLogStdMin), kLogStdMax);   // torch.clamp(log_std, -20, 2)
        }
    cudaFree(d_s); cudaFree(d_h);
    return SACB_OK;
}

namespace sacb {
// head_raw [n, 2A] (+ eps [n, A], or Philox draws) -> action [n, A], log_prob [n]: one warp per row, the arithmetic of the update's
// T_SAMPLE task (sample_elem), log-prob summed over the action components in lane order + warp tree (networks_model1.py:78-99)
__global__ void policy_sample_kernel(const float *head, const float *eps, int n, int A, float scale, float bias, float *act, float *logp,
                                     uint64_t seed, uint32_t counter) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= n) return;
    float lp = 0.f;
    for (int c = lane; c < A; c += 32) {
        const float mean = head[(int64_t)row * 2 * A + c], ls = head[(int64_t)row * 2 * A + A + c];
        const float e = eps ? eps[(int64_t)row * A + c] : philox_normal(seed, 0x5a3b1eu, counter, (uint32_t)row, (uint32_t)c);
        const SampleElem s = sample_elem(mean, ls, e, scale, bias);
        act[(int64_t)row * A + c] = s.action;
        lp += s.logp;
    }
    lp = warp_sum(lp);
    if (lane == 0) logp[row] = lp;
}
}  // namespace sacb

extern "C" int sacb_policy_sample(sacb_handle h, int agent, const float *s, int64_t n, const float *eps, float *action_out, float *log_prob_out) {
    if (!h || !s || !action_out || !log_prob_out || n < 1 || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    const int O = h->cfg.obs_dim, A = h->cfg.act_dim;
    float *d_s, *d_h, *d_e = nullptr, *d_a, *d_l;
    SACB_CUDA(cudaMalloc(&d_s, sizeof(float) * n * O)); SACB_CUDA(cudaMalloc(&d_h, sizeof(float) * n * 2 * A));
    SACB_CUDA(cudaMalloc(&d_a, sizeof(float) * n * A)); SACB_CUDA(cudaMalloc(&d_l, sizeof(float) * n));
    SACB_CUDA(cudaMemcpyAsync(d_s, s, sizeof(float) * n * O, cudaMemcpyHostToDevice, h->stream));
    if (eps) {
        SACB_CUDA(cudaMalloc(&d_e, sizeof(float) * n * A));
        SACB_CUDA(cudaMemcpyAsync(d_e, eps, sizeof(float) * n * A, cudaMemcpyHostToDevice, h->stream));
    }
    MlpArgs m = mlp_args(h, agent, SACB_NET_POLICY);
    mlp_rows_kernel<<<(int)n, 512, mlp_smem(m), h->stream>>>(m, d_s, O, nullptr, 0, d_h, 2 * A);
    policy_sample_kernel<<<(int)((n + 7) / 8), 256, 0, h->stream>>>(d_h, d_e, (int)n, A, h->cfg.action_scale, h->cfg.action_bias, d_a, d_l, h->cfg.seed, h->act_counter++);
    h->kernel_launches += 2;
    SACB_CUDA(cudaGetLastError());
    SACB_CUDA(cudaMemcpyAsync(action_out, d_a, sizeof(float) * n * A, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaMemcpyAsync(log_prob_out, d_l, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(d_s); cudaFree(d_h); cudaFree(d_e); cudaFree(d_a); cudaFree(d_l);
    return SACB_OK;
}

// ---- data-parallel mode: implemented in dp.cu ---------------------------------------------------------------------

// ---- self test: TMA + tcgen05 tile vs FFMA tile vs host float64, all on the same bf16-pair operands ------------------
namespace sacb {
template <int kMath>
__global__ void __launch_bounds__(kThreads, 1) gemm_selftest_kernel(const Task *tp, AgentBases bases, int *error_flag) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ uint64_t s_bars[2 * kTStages + 1];
    __shared__ uint32_t s_tmem;
    const Task &t = *tp;
    tc::TcState st;
    st.g = 0; st.accum_uses = 0; st.tmem_base = 0; st.full_bar = s_bars; st.empty_bar = s_bars + kTStages; st.accum_bar = s_bars + 2 * kTStages; st.trace = nullptr;
    constexpr bool kTc = kMath != SACB_MATH_FP32;
    st.tiles = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    if (kTc) {
        if (threadIdx.x == 0) { for (int i = 0; i <= 2 * kTStages; i++) tc::mbar_init(&s_bars[i], 1); tc::fence_barrier_init(); }
        if (threadIdx.x < 32) tc::tmem_alloc(&s_tmem, kTN);
        tc::tc_fence_before(); __syncthreads(); tc::tc_fence_after();
        st.tmem_base = s_tmem;
    }
    for (int tile = blockIdx.x; tile < t.n_tiles; tile += gridDim.x) {
        if (kTc) gemm_tile_tc(t, tp, tile, bases, 0, nullptr, st, error_flag, false, 0ull);
        else gemm_tile_ffma(t, tile, bases, 0, nullptr, reinterpret_cast<float *>(smem_raw));
    }
    if (kTc) { tc::tc_fence_before(); __syncthreads(); if (threadIdx.x < 32) tc::tmem_dealloc(st.tmem_base, kTN); }
}

static uint16_t host_bf16_rn(float x) {
    uint32_t u; memcpy(&u, &x, 4);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
static float host_bf16_to_float(uint16_t b) { uint32_t u = (uint32_t)b << 16; float f; memcpy(&f, &u, 4); return f; }
}  // namespace sacb

namespace sacb {
__global__ void __launch_bounds__(stream::kThreads, 1) stream_selftest_kernel(const __grid_constant__ Program P, const __grid_constant__ Stage stage) {
    extern __shared__ __align__(1024) uint8_t smem_stream[];
    if ((tc::smem_u32(smem_stream) & 1023u) != 0) { if (threadIdx.x == 0) atomicExch(P.error_flag, 3); return; }
    stream::gemm_stage(P, stage, smem_stream, 0ull);
}
}  // namespace sacb

/* the stream kernel's tile (128 rows x bn = 64 | 128 | 256 columns, decoupled producer / MMA / epilogue over a round-robin tile list, `ctas`
 * resident CTAs) against the FFMA tile on the same bf16-pair operands */
extern "C" int sacb_selftest_gemm_stream(int device, int M, int N, int K, int a_mn, int b_mn, int b_r0, int bn, int ctas, float *rel_err_out) {
    if (M < 1 || N < 1 || K < 1 || b_r0 < 0 || (b_mn && b_r0 % 8) || !rel_err_out || (bn != 64 && bn != 128 && bn != 256) || ctas < 1) return fail(SACB_ERR_ARG, "bad argument");
    SACB_CUDA(cudaSetDevice(device));
    const int NB = N + b_r0;
    const int a_rows = a_mn ? K : M, a_cols = a_mn ? M : K, b_rows = b_mn ? K : NB, b_cols = b_mn ? NB : K;
    const int lda = (int)align_up(a_cols, 8) + 8, ldb = (int)align_up(b_cols, 8) + 8;
    const int64_t na = (int64_t)a_rows * lda, nb = (int64_t)b_rows * ldb, nc = (int64_t)M * N;
    std::vector<uint16_t> pa(2 * na, 0), pb(2 * nb, 0);
    std::vector<float> c0(nc), c1(nc);
    uint32_t sd = 777u;
    auto rnd = [&]() { sd = sd * 1664525u + 1013904223u; return ((sd >> 8) & 0xFFFF) / 65536.0f - 0.5f; };
    auto fill = [&](std::vector<uint16_t> &p, int rows, int ld, int64_t n) {
        for (int r = 0; r < rows; r++)
            for (int c = 0; c < ld; c++) {
                const float x = rnd();
                const uint16_t hi = host_bf16_rn(x), lo = host_bf16_rn(x - host_bf16_to_float(hi));
                p[(int64_t)r * ld + c] = hi; p[n + (int64_t)r * ld + c] = lo;
            }
    };
    fill(pa, a_rows, lda, na);
    fill(pb, b_rows, ldb, nb);
    const int64_t oa = 0, ob = align_up(na, 32), oc0 = ob + align_up(nb, 32), oc1 = oc0 + align_up(nc, 32), total = oc1 + align_up(nc, 32);
    float *d; Task *d_tasks; int *flag;
    SACB_CUDA(cudaMalloc(&d, sizeof(float) * total));
    SACB_CUDA(cudaMemset(d, 0, sizeof(float) * total));
    SACB_CUDA(cudaMalloc(&d_tasks, 2 * sizeof(Task)));
    SACB_CUDA(cudaMalloc(&flag, 64)); SACB_CUDA(cudaMemset(flag, 0, 64));
    SACB_CUDA(cudaMemcpy(d + oa, pa.data(), 2 * na * sizeof(uint16_t), cudaMemcpyHostToDevice));
    SACB_CUDA(cudaMemcpy(d + ob, pb.data(), 2 * nb * sizeof(uint16_t), cudaMemcpyHostToDevice));
    AgentBases bases{d, d, 0, 0};
    Task tk[2];
    for (int v = 0; v < 2; v++) {
        Task &t = tk[v]; memset(&t, 0, sizeof(t));
        t.bm = v ? stream::kBM : kSM; t.bn = v ? bn : kSN;
        t.type = T_GEMM; t.M = M; t.N = N; t.K = K; t.epi = EPI_F32;
        t.A.pm.base = make_ref(0, oa); t.A.pm.ld = lda; t.A.pm.plane = na; t.A.mn_major = a_mn; t.A.r0 = 0;
        t.B.pm.base = make_ref(0, ob); t.B.pm.ld = ldb; t.B.pm.plane = nb; t.B.mn_major = b_mn; t.B.r0 = b_r0;
        t.C = make_ref(0, v ? oc1 : oc0); t.ldc = N; t.bias = null_ref();
        t.Cpm = t.mask = null_pm(); t.adam.shadow = t.adam.shadow2 = null_pm();
        t.tiles_m = cdiv(M, t.bm); t.tiles_n = cdiv(N, t.bn); t.n_tiles = t.tiles_m * t.tiles_n;
    }
    int rc = make_pm_tensor_map(&tk[1].tmA, d + oa, a_cols, a_rows, lda, na, 0, 1, a_mn ? 64 : stream::kBM);
    if (rc == SACB_OK) rc = make_pm_tensor_map(&tk[1].tmB, d + ob, b_cols, b_rows, ldb, nb, 0, 1, b_mn ? 64 : bn);
    if (rc) { cudaFree(d); cudaFree(d_tasks); cudaFree(flag); return rc; }
    SACB_CUDA(cudaMemcpy(d_tasks, tk, sizeof(tk), cudaMemcpyHostToDevice));
    gemm_selftest_kernel<SACB_MATH_FP32><<<tk[0].n_tiles, kThreads, kSimtSmemBytes>>>(d_tasks, bases, flag);
    Program P; memset(&P, 0, sizeof(P));
    P.tasks = d_tasks; P.n_agents = 1; P.bases = bases; P.scalars = null_ref(); P.error_flag = flag;
    Stage sg; memset(&sg, 0, sizeof(sg));
    sg.task_begin = 1; sg.task_end = 2; sg.n_tiles = tk[1].n_tiles;
    SACB_CUDA(cudaFuncSetAttribute(stream_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, stream::kSmemBytes));
    stream_selftest_kernel<<<std::min(tk[1].n_tiles, ctas), stream::kThreads, stream::kSmemBytes>>>(P, sg);
    SACB_CUDA(cudaDeviceSynchronize());
    int hf = 0;
    SACB_CUDA(cudaMemcpy(&hf, flag, sizeof(int), cudaMemcpyDeviceToHost));
    SACB_CUDA(cudaMemcpy(c0.data(), d + oc0, sizeof(float) * nc, cudaMemcpyDeviceToHost));
    SACB_CUDA(cudaMemcpy(c1.data(), d + oc1, sizeof(float) * nc, cudaMemcpyDeviceToHost));
    cudaFree(d); cudaFree(d_tasks); cudaFree(flag);
    if (hf) return fail(SACB_ERR_DEVICE, hf == 3 ? "stream kernel: dynamic shared memory is not 1024-byte aligned" : "tcgen05 / TMA pipeline watchdog fired in the stream self test");
    double maxref = 0, maxdiff = 0;
    for (int64_t i = 0; i < nc; i++) { maxref = std::max(maxref, (double)fabsf(c0[i])); maxdiff = std::max(maxdiff, (double)fabsf(c0[i] - c1[i])); }
    *rel_err_out = (float)(maxdiff / std::max(maxref, 1e-30));
    return SACB_OK;
}

extern "C" int sacb_selftest_gemm(int device, int M, int N, int K, int a_mn, int b_mn, int b_r0, float *rel_err_out) {
    return sacb_selftest_gemm_tile(device, M, N, K, a_mn, b_mn, b_r0, kTM, kTN, rel_err_out);
}

extern "C" int sacb_selftest_gemm_tile(int device, int M, int N, int K, int a_mn, int b_mn, int b_r0, int bm, int bn, float *rel_err_out) {
    if (M < 1 || N < 1 || K < 1 || b_r0 < 0 || (b_mn && b_r0 % 8) || !rel_err_out) return fail(SACB_ERR_ARG, "bad argument (an MN-major operand offset must be a multiple of 8)");
    if ((bm != 64 && bm != 128) || (bn != 32 && bn != 64) || (bn == 32 && b_mn)) return fail(SACB_ERR_ARG, "tile shape must be 64|128 x 32|64 (32 columns only with a K-major B operand)");
    SACB_CUDA(cudaSetDevice(device));
    // stored shapes: K-major [R, K], MN-major [K, R]; the B matrix has b_r0 leading rows/columns that are not part of the operand
    const int NB = N + b_r0;
    const int a_rows = a_mn ? K : M, a_cols = a_mn ? M : K, b_rows = b_mn ? K : NB, b_cols = b_mn ? NB : K;
    const int lda = (int)align_up(a_cols, 8) + 8, ldb = (int)align_up(b_cols, 8) + 8;
    const int64_t na = (int64_t)a_rows * lda, nb = (int64_t)b_rows * ldb, nc = (int64_t)M * N;
    std::vector<uint16_t> pa(2 * na, 0), pb(2 * nb, 0);
    std::vector<float> va(na, 0.f), vb(nb, 0.f), c0(nc), c1(nc);     // values the pairs actually represent (hi + lo)
    uint32_t s = 12345u;
    auto rnd = [&]() { s = s * 1664525u + 1013904223u; return ((s >> 8) & 0xFFFF) / 65536.0f - 0.5f; };
    auto fill = [&](std::vector<uint16_t> &p, std::vector<float> &v, int rows, int cols, int ld, int64_t n) {
        for (int r = 0; r < rows; r++)
            for (int c = 0; c < ld; c++) {     // the padding columns hold garbage on purpose: the TMA extent must hide them
                const float x = rnd();
                const uint16_t hi = host_bf16_rn(x), lo = host_bf16_rn(x - host_bf16_to_float(hi));
                p[(int64_t)r * ld + c] = hi; p[n + (int64_t)r * ld + c] = lo;
                if (c < cols) v[(int64_t)r * ld + c] = host_bf16_to_float(hi) + host_bf16_to_float(lo);
            }
    };
    fill(pa, va, a_rows, a_cols, lda, na);
    fill(pb, vb, b_rows, b_cols, ldb, nb);
    // device buffer in float units: [PM A | PM B | C0 | C1]
    const int64_t oa = 0, ob = align_up(na, 32), oc0 = ob + align_up(nb, 32), oc1 = oc0 + align_up(nc, 32), total = oc1 + align_up(nc, 32);
    float *d; Task *d_tasks; int *flag;
    SACB_CUDA(cudaMalloc(&d, sizeof(float) * total));
    SACB_CUDA(cudaMemset(d, 0, sizeof(float) * total));
    SACB_CUDA(cudaMalloc(&d_tasks, 2 * sizeof(Task)));
    SACB_CUDA(cudaMalloc(&flag, 64)); SACB_CUDA(cudaMemset(flag, 0, 64));
    SACB_CUDA(cudaMemcpy(d + oa, pa.data(), 2 * na * sizeof(uint16_t), cudaMemcpyHostToDevice));
    SACB_CUDA(cudaMemcpy(d + ob, pb.data(), 2 * nb * sizeof(uint16_t), cudaMemcpyHostToDevice));
    AgentBases bases{d, d, 0, 0};
    Task tk[2];
    for (int v = 0; v < 2; v++) {
        Task &t = tk[v]; memset(&t, 0, sizeof(t));
        const int tm = v ? bm : kSM, tn = v ? bn : kSN;
        t.bm = tm; t.bn = tn;
        t.type = T_GEMM; t.M = M; t.N = N; t.K = K; t.epi = EPI_F32;
        t.A.pm.base = make_ref(0, oa); t.A.pm.ld = lda; t.A.pm.plane = na; t.A.mn_major = a_mn; t.A.r0 = 0;
        t.B.pm.base = make_ref(0, ob); t.B.pm.ld = ldb; t.B.pm.plane = nb; t.B.mn_major = b_mn; t.B.r0 = b_r0;
        t.C = make_ref(0, v ? oc1 : oc0); t.ldc = N; t.bias = null_ref();
        t.Cpm = t.mask = null_pm(); t.adam.shadow = t.adam.shadow2 = null_pm();
        t.tiles_m = cdiv(M, tm); t.tiles_n = cdiv(N, tn); t.n_tiles = t.tiles_m * t.tiles_n;
    }
    int rc = make_pm_tensor_map(&tk[1].tmA, d + oa, a_cols, a_rows, lda, na, 0, 1, a_mn ? 64 : bm);
    if (rc == SACB_OK) rc = make_pm_tensor_map(&tk[1].tmB, d + ob, b_cols, b_rows, ldb, nb, 0, 1, b_mn ? 64 : bn);
    if (rc) { cudaFree(d); cudaFree(d_tasks); cudaFree(flag); return rc; }
    SACB_CUDA(cudaMemcpy(d_tasks, tk, sizeof(tk), cudaMemcpyHostToDevice));
    gemm_selftest_kernel<SACB_MATH_FP32><<<tk[0].n_tiles, kThreads, kSimtSmemBytes>>>(d_tasks, bases, flag);
    SACB_CUDA(cudaFuncSetAttribute(gemm_selftest_kernel<SACB_MATH_BF16X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes));
    gemm_selftest_kernel<SACB_MATH_BF16X3><<<std::min(tk[1].n_tiles, 148), kThreads, kTcSmemBytes>>>(d_tasks + 1, bases, flag);
    SACB_CUDA(cudaDeviceSynchronize());
    int hf = 0;
    SACB_CUDA(cudaMemcpy(&hf, flag, sizeof(int), cudaMemcpyDeviceToHost));
    SACB_CUDA(cudaMemcpy(c0.data(), d + oc0, sizeof(float) * nc, cudaMemcpyDeviceToHost));
    SACB_CUDA(cudaMemcpy(c1.data(), d + oc1, sizeof(float) * nc, cudaMemcpyDeviceToHost));
    cudaFree(d); cudaFree(d_tasks); cudaFree(flag);
    // host reference in double on a sample of entries pins the FFMA tile itself
    double maxref = 0, maxdiff = 0, maxdiff_host = 0;
    for (int64_t i = 0; i < nc; i++) { maxref = std::max(maxref, (double)fabsf(c0[i])); maxdiff = std::max(maxdiff, (double)fabsf(c0[i] - c1[i])); }
    for (int64_t i = 0; i < nc; i += std::max<int64_t>(1, nc / 257)) {
        const int m = (int)(i / N), n = (int)(i % N) + b_r0;
        double acc = 0;
        for (int k = 0; k < K; k++) acc += (double)(a_mn ? va[(int64_t)k * lda + m] : va[(int64_t)m * lda + k]) * (double)(b_mn ? vb[(int64_t)k * ldb + n] : vb[(int64_t)n * ldb + k]);
        maxdiff_host = std::max(maxdiff_host, fabs(acc - (double)c0[i]));
    }
    if (hf) return fail(SACB_ERR_DEVICE, "tcgen05 / TMA pipeline watchdog fired in the self test");
    if (maxdiff_host > 1e-4 * std::max(1.0, maxref)) return fail(SACB_ERR_DEVICE, "FFMA tile disagrees with the host reference");
    *rel_err_out = (float)(maxdiff / std::max(maxref, 1e-30));
    return SACB_OK;
}
