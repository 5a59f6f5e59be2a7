// C-ABI entry points: handle life cycle, state_dict plumbing, update_parameters, select_action, timing.
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <cmath>
#include <functional>
#include <vector>

#include "handle.h"
#include "gemm.cuh"

namespace sacb {
static thread_local std::string g_err;
void set_error(const std::string &m) { g_err = m; }
int fail(int code, const std::string &m) { g_err = m; return code; }
int init_kernel_attributes(sacb_handle h);
}  // namespace sacb
using namespace sacb;

extern "C" const char *sacb_last_error(void) { return g_err.c_str(); }
extern "C" const char *sacb_version(void) { return "sacb200 0.1 (sm_100a)"; }

extern "C" void sacb_default_config(sacb_config *c) {
    memset(c, 0, sizeof(*c));
    c->hidden_dim = 256; c->n_hidden = 2;
    c->gamma = 0.99f; c->tau = 0.005f; c->lr = 3e-4f; c->alpha0 = 0.2f; c->auto_entropy = 1;   // sac_imp.py:13-18
    c->action_scale = 0.4f; c->action_bias = 0.0f;                                                // networks_model1.py:52-55
    c->replay_kind = SACB_REPLAY_UNIFORM; c->capacity = 1000000;                                  // replay_buffer.py:7
    c->per_alpha = 0.6f; c->per_beta_start = 0.4f; c->per_beta_frames = 100000;                   // replay_buffer.py:26
    c->max_batch = 256; c->n_agents = 1;
    c->math_mode = SACB_MATH_BF16X3; c->launch_mode = SACB_LAUNCH_STAGED; c->device = 0; c->seed = 0x5ac0b200ull;
}

extern "C" int sacb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n; i++) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ok++;
    }
    return ok;
}

static int scalars_init(sacb_handle h) {
    std::vector<float> sc(32, 0.f);
    sc[SC_ALPHA0] = sc[SC_ALPHA1] = h->cfg.alpha0;     // python float 0.2 until the first update (quirk Q1)
    sc[SC_LR] = h->cfg.lr; sc[SC_GAMMA] = h->cfg.gamma; sc[SC_TAU] = h->cfg.tau;
    sc[SC_TARGET_ENTROPY] = -(float)h->cfg.act_dim;    // sac_imp.py:46
    for (int slot = SC_STEP_POLICY; slot <= SC_STEP_ALPHA; slot++) adam_factors_store(sc.data(), slot, 0);
    for (int a = 0; a < h->cfg.n_agents; a++)
        SACB_CUDA(cudaMemcpyAsync(h->arena + a * h->L.arena_size + h->L.scalars, sc.data(), 32 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    return cudaStreamSynchronize(h->stream) == cudaSuccess ? SACB_OK : SACB_ERR_DEVICE;
}

extern "C" int sacb_create(const sacb_config *cfg, sacb_handle *out) {
    if (!cfg || !out) return fail(SACB_ERR_ARG, "null argument");
    if (cfg->obs_dim < 1 || cfg->act_dim < 1 || cfg->hidden_dim < 8 || cfg->hidden_dim % 8) return fail(SACB_ERR_ARG, "bad dims (hidden_dim must be a multiple of 8)");
    if (cfg->n_hidden != 2 && cfg->n_hidden != 3) return fail(SACB_ERR_ARG, "n_hidden must be 2 (networks_model1) or 3 (networks_model2)");
    if (cfg->max_batch < 1 || cfg->n_agents < 1 || cfg->capacity < 1) return fail(SACB_ERR_ARG, "bad max_batch / n_agents / capacity");
    if (2 * cfg->act_dim > 256) return fail(SACB_ERR_ARG, "act_dim > 128 unsupported");
    if (cfg->layer_norm && cfg->n_agents != 1) return fail(SACB_ERR_ARG, "layer_norm: single-agent handles only (the population programs are not validated with it)");
    if (cfg->replay_kind == SACB_REPLAY_PER && cfg->n_agents > 1 && cfg->capacity > kPopulationPerCapacity)
        return fail(SACB_ERR_ARG, "prioritized population: capacity <= 2096128 per agent (the tail-free sampler form)");
    if (cfg->layer_norm && cfg->hidden_dim > 1024) return fail(SACB_ERR_ARG, "layer_norm: hidden_dim > 1024 unsupported (a row is normalised in registers)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device >= ndev) { cudaGetLastError(); return fail(SACB_ERR_DEVICE, "no CUDA device: this library has no CPU fallback"); }
    cudaDeviceProp prop;
    SACB_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10) return fail(SACB_ERR_DEVICE, "device is not sm_100 (B200): kernels are compiled for sm_100a only");
    SACB_CUDA(cudaSetDevice(cfg->device));
    sacb_handle h = new sacb_handle_s();
    h->cfg = *cfg;
    h->sm_count = prop.multiProcessorCount;
    h->use_pdl = getenv("SACB_NO_PDL") ? 0 : 1;
    h->L.build(cfg->obs_dim, cfg->act_dim, cfg->hidden_dim, cfg->n_hidden, cfg->max_batch, cfg->layer_norm != 0);
    const int n = cfg->n_agents;
    auto bail = [&](int rc) { sacb_destroy(h); return rc; };
    {   // the update runs on the highest-priority stream: when sacb_per_step overlaps replay work (second, lowest-priority stream) with the
        // tail of the update, a freed SM goes to a waiting stage CTA first
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        if (cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) return bail(fail(SACB_ERR_DEVICE, "stream create failed"));
    }
    if (cudaMalloc(&h->arena, sizeof(float) * h->L.arena_size * n) != cudaSuccess ||
        cudaMalloc(&h->ws, sizeof(float) * h->L.ws_size * n) != cudaSuccess ||
        cudaMalloc(&h->barrier, 64) != cudaSuccess || cudaMalloc(&h->error_flag, 64) != cudaSuccess ||
        cudaMalloc(&h->slots, sizeof(int32_t) * cfg->max_batch * n) != cudaSuccess ||
        cudaMalloc(&h->slots_identity, sizeof(int32_t) * cfg->max_batch) != cudaSuccess)
        return bail(fail(SACB_ERR_NOMEM, "device allocation failed"));
    {
        std::vector<int32_t> ident(cfg->max_batch);
        for (int i = 0; i < cfg->max_batch; i++) ident[i] = i;
        cudaMemcpyAsync(h->slots_identity, ident.data(), sizeof(int32_t) * cfg->max_batch, cudaMemcpyHostToDevice, h->stream);
        cudaStreamSynchronize(h->stream);
    }
    cudaMemsetAsync(h->arena, 0, sizeof(float) * h->L.arena_size * n, h->stream);
    cudaMemsetAsync(h->ws, 0, sizeof(float) * h->L.ws_size * n, h->stream);
    cudaMemsetAsync(h->barrier, 0, 64, h->stream);
    cudaMemsetAsync(h->error_flag, 0, 64, h->stream);
    cudaMemsetAsync(h->slots, 0, sizeof(int32_t) * cfg->max_batch * n, h->stream);
    {   // Adam bias corrections for every step count that still differs from (1, 1) in float32
        std::vector<AdamBias> tab(kAdamTable);
        for (int t = 0; t < kAdamTable; t++) tab[t] = adam_bias(t);
        if (cudaMalloc(&h->adam_table, sizeof(AdamBias) * kAdamTable) != cudaSuccess) return bail(fail(SACB_ERR_NOMEM, "device allocation failed"));
        cudaMemcpyAsync(h->adam_table, tab.data(), sizeof(AdamBias) * kAdamTable, cudaMemcpyHostToDevice, h->stream);
        cudaStreamSynchronize(h->stream);
    }
    if (cfg->layer_norm) {      // LayerNorm weights start at 1 (torch.nn.LayerNorm), biases at 0 (the memset above)
        std::vector<float> ones(cfg->hidden_dim, 1.0f);
        for (int a = 0; a < n; a++)
            for (int net = 0; net < 5; net++) {
                const NetLayout &nl = net == 0 ? h->L.pol : h->L.q;
                for (int l = 0; l < nl.n_hidden; l++)
                    cudaMemcpyAsync(h->arena + (int64_t)a * h->L.arena_size + h->L.param[net] + nl.g[l], ones.data(), sizeof(float) * cfg->hidden_dim, cudaMemcpyHostToDevice, h->stream);
            }
        cudaStreamSynchronize(h->stream);
    }
    int rc = scalars_init(h);
    if (rc) return bail(fail(rc, "scalar init failed"));
    rc = init_kernel_attributes(h);
    if (rc) return bail(rc);
    rc = replay_create(h);
    if (rc) return bail(rc);
    h->pin_floats = (int64_t)cfg->max_batch * (2 * cfg->obs_dim + 3 * cfg->act_dim + 8) + 64;
    if (cudaMallocHost(&h->pin, sizeof(float) * h->pin_floats) != cudaSuccess) return bail(fail(SACB_ERR_NOMEM, "pinned allocation failed"));
    if (cudaMallocHost(&h->pin_small, sizeof(float) * 16) != cudaSuccess || cudaMallocHost(&h->pin_push, sizeof(float) * h->ring_row * kPinPushRows) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_push, cudaEventDisableTiming) != cudaSuccess)
        return bail(fail(SACB_ERR_NOMEM, "pinned allocation failed"));
    *out = h;
    return SACB_OK;
}

extern "C" int sacb_destroy(sacb_handle h) {
    if (!h) return SACB_OK;
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    free_programs(h);
    replay_destroy(h);
    for (int p = 0; p < h->dp_world; p++)      // peers' arenas mapped for the data-parallel exchange
        if (p != h->dp_rank && h->dp_peer_arena[p]) cudaIpcCloseMemHandle(h->dp_peer_arena[p]);
    cudaFree(h->arena); cudaFree(h->ws); cudaFree(h->barrier); cudaFree(h->error_flag); cudaFree(h->slots); cudaFree(h->slots_identity); cudaFree(h->adam_table); cudaFree(h->slots_staged);
    if (h->pin) cudaFreeHost(h->pin);
    if (h->pin_small) cudaFreeHost(h->pin_small);
    if (h->pin_hist) cudaFreeHost(h->pin_hist);
    if (h->pin_push) cudaFreeHost(h->pin_push);
    if (h->pin_u) cudaFreeHost(h->pin_u);
    if (h->ev_u) cudaEventDestroy(h->ev_u);
    if (h->ev_loss) cudaEventDestroy(h->ev_loss);
    cudaFree(h->act_ws);
    if (h->pin_act) cudaFreeHost(h->pin_act);
    if (h->ev_push) cudaEventDestroy(h->ev_push);
    if (h->ev_slots) cudaEventDestroy(h->ev_slots);
    if (h->pin_rows) cudaFreeHost(h->pin_rows);
    if (h->stream2) { cudaStreamSynchronize(h->stream2); cudaStreamDestroy(h->stream2); }
    if (h->ev_td) cudaEventDestroy(h->ev_td);
    if (h->ev_sampled) cudaEventDestroy(h->ev_sampled);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return SACB_OK;
}

extern "C" int sacb_invalidate_shadows(sacb_handle h) {
    if (!h) return fail(SACB_ERR_ARG, "null handle");
    h->shadows_valid = false;
    return SACB_OK;
}

extern "C" int sacb_get_stream(sacb_handle h, void **stream_out) {
    if (!h || !stream_out) return fail(SACB_ERR_ARG, "null argument");
    *stream_out = (void *)h->stream;
    return SACB_OK;
}

extern "C" int sacb_synchronize(sacb_handle h) {
    if (!h) return fail(SACB_ERR_ARG, "null handle");
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return check_error_flag(h);
}

// ---- state_dict plumbing -----------------------------------------------------------------------------------------
static const NetLayout &net_layout(sacb_handle h, int net) { return net == SACB_NET_POLICY ? h->L.pol : h->L.q; }

extern "C" int sacb_num_tensors(sacb_handle h, int net) {
    if (!h || net < 0 || net > 4) return fail(SACB_ERR_ARG, "bad net id");
    return net_layout(h, net).n_tensors();
}

static int tensor_offset(sacb_handle h, int agent, int net, int slot, int tensor, int64_t *off, int64_t *n) {
    if (!h || net < 0 || net > 4 || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad net / agent id");
    const NetLayout &nl = net_layout(h, net);
    if (tensor < 0 || tensor >= nl.n_tensors()) return fail(SACB_ERR_ARG, "bad tensor index");
    int64_t o, r, c;
    nl.tensor(tensor, o, r, c);
    int64_t base;
    if (slot == SACB_SLOT_PARAM) base = h->L.param[net];
    else {
        if (net > SACB_NET_Q2) return fail(SACB_ERR_ARG, "target networks have no optimizer state");
        base = slot == SACB_SLOT_ADAM_M ? h->L.adam_m[net] : slot == SACB_SLOT_ADAM_V ? h->L.adam_v[net] : h->L.grad[net];
        if (slot < 0 || slot > SACB_SLOT_GRAD) return fail(SACB_ERR_ARG, "bad slot");
    }
    *off = (int64_t)agent * h->L.arena_size + base + o;
    *n = r * c;
    return SACB_OK;
}

extern "C" int sacb_tensor_info(sacb_handle h, int net, int tensor, int64_t *rows, int64_t *cols, int64_t *arena_offset) {
    if (!h || net < 0 || net > 4) return fail(SACB_ERR_ARG, "bad net id");
    const NetLayout &nl = net_layout(h, net);
    if (tensor < 0 || tensor >= nl.n_tensors()) return fail(SACB_ERR_ARG, "bad tensor index");
    int64_t o, r, c;
    nl.tensor(tensor, o, r, c);
    if (rows) *rows = r;
    if (cols) *cols = c;
    if (arena_offset) *arena_offset = h->L.param[net] + o;
    return SACB_OK;
}

extern "C" int sacb_tensor_dev(sacb_handle h, int agent, int net, int slot, int tensor, void **dev_ptr) {
    int64_t off, n;
    int rc = tensor_offset(h, agent, net, slot, tensor, &off, &n);
    if (rc) return rc;
    *dev_ptr = h->arena + off;
    return SACB_OK;
}

extern "C" int sacb_import_tensor(sacb_handle h, int agent, int net, int slot, int tensor, const float *src, int64_t n) {
    int64_t off, cnt;
    int rc = tensor_offset(h, agent, net, slot, tensor, &off, &cnt);
    if (rc) return rc;
    if (n != cnt) return fail(SACB_ERR_ARG, "tensor size mismatch");
    if (slot == SACB_SLOT_PARAM) h->shadows_valid = false;
    SACB_CUDA(cudaMemcpyAsync(h->arena + off, src, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

extern "C" int sacb_export_tensor(sacb_handle h, int agent, int net, int slot, int tensor, float *dst, int64_t n) {
    int64_t off, cnt;
    int rc = tensor_offset(h, agent, net, slot, tensor, &off, &cnt);
    if (rc) return rc;
    if (n != cnt) return fail(SACB_ERR_ARG, "tensor size mismatch");
    SACB_CUDA(cudaMemcpyAsync(dst, h->arena + off, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

static inline int64_t f2i(float f) { int32_t i; memcpy(&i, &f, 4); return i; }
static inline float i2f(int64_t v) { int32_t i = (int32_t)v; float f; memcpy(&f, &i, 4); return f; }

extern "C" int sacb_get_scalars(sacb_handle h, int agent, sacb_scalars *out) {
    if (!h || !out || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    float sc[32];
    SACB_CUDA(cudaMemcpyAsync(sc, h->arena + agent * h->L.arena_size + h->L.scalars, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    out->n_updates = f2i(sc[SC_N_UPDATES]);
    out->log_alpha = sc[SC_LOG_ALPHA]; out->log_alpha_m = sc[SC_LOG_ALPHA_M]; out->log_alpha_v = sc[SC_LOG_ALPHA_V];
    out->alpha = sc[SC_ALPHA0 + (out->n_updates & 1)];
    out->step_policy = f2i(sc[SC_STEP_POLICY]); out->step_q1 = f2i(sc[SC_STEP_Q1]); out->step_q2 = f2i(sc[SC_STEP_Q2]);
    out->step_alpha = f2i(sc[SC_STEP_ALPHA]);
    out->act_counter = h->act_counter;
    return SACB_OK;
}

extern "C" int sacb_set_scalars(sacb_handle h, int agent, const sacb_scalars *in) {
    if (!h || !in || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    float sc[32];
    float *dev = h->arena + agent * h->L.arena_size + h->L.scalars;
    SACB_CUDA(cudaMemcpyAsync(sc, dev, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    sc[SC_LOG_ALPHA] = in->log_alpha; sc[SC_LOG_ALPHA_M] = in->log_alpha_m; sc[SC_LOG_ALPHA_V] = in->log_alpha_v;
    sc[SC_ALPHA0] = sc[SC_ALPHA1] = in->alpha;
    sc[SC_STEP_POLICY] = i2f(in->step_policy); sc[SC_STEP_Q1] = i2f(in->step_q1); sc[SC_STEP_Q2] = i2f(in->step_q2);
    sc[SC_STEP_ALPHA] = i2f(in->step_alpha); sc[SC_N_UPDATES] = i2f(in->n_updates);
    for (int slot = SC_STEP_POLICY; slot <= SC_STEP_ALPHA; slot++) adam_factors_store(sc, slot, (int)f2i(sc[slot]));
    SACB_CUDA(cudaMemcpyAsync(dev, sc, sizeof(sc), cudaMemcpyHostToDevice, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    h->act_counter = (uint32_t)in->act_counter;
    return SACB_OK;
}

// read-modify-write of an agent's scalar block, ordered on the handle's stream
static int edit_scalars(sacb_handle h, int agent, const std::function<void(float *)> &edit) {
    float sc[32];
    float *dev = h->arena + agent * h->L.arena_size + h->L.scalars;
    SACB_CUDA(cudaMemcpyAsync(sc, dev, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    edit(sc);
    SACB_CUDA(cudaMemcpyAsync(dev, sc, sizeof(sc), cudaMemcpyHostToDevice, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}
// a new SC_LR: the cached factors of the NEXT step of every optimizer follow it
static void refresh_factors(float *sc) {
    for (int slot = SC_STEP_POLICY; slot <= SC_STEP_ALPHA; slot++) adam_factors_store(sc, slot, (int)f2i(sc[slot]));
}

extern "C" int sacb_set_lr(sacb_handle h, float lr) {
    if (!h || !(lr > 0.f) || !std::isfinite(lr)) return fail(SACB_ERR_ARG, "bad learning rate");
    h->cfg.lr = lr;
    for (int a = 0; a < h->cfg.n_agents; a++)
        if (int rc = edit_scalars(h, a, [&](float *sc) { sc[SC_LR] = lr; refresh_factors(sc); })) return rc;
    return SACB_OK;
}

extern "C" int sacb_get_hparams(sacb_handle h, int agent, sacb_hparams *out) {
    if (!h || !out || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    float sc[32];
    SACB_CUDA(cudaMemcpyAsync(sc, h->arena + agent * h->L.arena_size + h->L.scalars, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    out->lr = sc[SC_LR]; out->gamma = sc[SC_GAMMA]; out->tau = sc[SC_TAU]; out->target_entropy = sc[SC_TARGET_ENTROPY];
    return SACB_OK;
}

extern "C" int sacb_set_hparams(sacb_handle h, int agent, const sacb_hparams *in) {
    if (!h || !in || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    if (!(in->lr > 0.f) || !std::isfinite(in->lr)) return fail(SACB_ERR_ARG, "lr must be finite and > 0");
    if (!(in->gamma >= 0.f && in->gamma <= 1.f)) return fail(SACB_ERR_ARG, "gamma must lie in [0, 1]");
    if (!(in->tau >= 0.f && in->tau <= 1.f)) return fail(SACB_ERR_ARG, "tau must lie in [0, 1]");
    if (!std::isfinite(in->target_entropy)) return fail(SACB_ERR_ARG, "target_entropy must be finite");
    return edit_scalars(h, agent, [&](float *sc) {
        sc[SC_LR] = in->lr; sc[SC_GAMMA] = in->gamma; sc[SC_TAU] = in->tau; sc[SC_TARGET_ENTROPY] = in->target_entropy;
        refresh_factors(sc);
    });
}

/* exploit step of population-based training: agent dst[i] takes over the whole learner state of agent src[i] (one contiguous arena
 * span: weights, targets, Adam moments, weight shadows, scalar block).  Replay rings and workspaces stay with their agent. */
extern "C" int sacb_copy_agents(sacb_handle h, const int32_t *dst, const int32_t *src, int n) {
    if (!h || n < 0 || (n > 0 && (!dst || !src))) return fail(SACB_ERR_ARG, "bad argument");
    const int na = h->cfg.n_agents;
    std::vector<char> is_dst(na, 0), is_src(na, 0);
    for (int i = 0; i < n; i++) {
        if (dst[i] < 0 || dst[i] >= na || src[i] < 0 || src[i] >= na) return fail(SACB_ERR_ARG, "agent index out of range");
        if (is_dst[dst[i]]) return fail(SACB_ERR_ARG, "an agent appears twice as a destination");
        is_dst[dst[i]] = 1; is_src[src[i]] = 1;
    }
    for (int a = 0; a < na; a++)
        if (is_dst[a] && is_src[a]) return fail(SACB_ERR_ARG, "an agent appears as a source and as a destination");
    const size_t bytes = sizeof(float) * h->L.arena_size;
    for (int i = 0; i < n; i++)
        SACB_CUDA(cudaMemcpyAsync(h->arena + (int64_t)dst[i] * h->L.arena_size, h->arena + (int64_t)src[i] * h->L.arena_size, bytes,
                                  cudaMemcpyDeviceToDevice, h->stream));
    return SACB_OK;
}

extern "C" int sacb_get_losses(sacb_handle h, int agent, float *losses_out) {
    if (!h || !losses_out || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    SACB_CUDA(cudaMemcpyAsync(losses_out, h->arena + agent * h->L.arena_size + h->L.scalars + SC_LOSS_Q1, 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return check_error_flag(h);
}

extern "C" int sacb_get_losses_all(sacb_handle h, float *losses_out) {
    if (!h || !losses_out) return fail(SACB_ERR_ARG, "bad argument");
    // one strided copy: the loss scalars sit at the same offset of every agent's arena
    SACB_CUDA(cudaMemcpy2DAsync(losses_out, 3 * sizeof(float), h->arena + h->L.scalars + SC_LOSS_Q1, sizeof(float) * h->L.arena_size, 3 * sizeof(float),
                                h->cfg.n_agents, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return check_error_flag(h);
}

// ---- update_parameters ---------------------------------------------------------------------------------------------
static int upload_eps(sacb_handle h, int agent, int64_t B, const float *eps_next, const float *eps_cur) {
    float *ws = h->ws + agent * h->L.ws_size;
    const int64_t n = B * h->cfg.act_dim;
    if (eps_next) SACB_CUDA(cudaMemcpyAsync(ws + h->L.eps, eps_next, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    if (eps_cur) SACB_CUDA(cudaMemcpyAsync(ws + h->L.eps + n, eps_cur, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    return SACB_OK;
}

// write_back_B > 0: the |TD| priority write-back of the minibatch (replay_buffer.py:84-87) is enqueued BEHIND the loss copy and the host
// waits for the copy only -- its launches cost the host nothing (the device is still busy with the update) and the device runs it
// while the caller is back in Python
static int finish_update(sacb_handle h, float *losses_out, uint32_t flags, int64_t write_back_B = 0) {
    if ((flags & SACB_NO_LOSS_READBACK) || !losses_out) {
        if (write_back_B > 0) { if (int rc = per_writeback_launch(h, h->stream, write_back_B, true, 0, h->cfg.n_agents)) return rc; }
        return (flags & SACB_NO_LOSS_READBACK) ? SACB_OK : sacb_synchronize(h);
    }
    // the three losses (the `.item()` calls of sac_imp.py:141-143) and the device error flag: the last stage of the step (T_FINISH) has
    // stored them into the pinned block itself (Program::host_losses), ONE synchronisation and no copy behind the step.
    // (population handles: one D2H copy of the five floats)
    static_assert(SC_ERROR_FLAG == SC_LOSS_Q1 + 4, "losses and the flag copy are contiguous");
    if (h->cfg.n_agents != 1)
        SACB_CUDA(cudaMemcpyAsync(h->pin_small, h->arena + h->L.scalars + SC_LOSS_Q1, 5 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (write_back_B > 0) {
        if (!h->ev_loss) SACB_CUDA(cudaEventCreateWithFlags(&h->ev_loss, cudaEventDisableTiming));
        SACB_CUDA(cudaEventRecord(h->ev_loss, h->stream));
        if (int rc = per_writeback_launch(h, h->stream, write_back_B, true, 0, h->cfg.n_agents)) return rc;
        SACB_CUDA(cudaEventSynchronize(h->ev_loss));
    } else {
        SACB_CUDA(cudaStreamSynchronize(h->stream));
    }
    memcpy(losses_out, h->pin_small, 3 * sizeof(float));
    int32_t flag;
    memcpy(&flag, h->pin_small + 4, sizeof(flag));
    return flag ? check_error_flag(h) : SACB_OK;
}

extern "C" int sacb_update_batch(sacb_handle h, int64_t B, const float *s, const float *a, const float *r, const float *s2,
                                 const float *done, const float *isw, const float *eps_next, const float *eps_cur,
                                 float *losses_out, float *td_abs_out, uint32_t flags) {
    if (!h || !s || !a || !r || !s2 || !done) return fail(SACB_ERR_ARG, "null minibatch pointer");
    if (h->cfg.n_agents != 1) return fail(SACB_ERR_ARG, "sacb_update_batch drives a single agent");
    if ((eps_next == nullptr) != (eps_cur == nullptr)) return fail(SACB_ERR_ARG, "pass both eps arrays or neither");
    const Layout &L = h->L;
    if (B < 1 || B > L.maxB) return fail(SACB_ERR_ARG, "batch size out of range");
    float *ws = h->ws;
    // pack the minibatch as replay rows [s | s2 | a | r | d] in pinned memory, one H2D copy into the staging rows;
    // the program's gather stage (slots = identity) then builds the bf16 pair operands exactly as it does from the ring
    const int64_t row = h->ring_row;
    if (B > h->stage_rows_cap) return fail(SACB_ERR_ARG, "batch exceeds the staging capacity");
    if (h->pin_rows_cap < B) {
        if (h->pin_rows) cudaFreeHost(h->pin_rows);
        h->pin_rows = nullptr; h->pin_rows_cap = 0;
        if (cudaMallocHost(&h->pin_rows, sizeof(float) * row * B) != cudaSuccess) return fail(SACB_ERR_NOMEM, "pinned allocation failed");
        h->pin_rows_cap = B;
    }
    SACB_CUDA(cudaStreamSynchronize(h->stream));     // the previous upload out of the pinned rows has completed
    for (int64_t b = 0; b < B; b++) {
        float *dst = h->pin_rows + b * row;
        memcpy(dst, s + b * L.obs, sizeof(float) * L.obs);
        memcpy(dst + L.obs, s2 + b * L.obs, sizeof(float) * L.obs);
        memcpy(dst + 2 * L.obs, a + b * L.act, sizeof(float) * L.act);
        dst[2 * L.obs + L.act] = r[b];
        dst[2 * L.obs + L.act + 1] = done[b];
    }
    SACB_CUDA(cudaMemcpyAsync(h->stage_rows, h->pin_rows, sizeof(float) * row * B, cudaMemcpyHostToDevice, h->stream));
    if (isw) SACB_CUDA(cudaMemcpyAsync(ws + L.isw, isw, sizeof(float) * B, cudaMemcpyHostToDevice, h->stream));
    int rc = upload_eps(h, 0, B, eps_next, eps_cur);
    if (rc) return rc;
    rc = run_update(h, update_key(h, (int)B, 2, (flags & SACB_EXPORT_GRADS) ? 1 : 0, eps_next ? 0 : 1, isw ? 1 : 0));
    if (rc) return rc;
    if (td_abs_out) {
        SACB_CUDA(cudaMemcpyAsync(td_abs_out, ws + L.td, sizeof(float) * B, cudaMemcpyDeviceToHost, h->stream));
        SACB_CUDA(cudaStreamSynchronize(h->stream));
    }
    return finish_update(h, losses_out, flags);
}

namespace sacb { int replay_stage_slots(sacb_handle h, const int64_t *idx, int64_t B); }

extern "C" int sacb_update(sacb_handle h, int64_t B, const int64_t *idx, const float *eps_next, const float *eps_cur,
                           float *losses_out, uint32_t flags) {
    if (!h) return fail(SACB_ERR_ARG, "null handle");
    if (B < 1 || B > h->L.maxB) return fail(SACB_ERR_ARG, "batch size out of range");
    if ((eps_next == nullptr) != (eps_cur == nullptr)) return fail(SACB_ERR_ARG, "pass both eps arrays or neither");
    int rc, gather_mode = 1;
    if (idx) {
        rc = replay_stage_slots(h, idx, B);
        if (rc) return rc;
    } else if (h->staged_steps > 0 && !(flags & SACB_DEVICE_INDICES) && !(flags & SACB_USE_LAST_SAMPLE)) {
        const int64_t k = h->staged_next % h->staged_steps;
        h->staged_next++;
        SACB_CUDA(cudaMemcpyAsync(h->slots, h->slots_staged + k * h->cfg.n_agents * h->staged_B, sizeof(int32_t) * h->staged_B * h->cfg.n_agents,
                                  cudaMemcpyDeviceToDevice, h->stream));
    } else if (flags & SACB_DEVICE_INDICES) {      // positions drawn inside the gather stage (uniform ring, without replacement)
        if (h->cfg.replay_kind != SACB_REPLAY_UNIFORM) return fail(SACB_ERR_ARG, "SACB_DEVICE_INDICES needs the uniform replay ring (the prioritized one has sacb_per_step)");
        for (int a = 0; a < h->cfg.n_agents; a++)
            if (B > h->r_len[a]) return fail(SACB_ERR_STATE, "Sample larger than population or is negative");
        if ((rc = upload_ring_meta(h))) return rc;
        gather_mode = 3;
    } else if (!(flags & SACB_USE_LAST_SAMPLE)) {
        return fail(SACB_ERR_ARG, "no indices: pass idx, stage them, set SACB_DEVICE_INDICES or SACB_USE_LAST_SAMPLE");
    } else if (h->cfg.replay_kind == SACB_REPLAY_PER) {
        // set_priorities / clear / a sample of another size leave no (or a stale) minibatch behind; a population needs every agent's
        for (int a = 0; a < h->cfg.n_agents; a++)
            if (h->sample_k[a] != B) return fail(SACB_ERR_STATE, "SACB_USE_LAST_SAMPLE: the last prioritized sample does not hold B rows (sample again)");
    }
    if (eps_next) for (int a = 0; a < h->cfg.n_agents; a++) {
        const int64_t n = B * h->cfg.act_dim;
        rc = upload_eps(h, a, B, eps_next + a * n, eps_cur + a * n);
        if (rc) return rc;
    }
    const int use_isw = (h->cfg.per_weighted_loss && h->cfg.replay_kind == SACB_REPLAY_PER) ? 1 : 0;
    rc = run_update(h, update_key(h, (int)B, gather_mode, (flags & SACB_EXPORT_GRADS) ? 1 : 0, eps_next ? 0 : 1, use_isw));
    if (rc) return rc;
    int64_t write_back_B = 0;
    if (flags & SACB_WRITE_BACK_TD) {
        if (h->cfg.replay_kind != SACB_REPLAY_PER || !(flags & SACB_USE_LAST_SAMPLE))
            return fail(SACB_ERR_ARG, "SACB_WRITE_BACK_TD: needs the prioritized buffer and SACB_USE_LAST_SAMPLE");
        write_back_B = B;
    }
    return finish_update(h, losses_out, flags, write_back_B);
}

// ---- test hook: read back a hidden activation matrix of the last update ----------------------------------------------
/* One learner step over the prioritized buffer with every input resident in HBM, software-pipelined across two streams:
 *   stream : update stages up to the updated-critic forward (TD errors exist) ... rest of the update (actor loss, dL/da, policy backward)
 *   stream2:                                          priority write-back |q1 - y| -> prioritized sample for the NEXT step
 * Same kernels, same order of the dependent operations and therefore the same values as sacb_per_sample -> sacb_update(USE_LAST_SAMPLE)
 * -> sacb_per_update_from_td called in sequence (tests/test_gpu_replay.py::test_pipelined_step_equals_sequential). */
static int per_step_enqueue(sacb_handle h, int64_t B) {
    if (!h || h->cfg.replay_kind != SACB_REPLAY_PER || h->cfg.n_agents != 1) return fail(SACB_ERR_ARG, "handle has no prioritized buffer");
    if (B < 1 || B > h->L.maxB) return fail(SACB_ERR_ARG, "batch size out of range");
    if (!h->stream2) {
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        SACB_CUDA(cudaStreamCreateWithPriority(&h->stream2, cudaStreamNonBlocking, prio_lo));
        SACB_CUDA(cudaEventCreateWithFlags(&h->ev_td, cudaEventDisableTiming));
        SACB_CUDA(cudaEventCreateWithFlags(&h->ev_sampled, cudaEventDisableTiming));
    }
    // a frame counter set since the last sample reaches the device ahead of the step, whichever form enqueues it (the main stream has
    // joined the previous step's sample)
    int rc = upload_per_frame(h, h->stream);
    if (rc) return rc;
    const int64_t k = std::min<int64_t>(B, h->r_len[0]);
    if (h->sample_k[0] != k) {      // first call (or the batch size changed): draw this step's minibatch now
        rc = per_sample_launch(h, h->stream, nullptr, B, nullptr, 0, 1);
        if (rc) return rc;
    }
    ProgramKey key = update_key(h, (int)k, 1, 0, 1, h->cfg.per_weighted_loss ? 1 : 0);
    ProgramInst *p;
    rc = get_program(h, key, &p);
    if (rc) return rc;
    // the whole step -- update stages, forked write-back + next sample, join -- as ONE graph launch, else the same launches directly
    rc = launch_per_step_graph(h, *p, B, k);
    if (rc == 1) rc = enqueue_per_step(h, *p, B, k);
    if (rc) return rc;
    after_update_launch(h, key);
    return SACB_OK;
}

extern "C" int sacb_per_step(sacb_handle h, int64_t B, float *losses_out, uint32_t flags) {
    int rc = per_step_enqueue(h, B);
    if (rc) return rc;
    return finish_update(h, losses_out, flags);
}

/* K learner steps per call, nothing of a step touches the host (SURVEY 8f rank 3: "multi-step fused launches with on-device index
 * draw"): K replays of the step graph(s) back to back -- prioritized ring: the sacb_per_step pipeline; uniform ring: positions drawn
 * inside the gather stage (SACB_DEVICE_INDICES) -- then ONE device->host copy of the scalar block and the loss history ring.
 * Bitwise equal to K single calls. */
extern "C" int sacb_update_steps(sacb_handle h, int64_t B, int K, float *losses_out, uint32_t flags) {
    if (!h || K < 1 || K > kLossHist) return fail(SACB_ERR_ARG, "K must be 1..64");
    if (h->cfg.n_agents != 1 && losses_out) return fail(SACB_ERR_ARG, "loss read-back of sacb_update_steps serves a single agent (use sacb_get_losses per agent)");
    int rc;
    for (int i = 0; i < K; i++) {
        if (h->cfg.replay_kind == SACB_REPLAY_PER) rc = per_step_enqueue(h, B);
        else rc = sacb_update(h, B, nullptr, nullptr, nullptr, nullptr, (flags & ~SACB_USE_LAST_SAMPLE) | SACB_DEVICE_INDICES | SACB_NO_LOSS_READBACK);
        if (rc) return rc;
    }
    if ((flags & SACB_NO_LOSS_READBACK) || !losses_out) return (flags & SACB_NO_LOSS_READBACK) ? SACB_OK : sacb_synchronize(h);
    constexpr int kN = 32 + 4 * kLossHist;
    if (!h->pin_hist && cudaMallocHost(&h->pin_hist, sizeof(float) * kN) != cudaSuccess) return fail(SACB_ERR_NOMEM, "pinned allocation failed");
    SACB_CUDA(cudaMemcpyAsync(h->pin_hist, h->arena + h->L.scalars, sizeof(float) * 32, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaMemcpyAsync(h->pin_hist + 32, h->arena + h->L.loss_hist, sizeof(float) * 4 * kLossHist, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    int32_t pos, flag;
    memcpy(&pos, h->pin_hist + SC_HIST_POS, 4);
    memcpy(&flag, h->pin_hist + SC_ERROR_FLAG, 4);
    for (int i = 0; i < K; i++) {
        const int slot = ((pos - K + i) % kLossHist + kLossHist) % kLossHist;
        memcpy(losses_out + 3 * i, h->pin_hist + 32 + 4 * slot, 3 * sizeof(float));
    }
    return flag ? check_error_flag(h) : SACB_OK;
}

extern "C" int sacb_debug_read_activation(sacb_handle h, int agent, int group, int k, int layer, int64_t B, float *out) {
    if (!h || !out || agent < 0 || agent >= h->cfg.n_agents || group < 0 || group > 3 || k < 0 || k > 1 || layer < 0 || layer >= h->L.n_hidden ||
        B < 1 || B > h->L.maxB)
        return fail(SACB_ERR_ARG, "bad argument");
    const Layout &L = h->L;
    const int64_t H = L.hidden, maxB = L.maxB;
    int64_t off, plane, row0 = 0;
    if (group == 0) { off = L.hp[layer]; plane = 2 * maxB * H; row0 = B; }          // rows [B, 2B) = current states
    else { off = group == 1 ? L.hc[k][layer] : group == 2 ? L.ha[k][layer] : L.ht[k][layer]; plane = maxB * H; }
    const uint16_t *base = reinterpret_cast<const uint16_t *>(h->ws + agent * L.ws_size + off) + row0 * H;
    std::vector<uint16_t> hi(B * H), lo(B * H);
    SACB_CUDA(cudaMemcpyAsync(hi.data(), base, sizeof(uint16_t) * B * H, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaMemcpyAsync(lo.data(), base + plane, sizeof(uint16_t) * B * H, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    for (int64_t i = 0; i < B * H; i++) {
        uint32_t a = (uint32_t)hi[i] << 16, b = (uint32_t)lo[i] << 16;
        float fa, fb;
        memcpy(&fa, &a, 4); memcpy(&fb, &b, 4);
        out[i] = fa + fb;
    }
    return SACB_OK;
}

extern "C" int sacb_debug_read_slots(sacb_handle h, int agent, int32_t *slots_out, int64_t B) {
    if (!h || !slots_out || agent < 0 || agent >= h->cfg.n_agents || B < 1 || B > h->L.maxB) return fail(SACB_ERR_ARG, "bad argument");
    SACB_CUDA(cudaMemcpyAsync(slots_out, h->slots + (int64_t)agent * h->cfg.max_batch, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

// ---- instrumentation ---------------------------------------------------------------------------------------------
extern "C" int sacb_get_stats(sacb_handle h, sacb_stats *out) {
    if (!h || !out) return fail(SACB_ERR_ARG, "null argument");
    memset(out, 0, sizeof(*out));
    out->kernel_launches = h->kernel_launches;
    out->sm_count = h->sm_count; out->block = kThreads;
    out->n_programs = (int)h->programs.size();
    out->smem_bytes = (int)math_smem(h->cfg.math_mode);
    for (auto &kv : h->programs) {
        out->n_stages = (int)kv.second.stages.size(); out->n_tasks = (int)kv.second.tasks.size();
        out->n_tiles = kv.second.n_tiles_total; out->grid = kv.second.max_stage_tiles;
    }
    return SACB_OK;
}

extern "C" int sacb_time_update(sacb_handle h, int64_t B, int iters, float *ms_per_step) {
    if (!h || !ms_per_step || iters < 1) return fail(SACB_ERR_ARG, "bad argument");
    ProgramInst *p;
    int rc = steady_program(h, B, &p);
    if (rc) return rc;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int i = 0; i < 3; i++) if ((rc = launch_program(h, *p))) return rc;
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    cudaEventRecord(e0, h->stream);
    for (int i = 0; i < iters; i++) if ((rc = launch_program(h, *p))) return rc;
    cudaEventRecord(e1, h->stream);
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *ms_per_step = ms / iters;
    return check_error_flag(h);
}

static cudaEvent_t g_ev0 = nullptr, g_ev1 = nullptr;
extern "C" int sacb_timer_start(sacb_handle h) {
    if (!h) return fail(SACB_ERR_ARG, "null handle");
    if (!g_ev0) { SACB_CUDA(cudaEventCreate(&g_ev0)); SACB_CUDA(cudaEventCreate(&g_ev1)); }
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    SACB_CUDA(cudaEventRecord(g_ev0, h->stream));
    return SACB_OK;
}
extern "C" int sacb_timer_stop(sacb_handle h, float *ms_out) {
    if (!h || !ms_out || !g_ev0) return fail(SACB_ERR_ARG, "timer not started");
    SACB_CUDA(cudaEventRecord(g_ev1, h->stream));
    SACB_CUDA(cudaEventSynchronize(g_ev1));
    SACB_CUDA(cudaEventElapsedTime(ms_out, g_ev0, g_ev1));
    return check_error_flag(h);
}
