/* sacb200.h -- C ABI of the B200-native SAC learner hot path (libsacb200.so).
 *
 * The reference (FilippoCrc/Humanoid-walking-with-SAC) is pure Python: it has no FFI.  Its boundary for
 * this path is the Python class API of sac_imp.SAC, replay_buffer.ReplayBuffer and
 * replay_buffer.PrioritizedReplayBuffer.  Each entry point below names the reference method it serves
 * (paths relative to the reference checkout); the Python mirror classes in
 * humanoid-walking-with-sac_b200/{sac_imp,replay_buffer}.py bind them through ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, a negative sacb_status otherwise; sacb_last_error() gives text.
 *   - all pointers are HOST pointers owned by the caller unless the name ends in _dev.
 *   - float = IEEE binary32, idx = int64 (numpy default), uniforms = binary64 (RandomState.random_sample).
 *   - one handle = one agent population on one GPU (n_agents >= 1), one private CUDA stream; calls on a
 *     handle are not re-entrant (the reference is single-threaded, trainer.py:182-205).
 *   - there is NO CPU fallback: if no sm_100 device is present sacb_create fails with SACB_ERR_DEVICE.
 */
#ifndef SACB200_H
#define SACB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sacb_handle_s *sacb_handle;

typedef enum {
    SACB_OK = 0,
    SACB_ERR_ARG = -1,       /* bad argument / shape (Python shim raises ValueError) */
    SACB_ERR_DEVICE = -2,    /* no usable sm_100 device / CUDA failure (RuntimeError) */
    SACB_ERR_STATE = -3,     /* e.g. sample larger than population (ValueError, as random.sample does) */
    SACB_ERR_NOMEM = -4
} sacb_status;

/* GEMM arithmetic of the update.  Every GEMM operand (minibatch, activations, gradients, weight shadows) is stored
 * as a bf16 hi/lo pair (x ~= hi + lo, 2^-17 relative); master weights, Adam state and accumulators are fp32. */
enum { SACB_MATH_FP32 = 0,    /* CUDA-core FFMA on the pair operands, fp32 products and accumulate (checker / strict mode) */
       SACB_MATH_BF16X3 = 1   /* TMA-fed tcgen05.mma kind::f16: a_lo*b_hi + a_hi*b_lo + a_hi*b_hi, fp32 accumulate in TMEM
                                 (default; agrees with SACB_MATH_FP32 to ~1e-5 relative) */ };

/* how one update step is launched: */
enum { SACB_LAUNCH_STAGED = 0,     /* one kernel per dependency stage, whole step captured in one CUDA graph */
       SACB_LAUNCH_PERSISTENT = 1 }; /* ONE cooperative launch per step, grid barriers between stages        */

enum { SACB_NET_POLICY = 0, SACB_NET_Q1 = 1, SACB_NET_Q2 = 2, SACB_NET_Q1_TARGET = 3, SACB_NET_Q2_TARGET = 4 };
enum { SACB_SLOT_PARAM = 0, SACB_SLOT_ADAM_M = 1, SACB_SLOT_ADAM_V = 2, SACB_SLOT_GRAD = 3 };
enum { SACB_REPLAY_UNIFORM = 0, SACB_REPLAY_PER = 1 };

/* Constructor arguments of sac_imp.SAC.__init__ (sac_imp.py:9-52) + the network variant it imports
 * (sac_imp.py:4: networks_model1 = 2 hidden layers, networks_model2 = 3) + replay_buffer.py ctor args. */
typedef struct {
    int32_t obs_dim, act_dim, hidden_dim;
    int32_t n_hidden;              /* 2 (networks_model1.py:15-17) or 3 (networks_model2.py:24-27) */
    float gamma, tau, lr, alpha0;  /* sac_imp.py:13-17 */
    int32_t auto_entropy;          /* sac_imp.py:18 */
    float action_scale, action_bias; /* networks_model1.py:52-55 */
    int32_t replay_kind;           /* SACB_REPLAY_*; a population (n_agents > 1) gives every agent its own ring, and with
                                      SACB_REPLAY_PER its own priority table, frame counter and sampler workspace */
    int64_t capacity;              /* replay_buffer.py:7 / :26, per agent.  SACB_REPLAY_PER with n_agents > 1: <= 2 096 128
                                      (the sampler form without serial tails), SACB_ERR_ARG at sacb_create otherwise */
    float per_alpha, per_beta_start; /* replay_buffer.py:26 */
    int64_t per_beta_frames;
    int32_t max_batch;             /* largest batch_size update/sample will be called with */
    int32_t n_agents;              /* independent agents (population mode, BASELINE.json configs[4]); 1 = reference */
    int32_t math_mode;             /* SACB_MATH_* */
    int32_t launch_mode;           /* SACB_LAUNCH_* */
    int32_t device;                /* CUDA ordinal */
    uint64_t seed;                 /* Philox key for on-device eps / index draws (production mode) */
    int32_t per_weighted_loss;     /* extension (SURVEY H10): IS-weighted critic loss + |td| priority write-back */
    int32_t layer_norm;            /* extension, default 0 (the reference has none: networks_model2.py:86 is a comment): LayerNorm with
                                      affine parameters between every hidden Linear and its ReLU of all five networks; parameter
                                      tensors per hidden layer then are weight, bias, ln.weight, ln.bias.  No reference parity.  Single-agent
                                      handles only (n_agents = 1, no sacb_dp_*): SACB_ERR_ARG otherwise. */
    int32_t reserved[6];
} sacb_config;

void sacb_default_config(sacb_config *cfg);
const char *sacb_last_error(void);
const char *sacb_version(void);
/* number of CUDA devices usable by this library (sm_100); 0 if none. */
int sacb_device_count(void);

/* SAC.__init__ (sac_imp.py:9-52): allocates arena (params, targets, Adam m/v), workspaces, replay ring.
 * Parameters start at zero: the host shim uploads the initial weights with sacb_import_tensor. */
int sacb_create(const sacb_config *cfg, sacb_handle *out);
int sacb_destroy(sacb_handle h);
int sacb_synchronize(sacb_handle h);

/* ---- state_dict plumbing: SAC.save/load/save_checkpoint/load_checkpoint (sac_imp.py:154-233) -------------
 * tensor index = position in Module.parameters() order (fc1.weight, fc1.bias, ..., see sacb_tensor_info). */
int sacb_num_tensors(sacb_handle h, int net);
int sacb_tensor_info(sacb_handle h, int net, int tensor, int64_t *rows, int64_t *cols, int64_t *arena_offset);
/* device pointer of a tensor (agent-major arenas): lets the host alias it as a torch tensor (zero copy). */
int sacb_tensor_dev(sacb_handle h, int agent, int net, int slot, int tensor, void **dev_ptr);
int sacb_import_tensor(sacb_handle h, int agent, int net, int slot, int tensor, const float *src, int64_t n);
int sacb_export_tensor(sacb_handle h, int agent, int net, int slot, int tensor, float *dst, int64_t n);
/* The GEMMs read bf16 hi/lo shadows of the weights that the update's own Adam / Polyak epilogues keep current.  A write of fp32
 * weights from OUTSIDE the library (through the torch aliases of sacb_tensor_dev: load_state_dict, in-place edits) must be followed
 * by this call; the next update then re-derives every shadow first.  sacb_import_tensor does it implicitly. */
int sacb_invalidate_shadows(sacb_handle h);
/* scalars: log_alpha + its Adam state (sac_imp.py:48-49), alpha (:23,:135), per-optimizer step counts. */
typedef struct {
    float log_alpha, alpha, log_alpha_m, log_alpha_v;
    int64_t step_policy, step_q1, step_q2, step_alpha, n_updates;
    int64_t act_counter;   /* Philox counter of select_action's exploration draws (per handle; saved by save_checkpoint) */
} sacb_scalars;
int sacb_get_scalars(sacb_handle h, int agent, sacb_scalars *out);
int sacb_set_scalars(sacb_handle h, int agent, const sacb_scalars *in);
/* torch.optim.Adam.load_state_dict restores param_groups[0]['lr'] (sac_imp.py:215-218): sets the learning rate of every agent (all
 * four optimizers of an agent share it, sac_imp.py:39-49) and refreshes their cached bias-correction factors.  No program is rebuilt. */
int sacb_set_lr(sacb_handle h, float lr);
/* Hyperparameters of one agent, kept in its scalar block on the device: every update reads them there, so changing one never rebuilds
 * or re-captures an update program.  sacb_create gives every agent lr, gamma, tau of sacb_config and target_entropy = -act_dim
 * (sac_imp.py:46).  lr drives all four optimizers of the agent; target_entropy matters with auto_entropy only.  Per-agent alpha:
 * sacb_set_scalars.  sacb_set_hparams: lr finite and > 0, gamma and tau in [0, 1], target_entropy finite (SACB_ERR_ARG otherwise);
 * the agent's cached Adam factors follow the new lr at its current step counts.  Both calls are ordered on the handle's stream. */
typedef struct { float lr, gamma, tau, target_entropy; } sacb_hparams;
int sacb_get_hparams(sacb_handle h, int agent, sacb_hparams *out);
int sacb_set_hparams(sacb_handle h, int agent, const sacb_hparams *in);
/* Exploit step of population-based training: for each i, agent dst[i] takes over the whole learner state of agent src[i] -- weights,
 * Polyak targets, Adam moments, weight shadows and the scalar block (hyperparameters, step counts, log_alpha and its Adam state,
 * alpha, cached factors, loss history).  Replay rings and workspaces are not copied.  Device-to-device copies enqueued on the handle's
 * stream (no host synchronisation).  The destination keeps its own Philox streams: on-device draws are keyed by agent index, so after
 * the copy dst[i] continues with src[i]'s step count but draws its own minibatch positions and noise.  SACB_ERR_ARG for an index out
 * of range, a repeated dst, or an index that appears both as a src and as a dst in the same call. */
int sacb_copy_agents(sacb_handle h, const int32_t *dst, const int32_t *src, int n);

/* ---- replay: ReplayBuffer.push / PrioritizedReplayBuffer.push (replay_buffer.py:10-11, :36-46) ----------
 * n transitions, row-major float32 (the cast of sac_imp.py:81-85 happens in the shim); done as 0/1 floats. */
int sacb_push(sacb_handle h, int agent, const float *s, const float *a, const float *r, const float *s2,
              const float *done, int64_t n);
/* same, rows already packed by the caller as [s | s2 | a | r | d] padded to sacb_row_floats(): one H2D copy */
int sacb_push_rows(sacb_handle h, int agent, const float *rows, int64_t n);
int64_t sacb_row_floats(sacb_handle h);
int64_t sacb_len(sacb_handle h, int agent);                     /* __len__ (replay_buffer.py:21, :89) */
/* read back transitions by LOGICAL index (uniform: j-th oldest, deque order; PER: list position). */
int sacb_read_transitions(sacb_handle h, int agent, const int64_t *idx, int64_t n, float *s, float *a,
                          float *r, float *s2, float *done);
int sacb_clear_replay(sacb_handle h, int agent);

/* Host-side helper of that draw, no device work: random.sample(range(n), k) on CPython's set path is "the first k distinct values
 * below n of the Mersenne-Twister word stream, each word shifted right by 32 - n.bit_length()".  The shim fetches words from the
 * global `random` stream (exactly as many as picks are missing, so the stream never runs ahead) and hands them here: picks[0..n_have)
 * are the picks so far, the accepted values of words[0..n_words) are appended in stream order; returns the new count (<= k). */
int64_t sacb_host_first_distinct(const uint32_t *words, int64_t n_words, uint64_t n, int shift, int64_t *picks, int64_t n_have, int64_t k);
/* ReplayBuffer.sample (replay_buffer.py:13-19): gather rows idx[0..B) (logical indices drawn by the caller,
 * e.g. random.sample(range(len), B) -- identical picks and RNG consumption to random.sample(deque, B)). */
int sacb_sample_uniform(sacb_handle h, int agent, const int64_t *idx, int64_t B, float *s, float *a, float *r,
                        float *s2, float *done);

/* PrioritizedReplayBuffer.sample (replay_buffer.py:48-82) of one agent.  u = B float64 uniforms (what
 * np.random.random_sample(B) returns inside np.random.choice); NULL => drawn on device (splitmix64 of the key, the frame counter and
 * the row; agent a's key is cfg.seed for a = 0 and cfg.seed ^ splitmix64(a) otherwise, splitmix64(x) = the finaliser of x + 0x9E3779B97F4A7C15).
 * Outputs may be NULL to leave results on the device for sacb_update(..., SACB_USE_LAST_SAMPLE).
 * Every sacb_per_* entry point below takes agent in [0, n_agents) (SACB_ERR_ARG otherwise). */
int sacb_per_sample(sacb_handle h, int agent, const double *u, int64_t B, int64_t *idx_out, float *weights_out,
                    float *s, float *a, float *r, float *s2, float *done);
/* The same sample for EVERY agent of the handle in one chain of three launches: u_or_null [n_agents][B] (NULL: each agent draws from
 * its own key on the device), idx_out / weights_out [n_agents][B] or NULL.  Every agent's buffer must hold at least B transitions
 * (SACB_ERR_STATE otherwise), so each minibatch has B rows.  The minibatches stay on the device for sacb_update(SACB_USE_LAST_SAMPLE). */
int sacb_per_sample_all(sacb_handle h, const double *u_or_null, int64_t B, int64_t *idx_out_or_null, float *weights_out_or_null);
/* PrioritizedReplayBuffer.update_priorities (replay_buffer.py:84-87): sequential semantics, last duplicate wins. */
int sacb_per_update(sacb_handle h, int agent, const int64_t *idx, const float *prio, int64_t B);
/* same with prio already = float32(priority + 1e-6) computed by the caller in float64 (float64 inputs) */
int sacb_per_update_final(sacb_handle h, int agent, const int64_t *idx, const float *prio_final, int64_t B);
/* fused path: priorities <- |q1 - y| of the last update (extension, SURVEY H10), indices of the last sample */
int sacb_per_update_from_td(sacb_handle h, int agent, int64_t B);
/* throughput form of the trainer's learner step over the prioritized buffer (single-agent handles; SACB_ERR_ARG on a population) (trainer.py:202-205 with PER), everything resident
 * in HBM: update on the minibatch the previous call sampled -> priorities <- |q1 - y| -> sample (device uniforms) for the next
 * call.  The write-back and the next sample run on a second stream under the tail of the update (from the actor-loss stage on), overlapping the rest of
 * the update; values are identical to sacb_per_sample / sacb_update(SACB_USE_LAST_SAMPLE) / sacb_per_update_from_td in sequence.
 * A transition pushed between two calls can first be drawn by the call after the next one. */
int sacb_per_step(sacb_handle h, int64_t B, float *losses_out_or_null, uint32_t flags);
/* test hooks: read / overwrite the priority table and the p**alpha table (float32 pow is libm dependent). */
int sacb_per_get_priorities(sacb_handle h, int agent, float *prio, int64_t n);
int sacb_per_set_priorities(sacb_handle h, int agent, const float *prio, const float *p_alpha_or_null, int64_t n);
typedef struct { int64_t frame, pos, len, n_fine, n_flagged, n_exact_fallbacks; float total_f32; double cdf_last; } sacb_per_stats;
int sacb_per_get_stats(sacb_handle h, int agent, sacb_per_stats *out);
int sacb_per_set_frame(sacb_handle h, int agent, int64_t frame);

/* ---- SAC.update_parameters (sac_imp.py:74-144) --------------------------------------------------------- */
enum {
    SACB_USE_LAST_SAMPLE = 1,  /* minibatch = rows chosen by the last sacb_per_sample / sacb_stage_indices */
    SACB_NO_LOSS_READBACK = 2, /* do not sync / copy the three loss scalars (throughput mode)                 */
    SACB_EXPORT_GRADS = 4,     /* keep the critic/policy gradients in the SACB_SLOT_GRAD arena (tests)        */
    SACB_DEVICE_INDICES = 8,   /* uniform ring: the B positions are drawn on the device inside the gather stage (keyed bijection of
                                  [0, len): B distinct positions = sampling without replacement, replay_buffer.py:15); idx = NULL.
                                  Nothing of the step touches the host: population mode, K updates per call (sacb_update_steps) */
    SACB_WRITE_BACK_TD = 16    /* prioritized buffer, with SACB_USE_LAST_SAMPLE: priorities of the minibatch <- |q1 - y| + 1e-6
                                  (update_priorities, replay_buffer.py:84-87; = sacb_per_update_from_td) enqueued behind the loss copy:
                                  the call returns when the losses have arrived, the write-back runs while the caller is back in Python.
                                  A population writes back every agent's minibatch into its own table in one launch */
};
/* idx: B logical indices (NULL => SACB_USE_LAST_SAMPLE, or the next index set pre-staged with sacb_stage_indices; otherwise SACB_ERR_ARG);
 * eps_next / eps_cur: [B, act] N(0,1) draws of the two policy.sample calls (sac_imp.py:89, :116), NULL => Philox;
 * losses_out[3] = q1_loss, q2_loss, policy_loss (sac_imp.py:140-144). */
int sacb_update(sacb_handle h, int64_t B, const int64_t *idx, const float *eps_next, const float *eps_cur,
                float *losses_out, uint32_t flags);
/* K learner steps per call with nothing of a step on the host (trainer.py:190-205 batched; SURVEY 8f rank 3): prioritized ring =
 * K x the sacb_per_step pipeline (single-agent handles), uniform ring = K updates with SACB_DEVICE_INDICES; eps drawn on the device; then ONE read-back:
 * losses_out[K][3] (NULL or SACB_NO_LOSS_READBACK: none).  K <= 64.  Bitwise equal to K single calls. */
int sacb_update_steps(sacb_handle h, int64_t B, int K, float *losses_out, uint32_t flags);
/* update on a caller-supplied minibatch (no replay involved): test / bench entry. */
int sacb_update_batch(sacb_handle h, int64_t B, const float *s, const float *a, const float *r, const float *s2,
                      const float *done, const float *is_weights_or_null, const float *eps_next,
                      const float *eps_cur, float *losses_out, float *td_abs_out_or_null, uint32_t flags);
/* pre-stage indices for the next n_steps updates on the device (bench "inputs resident in HBM"). */
int sacb_stage_indices(sacb_handle h, const int64_t *idx, int64_t B, int64_t n_steps);
int sacb_get_losses(sacb_handle h, int agent, float *losses_out);
/* population: losses_out[n_agents][3] of the last update of every agent, one strided device->host copy */
int sacb_get_losses_all(sacb_handle h, float *losses_out);

/* ---- SAC.select_action (sac_imp.py:54-72) -------------------------------------------------------------- */
int sacb_select_action(sacb_handle h, int agent, const float *obs, int evaluate, const float *eps_or_null,
                       float *action_out);
/* population form (SURVEY 8f rank 1): obs [n_agents, obs_dim] -> action_out [n_agents, act_dim], agent i acts on row i with its
 * own policy; eps_or_null [n_agents, act_dim].  One chain of launches for the whole population. */
int sacb_select_action_batch(sacb_handle h, const float *obs, int evaluate, const float *eps_or_null, float *action_out);

/* ---- networks as callables (QNetwork.forward, GaussianPolicy.forward / .sample) on n rows -------------- */
int sacb_q_forward(sacb_handle h, int agent, int net, const float *s, const float *a, int64_t n, float *q_out);
int sacb_policy_forward(sacb_handle h, int agent, const float *s, int64_t n, float *mean_out, float *log_std_out);
/* GaussianPolicy.sample (networks_model1.py:78-99 == networks_model2.py:99-120) on n rows: reparameterised draw, tanh squash, scale /
 * bias, log-prob summed over the action components.  eps_or_null [n, act] = the N(0,1) draws of Normal.rsample; NULL => Philox. */
int sacb_policy_sample(sacb_handle h, int agent, const float *s, int64_t n, const float *eps_or_null, float *action_out,
                       float *log_prob_out);

/* ---- data-parallel mode (BASELINE.json configs[3]): gradients are exported, all-reduced by the host over
 * NCCL (torch.distributed), then applied.  phase 0 = critics (sac_imp.py:101-113), 1 = actor+alpha (:116-135). */
/* phase 0 takes this rank's minibatch: idx = B_local logical replay indices (NULL: indices staged earlier), eps_next /
 * eps_cur = [B_local, act] draws (NULL: Philox on device, give every rank its own sacb_config.seed); phase 1 reuses them. */
int sacb_dp_backward(sacb_handle h, int phase, int64_t B_local, const int64_t *idx, const float *eps_next, const float *eps_cur);
int sacb_dp_apply(sacb_handle h, int phase);
int sacb_dp_grad_buffer(sacb_handle h, int phase, void **dev_ptr, int64_t *n_floats);
/* Fused exchange over NVLink peer memory (one node, 1..8 replicas, one process per GPU): sacb_dp_ipc_handle gives the 64-byte CUDA IPC
 * handle of this replica's arena; after the host has gathered all of them (any transport: torch.distributed.all_gather_object),
 * sacb_dp_connect maps the peers' arenas.  sacb_dp_exchange_apply(phase) then replaces "all-reduce + sacb_dp_apply": a flag barrier
 * in peer memory, and ONE kernel that reads the W gradient slabs (own HBM + peers over NVLink), sums them in rank order and applies
 * Adam + Polyak -- the reduced gradient never touches memory; the log_alpha gradient and the loss scalars are averaged the same way
 * (sacb_dp_get_losses).  Without sacb_dp_connect (or world = 1) it is the plain vectorised apply. */
int sacb_dp_ipc_handle(sacb_handle h, void *handle_out_64_bytes);
int sacb_dp_connect(sacb_handle h, int rank, int world, const void *handles_world_x_64_bytes);
int sacb_dp_exchange_apply(sacb_handle h, int phase);
int sacb_dp_get_losses(sacb_handle h, float *losses_out);
/* the handle's private CUDA stream (a cudaStream_t): lets the host enqueue its collective between sacb_dp_backward and
 * sacb_dp_apply on the SAME stream (torch.cuda.ExternalStream), so a data-parallel step needs no host synchronisation. */
int sacb_get_stream(sacb_handle h, void **stream_out);

/* ---- instrumentation ---------------------------------------------------------------------------------- */
typedef struct {
    int64_t kernel_launches;   /* kernels of this library launched since create (graph nodes counted per replay) */
    int32_t n_stages, n_tasks, n_tiles;    /* of the current update program */
    int32_t grid, block, smem_bytes, sm_count;
    int32_t n_programs;        /* update programs built since create (one per batch size / mode; never per hyperparameter value) */
} sacb_stats;
int sacb_get_stats(sacb_handle h, sacb_stats *out);
/* CUDA-event stopwatch on the handle's stream (torch.cuda.Event only sees torch's stream). */
int sacb_timer_start(sacb_handle h);
int sacb_timer_stop(sacb_handle h, float *ms_out);
/* time `iters` replays of the update step with CUDA events on the handle's stream; returns ms per step. */
int sacb_time_update(sacb_handle h, int64_t B, int iters, float *ms_per_step);
/* device time of every stage kernel of one step (STAGED mode), in microseconds; n = min(cap, n_stages). */
int sacb_time_stages(sacb_handle h, int64_t B, float *us_out, int cap);
/* test hook: a hidden activation matrix [B, hidden] of the LAST update (bf16 pair reconstructed to float32).
 * group 0: policy layer `layer` on the current states (sac_imp.py:116) ; 1: critic k (0 = q1, 1 = q2) on (s, a) (:101-102) ;
 * 2: updated critic k on (s, a_new) (:117-118) ; 3: target critic k on (s2, a2) (:92-93).  The parity tests use the signs
 * (ReLU masks) to make the comparison with the oracle independent of pre-activations that round to either side of zero. */
int sacb_debug_read_activation(sacb_handle h, int agent, int group, int k, int layer, int64_t B, float *out);
/* test hook: physical ring slots of the minibatch rows of the LAST update (host-staged, pre-staged or device-drawn) */
int sacb_debug_read_slots(sacb_handle h, int agent, int32_t *slots_out, int64_t B);
/* standalone GEMM self-test of the TMA + tcgen05 tile against the FFMA tile and a host float64 product of the same
 * bf16-pair operands; returns max |diff| / max |ref|.  b_r0 = row/column offset of the B operand inside its matrix. */
int sacb_selftest_gemm(int device, int M, int N, int K, int a_mn_major, int b_mn_major, int b_r0, float *rel_err_out);
/* same with an explicit tensor-core tile shape: bm = 64 | 128 rows, bn = 32 | 64 columns (32 only with a K-major B operand) */
int sacb_selftest_gemm_tile(int device, int M, int N, int K, int a_mn_major, int b_mn_major, int b_r0, int bm, int bn, float *rel_err_out);

/* same for the throughput ("stream") form of a GEMM stage: 128 x bn (64 | 128) tiles walked by `ctas` resident CTAs with decoupled
 * TMA / tcgen05 / epilogue roles and two TMEM accumulators (csrc/stream.cuh) */
int sacb_selftest_gemm_stream(int device, int M, int N, int K, int a_mn_major, int b_mn_major, int b_r0, int bn, int ctas, float *rel_err_out);

#ifdef __cplusplus
}
#endif
#endif /* SACB200_H */
