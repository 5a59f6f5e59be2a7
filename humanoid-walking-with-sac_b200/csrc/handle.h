// Host-side handle, memory layout of the arena / workspace / replay ring, error plumbing.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/sacb200.h"
#include "common.cuh"

namespace sacb {

void set_error(const std::string &msg);
int fail(int code, const std::string &msg);

#define SACB_CUDA(call)                                                                              \
    do {                                                                                             \
        cudaError_t _e = (call);                                                                     \
        if (_e != cudaSuccess)                                                                       \
            return ::sacb::fail(SACB_ERR_DEVICE, std::string(#call) + ": " + cudaGetErrorString(_e)); \
    } while (0)

inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

// ---- one network inside the arena ----------------------------------------------------------------------------
// API tensor order = Module.parameters() order (fc1.weight, fc1.bias, ..., see sacb200.h).  Policy heads are
// stored fused: head.w [2A,H] = mean.weight rows then log_std.weight rows, head.b [2A] likewise.
struct NetLayout {
    int n_hidden = 0, in_dim = 0, hidden = 0, out_dim = 0;   // out_dim: 1 (Q) or 2A (policy head)
    bool is_policy = false;
    int64_t w[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0};         // hidden layer l (0-based) weight [H,in_l] / bias [H]
    int64_t w_out = 0, b_out = 0;                             // output layer / fused heads
    bool layer_norm = false;                                  // opt-in: LayerNorm (affine) between hidden Linear l and its ReLU
    int64_t g[4] = {0, 0, 0, 0}, be[4] = {0, 0, 0, 0};         // its weight (gamma) / bias (beta) [H]
    int64_t size = 0;                                         // floats, multiple of 32
    // bf16 hi/lo shadow PMs of the GEMM weights (offsets in floats inside the net's shadow block):
    // hidden layer l: [hidden, sh_ld[l]] ; policy heads: [2A, hidden] (Q output layers are read as fp32 vectors)
    // critics additionally keep the action block fc1.weight[:, obs:] as its own PM [hidden, sh_act_ld] (TMA boxes must
    // start 16 B aligned along the contiguous dimension, column `obs` of the full shadow generally does not)
    int64_t sh_w[4] = {0, 0, 0, 0}, sh_out = 0, sh_act = 0, sh_size = 0;
    int sh_ld[4] = {0, 0, 0, 0}, sh_act_ld = 0;
    int in_of(int l) const { return l == 0 ? in_dim : hidden; }
    int per_layer() const { return layer_norm ? 4 : 2; }      // API tensors per hidden layer: weight, bias (, ln.weight, ln.bias)
    int n_tensors() const { return per_layer() * n_hidden + (is_policy ? 4 : 2); }
    // API tensor -> (offset in net, rows, cols)
    void tensor(int t, int64_t &off, int64_t &rows, int64_t &cols) const;
};

struct Layout {
    int obs = 0, act = 0, hidden = 0, n_hidden = 0, maxB = 0;
    int ldx = 0, ldg = 0;           // row strides (bf16 elements, multiples of 8) of the X and g_head PMs
    NetLayout pol, q;
    // arena (per agent): scalars | params pol,q1,q2,q1t,q2t | m pol,q1,q2 | v pol,q1,q2 | grad pol,q1,q2 | shadows x5
    int64_t scalars = 0;
    int64_t loss_hist = 0;          // [kLossHist][4] losses of the last updates (T_FINISH), see sacb_update_steps
    int64_t param[5] = {0, 0, 0, 0, 0};
    int64_t shadow[5] = {0, 0, 0, 0, 0};
    int64_t adam_m[3] = {0, 0, 0}, adam_v[3] = {0, 0, 0}, grad[3] = {0, 0, 0};
    int64_t grad_scalars = 0;       // exported log_alpha gradient
    int64_t dp_flags = 0;           // [kDpMaxWorld] uint32 epoch flags written by the data-parallel peers (dp.cu)
    int64_t arena_size = 0;
    // workspace (per agent)
    // fp32 vectors / small matrices
    int64_t r = 0, d = 0, isw = 0, y = 0, td = 0, dq[2] = {0, 0}, logp = 0, eps = 0;
    int64_t head_raw = 0, da[2] = {0, 0}, loss_part = 0, aloss_part = 0;
    // pair matrices (float offsets of the hi plane; the lo plane follows the whole hi plane, sized for maxB rows)
    int64_t X = 0, g_head = 0;                                           // [3*maxB, ldx], [maxB, ldg]
    int64_t hp[4] = {0, 0, 0, 0}, dhp[4] = {0, 0, 0, 0};                 // policy activations [2*maxB,H] / grads [maxB,H]
    int64_t ht[2][4], hc[2][4], ha[2][4], dhc[2][4], dha[2][4];          // [maxB,H]
    // LayerNorm variant only (else unused): pre-normalisation outputs z (fp32), row statistics (mean, rstd), dz PMs (the dh PMs then
    // hold dpre = gradient at the LayerNorm output), PMs of dpre * xhat (column sums = dgamma)
    bool layer_norm = false;
    int64_t zp[4], zt[2][4], zc[2][4], za[2][4];                         // [2*maxB,H] / [maxB,H] fp32
    int64_t sp[4], st[2][4], sc[2][4], sa[2][4];                         // [rows][2] fp32
    int64_t dzp[4], dzc[2][4], dza[2][4], ggp[4], ggc[2][4];             // PMs [maxB,H]
    int64_t ws_size = 0;
    void build(int obs, int act, int hidden, int n_hidden, int maxB, bool layer_norm = false);
};

struct ProgramKey {
    int B, with_gather, export_grads, device_eps, use_isw, dp_phase;
    // 1: the bf16 pair shadows of all five nets are current (the Adam / Polyak epilogues of the previous update refreshed them in
    // place and nobody wrote the fp32 weights since): the program has no shadow tasks.  0: stage 0 re-derives every shadow.
    int resident = 0;
    bool operator<(const ProgramKey &o) const {
        return std::tie(B, with_gather, export_grads, device_eps, use_isw, dp_phase, resident) <
               std::tie(o.B, o.with_gather, o.export_grads, o.device_eps, o.use_isw, o.dp_phase, o.resident);
    }
};

// One kernel launch of a staged program: one stage, or the stages [s0, s1) of a chain (Stage::chain_map) as `grid` CTAs in thread-block
// clusters of `cluster` CTAs, run by kernel variant `kind`
struct StageLaunch { int s0, s1, cluster, grid, kind; };

struct ProgramInst {
    std::vector<Task> tasks;
    std::vector<Stage> stages;
    std::vector<StageLaunch> launches;   // staged mode: the launches of one step, in order
    std::vector<int> stage_has_gemm;
    std::vector<int> stage_stream;       // 1: the stage holds only GEMM tasks and runs on the stream kernel (throughput programs, stream.cuh)
    std::vector<int> stage_kind;         // kernel variant (SACB_KERNEL_VARIANTS) that runs the stage in staged mode
    Task *d_tasks = nullptr;
    Stage *d_stages = nullptr;
    Program prog{};
    cudaGraphExec_t graph = nullptr;
    // the same step as two graphs split in front of the actor-loss stage (the TD errors exist since the critic-loss stage):
    // sacb_per_step runs the priority write-back and the next prioritized sample on a second stream under the tail of the update
    cudaGraphExec_t graph_part[2] = {nullptr, nullptr};
    int split = -1;                      // index into `launches`
    bool parts_built = false;
    // the whole pipelined learner step (sacb_per_step) as ONE graph: update stages on the main stream, priority write-back and the next
    // sample forked onto the second stream in front of stage `split`, joined at the end (valid for one buffer length / batch size)
    cudaGraphExec_t step_graph = nullptr;
    int64_t step_graph_n = -1, step_graph_k = -1;
    bool step_graph_failed = false;
    int step_graph_launches = 0;
    bool step_graph_fused = false;       // which form of the sampler the capture recorded (sacb_handle_s::per_fused)
    int n_tiles_total = 0, max_stage_tiles = 0;
    int kernels_per_step = 0;
};

}  // namespace sacb

struct sacb_handle_s {
    sacb_config cfg;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    bool per_fused = false;              // the last prioritized sample ran chunk pass + search as one launch (where its flagged count is kept)
    cudaStream_t stream2 = nullptr;      // prioritized replay work that overlaps the update (sacb_per_step)
    cudaEvent_t ev_td = nullptr, ev_sampled = nullptr;
    int64_t sample_k = 0;                // rows of the minibatch the last prioritized sample left on the device (0: none)
    sacb::Layout L;
    float *arena = nullptr, *ws = nullptr;
    unsigned int *barrier = nullptr;
    int32_t *error_flag = nullptr;
    int32_t *slots = nullptr;            // [n_agents, maxB] physical ring slots of the current minibatch
    float2 *adam_table = nullptr;        // [kAdamTable] Adam bias-correction factors per step count (host float64, lr of this handle)
    int32_t *slots_identity = nullptr;   // 0..maxB-1: "gather" straight from the upload staging rows (sacb_update_batch)
    int32_t *slots_staged = nullptr;     // pre-staged index sets (sacb_stage_indices)
    int64_t staged_steps = 0, staged_next = 0, staged_B = 0;
    std::map<sacb::ProgramKey, sacb::ProgramInst> programs;
    int64_t kernel_launches = 0;
    bool shadows_valid = false;          // see ProgramKey::resident; cleared by every write of fp32 weights from outside the update program
    int use_pdl = 1;                     // staged mode: programmatic dependent launch between the stage kernels (SACB_NO_PDL=1 disables)
    // data-parallel exchange over peer memory (dp.cu): rank / world of this replica, the peers' arenas (cudaIpcOpenMemHandle; own = arena)
    int dp_rank = 0, dp_world = 1;
    float *dp_peer_arena[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    uint32_t dp_epoch = 0;
    int dp_device_eps = 1;               // data-parallel mode: eps of the current step drawn on device (phase 1 follows phase 0)
    int coop_blocks_per_sm = 0;
    std::map<std::pair<int, int>, int> max_active_clusters;   // (kernel variant, cluster size) -> cudaOccupancyMaxActiveClusters
    // ---- replay (replay.cu) ----
    float *ring = nullptr;
    int64_t ring_row = 0;                // floats per transition: [s | s2 | a | r | d] padded to 4
    std::vector<int64_t> r_len, r_pos, r_head;   // per agent: count, next write slot, slot of the oldest entry
    int64_t *ring_meta = nullptr;        // device [n_agents][2] = (r_len, r_head) for on-device index draws; re-uploaded when a push changed it
    bool ring_meta_dirty = true;
    float *stage_rows = nullptr;         // device staging for pushes
    int64_t stage_rows_cap = 0;
    int32_t *gather_slots = nullptr;     // [stage_rows_cap] slots of a host-facing gather (sacb_read_transitions)
    // PER
    float *prio = nullptr, *p_alpha = nullptr;   // [n_agents, capacity]
    std::vector<int64_t> per_frame;
    bool per_frame_dirty = true;         // the device copy of per_frame[0] (read and advanced by the sample kernels) has to be uploaded
    void *per_ws = nullptr;                      // scan workspace (see replay.cu)
    int64_t *last_idx_dev = nullptr;             // [n_agents, maxB] logical indices of the last sample
    float *last_w_dev = nullptr;
    sacb_per_stats per_stats{};
    bool prio_max_valid = false;                 // per-CTA maxima of the priority table are current (replay.cu: per_refresh_max)
    // pinned host staging
    float *pin = nullptr;
    int64_t pin_floats = 0;
    float *pin_rows = nullptr;           // packed minibatch rows of sacb_update_batch
    float *pin_hist = nullptr;           // [32 + 4 * kLossHist] scalar block + loss history of agent 0 (sacb_update_steps: ONE read-back for K updates)
    float *pin_small = nullptr;          // [16] losses + error flag read back with ONE synchronisation (finish_update)
    cudaEvent_t ev_loss = nullptr;       // behind the loss copy: what the host waits for when more work (the |TD| write-back) is enqueued after it
    float *pin_push = nullptr;           // staging of small pushes (<= kPinPushRows rows): no synchronisation on the push path
    cudaEvent_t ev_push = nullptr;       // the H2D copy out of pin_push has completed
    bool push_in_flight = false;
    cudaEvent_t ev_slots = nullptr;      // the H2D copy of the minibatch slots out of `pin` has completed
    bool slots_in_flight = false;
    double *pin_u = nullptr;             // pinned block for the host-drawn PER uniforms
    cudaEvent_t ev_u = nullptr;
    bool u_in_flight = false;
    float *act_ws = nullptr, *pin_act = nullptr;   // select_action scratch (device) and pinned obs / eps / action block
    int act_rows = 0;
    uint32_t act_counter = 0;            // Philox counter of select_action's exploration draws (checkpointed through sacb_scalars)
    int64_t pin_rows_cap = 0;
};

namespace sacb {
constexpr int kPinPushRows = 64;
inline bool math_is_tc(int m) { return m != SACB_MATH_FP32; }
inline size_t math_smem(int m) { return math_is_tc(m) ? (size_t)kTcSmemBytes : (size_t)kSimtSmemBytes; }
// TMA descriptor of a pair-matrix view (program.cu): dims {cols, rows, 2 planes, n_agents}, box {64, box_rows, 2, 1},
// bf16, SWIZZLE_128B.  base = device pointer of the view's first hi element for agent 0.
int make_pm_tensor_map(CUtensorMap *out, const void *base, int64_t cols, int64_t rows, int64_t ld, int64_t plane_elems,
                       int64_t agent_stride_bytes, int n_agents, int box_rows);
const void *update_kernel_for(int math_mode, int variant);      // variant: index into SACB_KERNEL_VARIANTS (0 = everything)
bool variant_has_gemm(int variant);
bool variant_can_chain(int variant);      // the build carries the chained launch form
int variant_blocks_per_sm(int variant);      // resident CTAs per SM a build is compiled for (light column-sum builds: 2)
int pick_variant(uint32_t task_types, uint32_t epilogues, bool allow_light_colsum = true);
// program.cu
int get_program(sacb_handle h, const ProgramKey &key, ProgramInst **out);
int launch_program(sacb_handle h, ProgramInst &p);
int launch_program_part(sacb_handle h, ProgramInst &p, int part);
int launch_per_step_graph(sacb_handle h, ProgramInst &p, int64_t B, int64_t k);      // SACB_OK, an error, or 1: not available (caller falls back)   // 0: up to and including the critic-loss stage, 1: the rest
void free_programs(sacb_handle h);
int check_error_flag(sacb_handle h);
// the key of the program that serves the next update of this handle (fills ProgramKey::resident), and the bookkeeping behind its launch
ProgramKey update_key(sacb_handle h, int B, int with_gather, int export_grads, int device_eps, int use_isw);
void after_update_launch(sacb_handle h, const ProgramKey &key);
// replay.cu
int replay_create(sacb_handle h);
void replay_destroy(sacb_handle h);
int per_sample_launch(sacb_handle h, cudaStream_t st, const double *u, int64_t B, int64_t *k_out);   // kernels of one sample() call
int upload_ring_meta(sacb_handle h);                                                                   // (len, head) of every agent's ring -> device, if a push changed them
int per_writeback_launch(sacb_handle h, cudaStream_t st, int64_t B, bool pdl_ok = true);                                 // priorities <- |td| of the last update
}  // namespace sacb
