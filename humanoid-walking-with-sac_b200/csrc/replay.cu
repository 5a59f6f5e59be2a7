// HBM-resident replay: uniform ring (deque semantics) and prioritized buffer.
//
// Reference: replay_buffer.py:5-22 (ReplayBuffer) and :25-90 (PrioritizedReplayBuffer).
// Ring row = one transition [s (obs) | s2 (obs) | a (act) | r | d], fp32, padded to 16 B: a sampled row is one
// contiguous ~2.9 KB read (Humanoid), gathered by one warp with coalesced loads.
//
// PER sampling reproduces np.random.choice(len, B, p=probs) bit-for-bit downstream of the p**alpha table, in three launches per
// sample() call chained with programmatic dependent launch.  Up to 2 096 128 rows (the chunk prefixes fit into shared memory) there are
// no serial tails between them:
//   per_sum           CTA subtrees of numpy's pairwise-summation tree over p_alpha (float32, the exact same association)
//   per_chunk_notail  every CTA adds the top of that tree itself (<= 512 values) -> total; probs = p_alpha / total (float32), float64 chunk
//                     sums, count of "fine" elements
//   per_search_scan   every CTA scans the chunk sums itself (shared memory), per-sample inverse-CDF search + provable ambiguity test
//                     (see DESIGN.md "PER exactness"); the last group then runs the sequential float64 cumsum (numpy's own order) for
//                     samples the test could not certify, IS weights (N p)^-beta / max, logical indices, ring slots for the update's gather
// Above that the last CTA to arrive finishes the sum and the scan: per_sum(tail) -> per_chunk -> per_search, with the chunk prefixes
// in global memory.  Both forms are bit-identical.
// Populations (n_agents > 1, capacity <= 2 096 128 per agent): the tail-free chain takes an agent grid dimension (blockIdx.y), so ONE
// chain of three launches samples every agent's table (PerAgents below).
#include <cmath>
#include <cstring>
#include <algorithm>
#include <vector>

#include "handle.h"

namespace sacb {

// Programmatic dependent launch for the chain of small dependent kernels of one sample() call: every kernel first waits for
// its predecessor's results, then lets its successor become resident, so launch latencies overlap instead of adding up.
#define SACB_PDL_ENTER()                                                  \
    do {                                                                  \
        asm volatile("griddepcontrol.wait;" ::: "memory");                \
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   \
    } while (0)

constexpr int kChunk = 1024;          // elements per scan chunk (one warp, 32 per lane)
constexpr int kSumLeafMax = 128;      // numpy PW_BLOCKSIZE
constexpr int kSumBlockMax = 4096;    // elements of one CTA subtree in per_sum
constexpr int kSumHeap = 256;         // heap slots per CTA subtree (depth <= 7)
constexpr int kCarrySmem = 2048;      // chunk prefixes staged in shared memory by per_search when they fit (capacity <= 2 M)

struct PerWs {            // device workspace of one agent's PER sampler
    float *block_vals;    // heap of the top-level summation tree
    float *total;         // [1]
    double *chunk_sum;    // [n_chunks]
    double *chunk_carry;  // [n_chunks + 1] exclusive, last = cdf_last
    int *chunk_fine;      // [n_chunks]
    int *counters;        // [0] total fine, [1] flagged count (running), [2] exact fallbacks run, [3] flagged count of the last call
    int *tickets;         // completion tickets of the three sample() kernels (kTicketInts each)
    float *block_max;     // [128] per-CTA maxima of the priority table (push reads max(priorities), replay_buffer.py:38)
    double *cdf_exact;    // [n_chunks + 1] exact sequential cdf at the chunk starts, only touched by the exact pass (sized for capacity)
    double *u;            // [maxB]
    int *flagged;         // [maxB]
    int64_t *idx;         // [maxB]
    float *weights;       // [maxB]
};

// ---------------------------------------------------------------------------------------------------------------
// numpy pairwise sum tree: node (start,n) -> children (start,n2) , (start+n2, n-n2) with n2 = n/2 - (n/2)%8
// heap id 1 = root; path bits from the top give left(0)/right(1).  returns false if an ancestor was already a leaf.
// ---------------------------------------------------------------------------------------------------------------
__host__ __device__ inline bool pw_node(int64_t root_start, int64_t root_n, int limit, unsigned id, int64_t &start, int64_t &n, bool &is_leaf) {
    start = root_start; n = root_n;
#ifdef __CUDA_ARCH__
    const int depth = 31 - __clz((int)id);
#else
    const int depth = 31 - __builtin_clz(id);
#endif
    for (int b = depth - 1; b >= 0; b--) {
        if (n <= limit) return false;
        int64_t n2 = n / 2; n2 -= n2 % 8;
        if ((id >> b) & 1) { start += n2; n -= n2; } else { n = n2; }
    }
    is_leaf = n <= limit;
    return true;
}

// one numpy leaf (n <= 128) by 8 lanes (a quarter warp): lane k owns accumulator r[k] = a[k] + a[k+8] + a[k+16] + ... in that
// order; all of its <= 16 loads are issued before the first add.  Result valid in lane 0 of the group.
__device__ __forceinline__ float pw_leaf8(const float *a, int n, int k /* lane inside the 8-lane group */) {
    const unsigned lane = threadIdx.x & 31u, gmask = 0xffu << (lane & 24u);
    float res = 0.f;
    if (n < 8) {
        if (k == 0) for (int i = 0; i < n; i++) res = __fadd_rn(res, a[i]);
        return res;
    }
    const int full = n - (n % 8), cnt = full >> 3;      // cnt <= 16 terms per accumulator
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = i < cnt ? __ldg(a + k + 8 * i) : 0.f;
    float r = v[0];
#pragma unroll
    for (int i = 1; i < 16; i++) if (i < cnt) r = __fadd_rn(r, v[i]);
    const float r1 = __shfl_down_sync(gmask, r, 1, 8);
    const float p = __fadd_rn(r, r1);                       // k = 0,2,4,6: r0+r1, r2+r3, r4+r5, r6+r7
    const float p2 = __shfl_down_sync(gmask, p, 2, 8);
    const float q = __fadd_rn(p, p2);                       // k = 0,4: (r0+r1)+(r2+r3), (r4+r5)+(r6+r7)
    const float q4 = __shfl_down_sync(gmask, q, 4, 8);
    res = __fadd_rn(q, q4);
    if (k == 0) for (int i = full; i < n; i++) res = __fadd_rn(res, a[i]);
    return res;
}

// sum of the subtree (start,n), n <= kSumBlockMax, by one CTA (256 threads): leaves by 8-lane groups, then bottom-up heap
__device__ float pw_block_sum(const float *a, int64_t start, int n, float *s_heap, unsigned char *s_state, int *s_leaf) {
    const int tid = threadIdx.x;
    __shared__ int s_nleaf;
    if (tid == 0) s_nleaf = 0;
    __syncthreads();
    // classify heap nodes: 0 = absent, 1 = leaf, 2 = internal; leaves are queued (start offset and length packed)
    for (unsigned id = 1 + tid; id < kSumHeap; id += blockDim.x) {
        int64_t s, m; bool leaf = false;
        const bool ex = pw_node(start, n, kSumLeafMax, id, s, m, leaf);
        s_state[id] = ex ? (leaf ? 1 : 2) : 0;
        if (ex && leaf) { const int slot = atomicAdd(&s_nleaf, 1); s_leaf[3 * slot] = (int)id; s_leaf[3 * slot + 1] = (int)(s - start); s_leaf[3 * slot + 2] = (int)m; }
    }
    __syncthreads();
    const int group = tid >> 3, k = tid & 7, n_groups = blockDim.x >> 3;
    for (int i0 = 0; i0 < s_nleaf; i0 += n_groups) {      // warp-uniform trip count
        const int i = i0 + group;
        const bool on = i < s_nleaf;
        const float v = pw_leaf8(a + start + (on ? s_leaf[3 * i + 1] : 0), on ? s_leaf[3 * i + 2] : 0, k);
        if (on && k == 0) s_heap[s_leaf[3 * i]] = v;
    }
    __syncthreads();
    for (int depth = 6; depth >= 0; depth--) {      // heap ids [2^depth, 2^(depth+1))
        for (unsigned id = (1u << depth) + tid; id < (2u << depth); id += blockDim.x)
            if (s_state[id] == 2) s_heap[id] = __fadd_rn(s_heap[2 * id], s_heap[2 * id + 1]);
        __syncthreads();
    }
    return s_heap[1];
}

// The last CTA of a grid to finish (completion ticket: results, __threadfence, atomic) runs the grid's serial tail, so a
// reduction and its finishing step are ONE launch.  The ticket resets itself for the next launch.
// Two levels so that same-address atomics (which serialise in L2, ~14 ns each) stay short: CTAs take a ticket of their group
// (blockIdx % kTicketGroups, counters 128 B apart), the last CTA of a group takes one of the final counter.
constexpr int kTicketGroups = 8, kTicketStride = 32;      // ints
constexpr int kTicketInts = (kTicketGroups + 1) * kTicketStride;
__device__ __forceinline__ bool last_block_done(int *ticket, int n_blocks = -1, int block = -1) {      // default: the whole grid
    __shared__ int s_last;
    if (n_blocks < 0) { n_blocks = (int)gridDim.x; block = (int)blockIdx.x; }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const int G = min(kTicketGroups, n_blocks), g = block % G;
        const int group_size = (n_blocks - g + G - 1) / G;
        int last = 0;
        if (atomicAdd(ticket + g * kTicketStride, 1) == group_size - 1) {
            ticket[g * kTicketStride] = 0;
            __threadfence();
            if (atomicAdd(ticket + kTicketGroups * kTicketStride, 1) == G - 1) { ticket[kTicketGroups * kTicketStride] = 0; last = 1; }
        }
        s_last = last;
    }
    __syncthreads();
    if (s_last) __threadfence();
    return s_last != 0;
}

// Agent dimension of one sampler chain: blockIdx.y = agent - first.  Every per-agent table and workspace sits at a fixed stride from
// agent 0's, and the kernels receive agent 0's pointers.  meta = the (len, head) table of the rings (upload_ring_meta): each agent reads
// its own length there, the grid being sized for the longest agent.  A chain over ONE agent passes meta = null and that agent's length
// as `n`: a single-agent handle launches exactly the grids and argument values it launched before the agent dimension existed, and
// the kernels' kAgents = false instantiation (single-agent handles) compiles the agent offsets out.
struct PerAgents {
    const int64_t *meta;
    int first;
    int64_t pa_stride;      // floats between two agents' prio / p_alpha tables (capacity)
    int64_t ws_stride;      // bytes between two agents' sampler workspaces (PerWs)
    int64_t u_stride;       // bytes between two agents' uniforms (host-drawn: a pinned row of max_batch; device-drawn: ws_stride)
    int64_t batch_stride;   // entries between two agents' ring slots / last-sample indices (max_batch)
    int64_t isw_stride;     // floats between two agents' update workspaces (Layout::ws_size)
};
__device__ __forceinline__ int per_agent(const PerAgents &g) { return g.first + (int)blockIdx.y; }
template <typename T> __device__ __forceinline__ T *ws_at(T *p, const PerAgents &g, int a) { return (T *)((const char *)p + (int64_t)a * g.ws_stride); }
__device__ __forceinline__ int64_t agent_len(const PerAgents &g, int a, int64_t n) { return g.meta ? __ldcg(g.meta + 2 * a) : n; }

// depth of the top of numpy's summation tree above the CTA subtrees of <= kSumBlockMax elements
__host__ __device__ inline int top_depth_of(int64_t n) {
    int d = 0;
    while (n > kSumBlockMax) { int64_t n2 = n / 2; n2 -= n2 % 8; n = n - n2; d++; }   // the right child is the larger one
    return d;
}

// Key of agent a's device-drawn uniforms: seed ^ splitmix64(a) for a > 0 (splitmix64(x): x += 0x9E3779B97F4A7C15, then the
// finaliser of uniform_of below), the handle's seed itself for agent 0 -- agent 0 of a population draws what a one-agent handle draws.
__host__ __device__ inline uint64_t per_agent_seed(uint64_t seed, int a) {
    if (a == 0) return seed;
    uint64_t x = (uint64_t)a + 0x9E3779B97F4A7C15ull;
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
    return seed ^ x;
}

__device__ __forceinline__ double uniform_of(uint64_t seed, uint64_t counter, int j) {      // splitmix64 -> [0, 1) with 53 bits
    uint64_t x = seed ^ (counter * 0x9E3779B97F4A7C15ull + (uint64_t)j * 0xBF58476D1CE4E5B9ull);
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
    return (double)(x >> 11) * (1.0 / 9007199254740992.0);
}

// top of the summation tree (heap ids < 2^(top_depth+1) <= 4096) in shared memory: one read of the CTA results, then level by level
// in numpy's association.  Every thread of the CTA returns the float32 total.
__device__ float top_tree_sum(int64_t n, int top_depth, const float *top_vals) {
    __shared__ float s_top[4096];
    __shared__ unsigned char s_tstate[4096];
    const unsigned n_ids = 2u << top_depth;
    for (unsigned k = 1 + threadIdx.x; k < n_ids; k += blockDim.x) {
        int64_t s2, m2; bool lf = false;
        const bool ex = pw_node(0, n, kSumBlockMax, k, s2, m2, lf);
        s_tstate[k] = ex ? (lf ? 1 : 2) : 0;
        if (ex && lf) s_top[k] = __ldcg(top_vals + k);
    }
    __syncthreads();
    for (int depth = top_depth; depth >= 0; depth--) {
        for (unsigned k = (1u << depth) + threadIdx.x; k < (2u << depth); k += blockDim.x)
            if (s_tstate[k] == 2) s_top[k] = __fadd_rn(s_top[2 * k], s_top[2 * k + 1]);
        __syncthreads();
    }
    return s_top[1];
}

// grid = top heap size; CTA id+1 = heap id of the top tree (leaf threshold kSumBlockMax).  The last CTA to finish adds the
// top of the tree (numpy's association) and publishes the float32 total.  draw_B > 0: the B uniforms of this call are drawn here.
// tail = 0: no finishing step here -- the CTAs of the next kernel (per_chunk_notail) each add the top of the tree themselves (<= 512 values, the
// same function, the same association), which takes the completion ticket (two dependent atomics) and the one-CTA tail off the chain.
template <bool kAgents>
__global__ void __launch_bounds__(256) per_sum(const float *p_alpha, int64_t n, int top_depth, float *top_vals, float *total, int *ticket,
                                               double *u, int draw_B, uint64_t seed, const int64_t *frame, int tail, PerAgents g) {
    SACB_PDL_ENTER();
    __shared__ float s_heap[kSumHeap];
    __shared__ unsigned char s_state[kSumHeap];
    __shared__ int s_leaf[3 * 128];          // a CTA subtree of <= kSumBlockMax elements has at most 128 leaves
    if (kAgents) {      // CTAs beyond this agent's tree find no leaf below (pw_node)
        const int ag = per_agent(g);
        p_alpha += ag * g.pa_stride;
        top_vals = ws_at(top_vals, g, ag); total = ws_at(total, g, ag); ticket = ws_at(ticket, g, ag); u = ws_at(u, g, ag); frame = ws_at(frame, g, ag);
        if (g.meta) { n = agent_len(g, ag, n); top_depth = top_depth_of(n); }
        seed = per_agent_seed(seed, ag);
    }
    const uint64_t counter = (uint64_t)__ldcg(frame);
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < draw_B; j += gridDim.x * blockDim.x) u[j] = uniform_of(seed, counter, j);
    const unsigned id = blockIdx.x + 1;
    int64_t s, m; bool leaf = false;
    if (pw_node(0, n, kSumBlockMax, id, s, m, leaf) && leaf) {      // CTA-uniform
        const float v = pw_block_sum(p_alpha, s, (int)m, s_heap, s_state, s_leaf);
        if (threadIdx.x == 0) top_vals[id] = v;
    }
    if (!tail || !last_block_done(ticket)) return;
    const float tot = top_tree_sum(n, top_depth, top_vals);
    if (threadIdx.x == 0) *total = tot;
}

// ---------------------------------------------------------------------------------------------------------------
// chunked float64 scan
// ---------------------------------------------------------------------------------------------------------------
// "fine" = the float32 probability, as a float64, is not an integer multiple of 2^-52 (only such elements can make a float64
// partial sum below 1 inexact).  Integer test on the float32 bits: lowest set bit of (2^23 | M) * 2^(E-150) below 2^-52.
__device__ __forceinline__ bool is_fine(float q) {
    const uint32_t b = __float_as_uint(q) & 0x7fffffffu;
    if (b == 0u) return false;
    const uint32_t E = b >> 23;
    const uint32_t m = (b & 0x7fffffu) | (E ? 0x800000u : 0u);
    return (int)(E ? E : 1u) - 150 + (__ffs((int)m) - 1) < -52;
}

// the 32 consecutive probabilities probs = p_alpha / total (float32 divide: `probs /= probs.sum()`) owned by a lane; 0 beyond n
__device__ __forceinline__ void lane_probs(const float *p_alpha, int64_t base, int64_t n, float total, float (&q)[32]) {
    if (base + 32 <= n) {
        const float4 *src = reinterpret_cast<const float4 *>(p_alpha + base);      // base is a multiple of 32 floats
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = __ldg(src + j);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            q[4 * j] = __fdiv_rn(v[j].x, total); q[4 * j + 1] = __fdiv_rn(v[j].y, total);
            q[4 * j + 2] = __fdiv_rn(v[j].z, total); q[4 * j + 3] = __fdiv_rn(v[j].w, total);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 32; j++) q[j] = base + j < n ? __fdiv_rn(p_alpha[base + j], total) : 0.f;
    }
}

// lane-local pass over its 32 probabilities: the lane sum in sequential order (adding the zeros beyond n is exact), fine count
__device__ __forceinline__ double lane_pass(const float (&q)[32], int &fine) {
    double acc = 0.0;
    fine = 0;
#pragma unroll
    for (int j = 0; j < 32; j++) {
        fine += is_fine(q[j]) ? 1 : 0;
        acc = __dadd_rn(acc, (double)q[j]);
    }
    return acc;
}

__device__ __forceinline__ double warp_excl_scan(double v, int lane, double &warp_total) {
    double incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl = __dadd_rn(t, incl);
    }
    warp_total = __shfl_sync(0xffffffffu, incl, 31);
    const double ex = __shfl_up_sync(0xffffffffu, incl, 1);
    return lane == 0 ? 0.0 : ex;
}

// exclusive scan of the chunk sums by ONE CTA (blockDim.x <= 1024): 4 consecutive entries per thread, shuffle scan inside a
// warp, warp totals through shared memory, running carry between passes of 4 * blockDim.x entries.  A prefix is at most
// 32 (lane) + 5 (warp) of the chunk sum + 4 + 5 + 32 + passes additions deep (the certification bound assumes <= 128).
__device__ void carry_scan(const double *chunk_sum, const int *chunk_fine, int n_chunks, double *carry, int *counters) {
    __shared__ double s_w[32];
    __shared__ int s_wf[32];
    __shared__ double s_run;
    __shared__ int s_frun;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    if (tid == 0) { s_run = 0.0; s_frun = 0; }
    __syncthreads();
    for (int base = 0; base < n_chunks; base += 4 * blockDim.x) {
        const int i0 = base + 4 * tid;
        double v[4]; int f[4];
#pragma unroll
        for (int j = 0; j < 4; j++) { v[j] = i0 + j < n_chunks ? __ldcg(chunk_sum + i0 + j) : 0.0; f[j] = i0 + j < n_chunks ? __ldcg(chunk_fine + i0 + j) : 0; }
        double inc[4];
        inc[0] = v[0]; inc[1] = __dadd_rn(inc[0], v[1]); inc[2] = __dadd_rn(inc[1], v[2]); inc[3] = __dadd_rn(inc[2], v[3]);
        int ft = f[0] + f[1] + f[2] + f[3];
        double wt;
        const double ex = warp_excl_scan(inc[3], lane, wt);      // exclusive over the lanes' totals, wt = warp total
        int fex = ft;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, fex, o); if (lane >= o) fex += t; }
        const int fwt = __shfl_sync(0xffffffffu, fex, 31);
        fex -= ft;
        if (lane == 0) { s_w[warp] = wt; s_wf[warp] = fwt; }
        __syncthreads();
        double wpre = s_run; int fpre = s_frun;
        for (int w = 0; w < warp; w++) { wpre = __dadd_rn(wpre, s_w[w]); fpre += s_wf[w]; }
        const double pre = __dadd_rn(wpre, ex);
#pragma unroll
        for (int j = 0; j < 4; j++) if (i0 + j < n_chunks) carry[i0 + j] = j ? __dadd_rn(pre, inc[j - 1]) : pre;
        __syncthreads();
        if (tid == 0) {
            double r = s_run; int fr = s_frun;
            for (int w = 0; w < nw; w++) { r = __dadd_rn(r, s_w[w]); fr += s_wf[w]; }
            s_run = r; s_frun = fr;
        }
        __syncthreads();
    }
    if (tid == 0) { carry[n_chunks] = s_run; counters[0] = s_frun; counters[1] = 0; }
}

// one warp per chunk of 1024 probabilities: float64 chunk sum + count of "fine" elements; the last CTA scans the chunk sums
__device__ __forceinline__ void chunk_group(const float *p_alpha, int64_t n, float total, int group, double *chunk_sum, int *chunk_fine) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t chunk = (int64_t)group * 8 + warp;
    if (chunk * kChunk < n) {
        int fine;
        float q[32];
        lane_probs(p_alpha, chunk * kChunk + lane * 32, n, total, q);
        const double v = lane_pass(q, fine);
        double wt;
        warp_excl_scan(v, lane, wt);
        for (int o = 16; o > 0; o >>= 1) fine += __shfl_xor_sync(0xffffffffu, fine, o);
        if (lane == 0) { chunk_sum[chunk] = wt; chunk_fine[chunk] = fine; }
    }
}
__global__ void __launch_bounds__(256) per_chunk(const float *p_alpha, int64_t n, const float *total, double *chunk_sum, int *chunk_fine,
                                                 int n_chunks, double *carry, int *counters, int *ticket) {
    SACB_PDL_ENTER();
    chunk_group(p_alpha, n, *total, (int)blockIdx.x, chunk_sum, chunk_fine);
    if (!last_block_done(ticket)) return;
    carry_scan(chunk_sum, chunk_fine, n_chunks, carry, counters);
}

// the same pass behind per_sum(tail = 0): every CTA first adds the top of the summation tree itself (CTA 0 publishes the total); no
// completion ticket, no scan tail -- the search CTAs scan the chunk sums themselves (per_search_scan)
template <bool kAgents>
__global__ void __launch_bounds__(256) per_chunk_notail(const float *p_alpha, int64_t n, int top_depth, const float *top_vals, float *total,
                                                        double *chunk_sum, int *chunk_fine, PerAgents g) {
    SACB_PDL_ENTER();
    if (kAgents) {
        const int ag = per_agent(g);
        if (g.meta) { n = agent_len(g, ag, n); top_depth = top_depth_of(n); }
        if (blockIdx.x > 0 && (int64_t)blockIdx.x * 8 * kChunk >= n) return;      // beyond this agent's chunks (grid sized for the longest agent)
        p_alpha += ag * g.pa_stride;
        top_vals = ws_at(top_vals, g, ag); total = ws_at(total, g, ag); chunk_sum = ws_at(chunk_sum, g, ag); chunk_fine = ws_at(chunk_fine, g, ag);
    }
    const float tot = top_tree_sum(n, top_depth, top_vals);
    if (blockIdx.x == 0 && threadIdx.x == 0) *total = tot;
    chunk_group(p_alpha, n, tot, (int)blockIdx.x, chunk_sum, chunk_fine);
}

// numpy's own algorithm -- cdf = cumsum(float64(probs)) strictly left to right, cdf /= cdf[-1], searchsorted(side='right') --
// evaluated exactly for the samples the test above could not certify, by ONE warp whose lanes all track the same running sum.
// The sequential sum is not walked element by element: a chunk of 1024 probabilities is JUMPED with one addition when that is
// provably what the element-wise loop computes:
//   * the chunk holds no "fine" element (every probability is an integer multiple of 2^-52), so its parallel float64 sum is exact, and
//   * S and S + chunk_sum lie in the same binade [2^e, 2^(e+1)), e <= 0: every partial sum then is a multiple of ulp = 2^(e-52) inside
//     that binade, i.e. exactly representable -- the sequential additions never round, and their result is S + chunk_sum.
// Chunks with a fine element or a binade crossing (a few dozen at most: the running sum only grows) are added element by element
// from shared memory.  Cost ~0.2 ms instead of ~50 ms for the plain loop over 1 M elements, so the rare fallback is no cliff.
__device__ __forceinline__ int f64_exponent(double x) { return (int)((__double_as_longlong(x) >> 52) & 0x7ff); }
__device__ void exact_pass(const float *p_alpha, int64_t n, float tot, double *carry_exact, const double *chunk_sum, const int *chunk_fine, int n_chunks,
                           const double *u, int B, const int *flagged, int64_t *idx_out, int *counters, float *s_q /* [kChunk] shared */) {
    const int lane = threadIdx.x;      // warp 0 only
    auto stage_chunk = [&](int c) {    // probabilities of chunk c into shared memory (0 beyond n: adding them is exact)
        const int64_t base = (int64_t)c * kChunk;
        __syncwarp();
        for (int k = lane; k < kChunk; k += 32) s_q[k] = base + k < n ? __fdiv_rn(p_alpha[base + k], tot) : 0.f;
        __syncwarp();
    };
    // the same argument one level down: inside a chunk that has to be walked, a lane's 32 consecutive probabilities are jumped when
    // they hold no fine element and do not leave the binade; only the other groups are added element by element
    auto walk_chunk = [&](int c, double S) {
        stage_chunk(c);
        double gs = 0.0;
        int gf = 0;
#pragma unroll 8
        for (int j = 0; j < 32; j++) { const float q = s_q[lane * 32 + j]; gf |= is_fine(q) ? 1 : 0; gs = __dadd_rn(gs, (double)q); }
        for (int g = 0; g < 32; g++) {
            const double gsg = __shfl_sync(0xffffffffu, gs, g);
            const int gfg = __shfl_sync(0xffffffffu, gf, g);
            const double T = __dadd_rn(S, gsg);
            if (!gfg && S > 0.0 && f64_exponent(T) == f64_exponent(S) && f64_exponent(S) <= 1023) S = T;
            else for (int j = 0; j < 32; j++) S = __dadd_rn(S, (double)s_q[g * 32 + j]);
        }
        return S;
    };
    double S = 0.0;
    for (int c0 = 0; c0 < n_chunks; c0 += 32) {      // chunk sums fetched 32 at a time (one coalesced read, then shuffles)
        const double cs_l = c0 + lane < n_chunks ? __ldcg(chunk_sum + c0 + lane) : 0.0;
        const int cf_l = c0 + lane < n_chunks ? __ldcg(chunk_fine + c0 + lane) : 0;
        for (int j = 0; j < 32 && c0 + j < n_chunks; j++) {
            const int c = c0 + j;
            if (lane == 0) carry_exact[c] = S;      // exact sequential cdf just before chunk c
            const double cs = __shfl_sync(0xffffffffu, cs_l, j);
            const int cf = __shfl_sync(0xffffffffu, cf_l, j);
            const double T = __dadd_rn(S, cs);
            if (cf == 0 && S > 0.0 && f64_exponent(T) == f64_exponent(S) && f64_exponent(S) <= 1023) S = T;
            else S = walk_chunk(c, S);
        }
    }
    if (lane == 0) { carry_exact[n_chunks] = S; counters[2] += 1; }
    const double last = S;
    __threadfence_block();
    __syncwarp();
    for (int j = 0; j < B; j++) {
        if (!__ldcg(flagged + j)) continue;      // warp-uniform
        const double uu = u[j];
        int lo = 0, hi = n_chunks - 1;           // last chunk c whose preceding cdf value is <= u (chunk 0 always qualifies)
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (__ddiv_rn(__ldcg(carry_exact + mid), last) <= uu) lo = mid; else hi = mid - 1;
        }
        stage_chunk(lo);
        double acc = __ldcg(carry_exact + lo);
        const int64_t base = (int64_t)lo * kChunk;
        int cnt = 0;
        for (int k = 0; k < kChunk && base + k < n; k++) {
            acc = __dadd_rn(acc, (double)s_q[k]);
            if (__ddiv_rn(acc, last) <= uu) cnt++; else break;      // monotone: the first cdf value above u ends the count
        }
        const int64_t idx = base + cnt;
        if (lane == 0) idx_out[j] = idx < n ? idx : n - 1;
    }
}

// one warp per sample: inverse-CDF search + ambiguity test.  The last CTA to finish runs the serial tail of sample():
// the exact pass for flagged samples (rare), IS weights (replay_buffer.py:67-68), ring slots for the update's gather.
struct SearchArgs {
    const float *p_alpha; int64_t n; const double *u; int B; int *counters; int64_t *idx_out; int *flagged; int *ticket;
    double *carry_exact; const double *chunk_sum; const int *chunk_fine; int n_chunks;
    float *weights; int32_t *slots; float *isw_ws; int64_t *idx_copy;
    // beta = min(1, beta_start + frame * (1 - beta_start) / beta_frames) (replay_buffer.py:53) from the DEVICE copy of the frame counter, which
    // the tail then advances: a captured learner step needs no per-step argument
    int64_t *frame; double beta_start, one_minus_start, beta_frames;
};
// group sg of n_sg: 8 samples, one per warp; cr = chunk prefixes (shared or global), F = number of fine elements.  The last group to
// finish runs the serial tail.  Returns true in that group only (after the tail).
// uu_pre >= 0: this warp's uniform, fetched by the caller ahead of its prologue (host-drawn uniforms are read from pinned host memory)
__device__ __forceinline__ bool search_group(const SearchArgs &a, const double *cr, int F, float tot, int sg, int n_sg, double uu_pre = -1.0) {
    const float *p_alpha = a.p_alpha; const int64_t n = a.n; const double *u = a.u; const int B = a.B, n_chunks = a.n_chunks;
    int *counters = a.counters; int64_t *idx_out = a.idx_out; int *flagged = a.flagged;
    double *carry_exact = a.carry_exact; const double *chunk_sum = a.chunk_sum; const int *chunk_fine = a.chunk_fine;
    float *weights = a.weights; int32_t *slots = a.slots; float *isw_ws = a.isw_ws; int64_t *idx_copy = a.idx_copy;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = sg * 8 + warp;
    if (j < B) {      // warp-uniform
        const double last = cr[n_chunks];
        const double uu = uu_pre >= 0.0 ? uu_pre : u[j];
        // cdf / last <= u (an IEEE divide per probed element, like numpy's cdf /= cdf[-1]) decided without the divide unless the
        // element is within 2^-49 relative of u * last: outside that band the rounded quotient cannot land on the other side of u
        const double t = __dmul_rn(uu, last), t_lo = __dmul_rn(t, 1.0 - 1.7763568394002505e-15), t_hi = __dmul_rn(t, 1.0 + 1.7763568394002505e-15);
        auto le_u = [&](double c) { return c < t_lo ? true : (c > t_hi ? false : __ddiv_rn(c, last) <= uu); };
        // Bound on |cdf_parallel / last_parallel - cdf_sequential / last_sequential| (eps = 2^-52, F = number of "fine" elements, i.e.
        // probabilities that are not multiples of eps; all partial sums are sums of non-negative numbers below 2):
        //  * an addition of two multiples of eps is exact; an addition A + B -> R can only round if an operand is not a multiple of
        //    ulp(R), i.e. a "dirty" operand (one holding a fine element) sits in a lower binade than R.  Charge the error (<= ulp(R)/2)
        //    to one fine element of that operand.  Along the path of a fine element through either evaluation order the partial sums
        //    only grow, so it enters every binade at most once: it is charged at most once per binade, sum_r 2^(r-53) < eps in total
        //    (2 eps if the sum reaches [1, 2)).  Hence |cdf_x - exact| <= 2 F eps for x = parallel scan and <= F eps + 2 eps for numpy's
        //    sequential sum (fine additions + binade crossings), |cdf_parallel - cdf_sequential| <= E = (3 F + 2) eps;
        //  * both are divided by their own last element, which differ by <= E as well: the quotients differ by <= 2 E / last, plus one
        //    rounding (<= eps / 2) per divide.
        // The window is twice that, plus 1e-13 for the crossing-only evaluation of the nearest cdf value below.  Measured on the
        // adversarial sets (1 M elements, F = 10 126): |parallel - sequential| = 0.12 F eps.  Zero when no element is fine.
        const double window = F == 0 ? 0.0 : ((12.0 * (double)F + 8.0) * 2.220446049250313e-16) / last + 4.440892098500626e-16 + 1e-13;
        // chunk: last c with carry[c]/last <= u
        int lo = 0, hi = n_chunks - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (le_u(cr[mid])) lo = mid; else hi = mid - 1;
        }
        const int c = lo;
        int fine;
        const int64_t base = (int64_t)c * kChunk + lane * 32;
        float q[32];
        lane_probs(p_alpha, base, n, tot, q);
        const double v = lane_pass(q, fine);
        double wt;
        const double ex = warp_excl_scan(v, lane, wt);
        // running cdf inside the lane (sequential order), count the elements with cdf <= u
        const double start = __dadd_rn(cr[c], ex);
        const int64_t rem = n - base;
        const int mine = rem >= 32 ? 32 : (rem > 0 ? (int)rem : 0);      // elements of this lane that exist
        int cnt = 0;
        {
            double acc = start;
#pragma unroll
            for (int k = 0; k < 32; k++) {
                acc = __dadd_rn(acc, (double)q[k]);
                cnt += (k < mine && le_u(acc)) ? 1 : 0;
            }
        }
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        // distance from u to the nearest cdf value.  The cdf is monotone (up to rounding between lanes), so the nearest values
        // sit at the crossing: chunk elements cnt-2 .. cnt+1, plus the boundary with the previous chunk when the crossing is
        // at the chunk start.  Only those take the divide.
        double mind = 1.0;
        if (c > 0 && cnt <= 1) mind = fabs(__ddiv_rn(cr[c], last) - uu);
        for (int e = cnt - 2; e <= cnt + 1; e++) {
            if (e < 0 || (e >> 5) != lane || (e & 31) >= mine) continue;
            double acc = start;
            const int ke = e & 31;
#pragma unroll
            for (int k = 0; k < 32; k++) if (k <= ke) acc = __dadd_rn(acc, (double)q[k]);
            mind = fmin(mind, fabs(__ddiv_rn(acc, last) - uu));
        }
        for (int o = 16; o > 0; o >>= 1) mind = fmin(mind, __shfl_xor_sync(0xffffffffu, mind, o));
        if (lane == 0) {
            int64_t idx = (int64_t)c * kChunk + cnt;
            const bool flag = (F != 0 && mind <= window) || idx >= n;
            if (idx >= n) idx = n - 1;
            idx_out[j] = idx;
            flagged[j] = flag ? 1 : 0;
            if (flag) atomicAdd(counters + 1, 1);
        }
    }
    if (!last_block_done(a.ticket, n_sg, sg)) return false;
    // ---- serial tail (one CTA) ----
    if (__ldcg(counters + 1) != 0) {      // CTA-uniform
        __shared__ float s_q[kChunk];
        if (threadIdx.x < 32) exact_pass(p_alpha, n, tot, carry_exact, chunk_sum, chunk_fine, n_chunks, u, B, flagged, idx_out, counters, s_q);
        __threadfence_block();
        __syncthreads();
    }
    __shared__ float s_max[32];
    const int64_t frame = __ldcg(a.frame);
    const float neg_beta = -(float)fmin(1.0, __dadd_rn(a.beta_start, __ddiv_rn(__dmul_rn((double)frame, a.one_minus_start), a.beta_frames)));
    float m = -INFINITY;
    for (int q = threadIdx.x; q < B; q += blockDim.x) {
        const int64_t ix = __ldcg(idx_out + q);
        const float prob = __fdiv_rn(p_alpha[ix], tot);
        const float w = powf((float)n * prob, neg_beta);
        weights[q] = w;                // unnormalised for now (same thread rewrites it below)
        m = fmaxf(m, w);
        slots[q] = (int32_t)ix;
        idx_copy[q] = ix;              // indices of the last sample (update_priorities without an index argument, TD write-back)
    }
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) s_max[warp] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = threadIdx.x < (blockDim.x >> 5) ? s_max[threadIdx.x] : -INFINITY;
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (threadIdx.x == 0) s_max[0] = m;
    }
    __syncthreads();
    const float wmax = s_max[0];
    for (int q = threadIdx.x; q < B; q += blockDim.x) {
        const float wn = __fdiv_rn(weights[q], wmax);
        weights[q] = wn;
        if (isw_ws) isw_ws[q] = wn;
    }
    if (threadIdx.x == 0) *a.frame = frame + 1;      // every reader of this call's value (uniform draws, beta) is done
    return true;
}

// per_search behind per_chunk (capacity above 2 M: the chunk prefixes do not fit into shared memory and are read from global memory)
__global__ void __launch_bounds__(256) per_search(const float *total, const double *carry, SearchArgs a) {
    SACB_PDL_ENTER();
    if (!search_group(a, carry, a.counters[0], *total, (int)blockIdx.x, (int)gridDim.x)) return;
    if (threadIdx.x == 0) { a.counters[3] = a.counters[1]; a.counters[1] = 0; }      // flagged count of this call; reset for the next one
}

// per_search behind per_chunk_notail (capacity <= 2 M: the chunk prefixes fit into shared memory): every search group scans the chunk sums
// itself (1 K additions by carry_scan, the function the tail of per_chunk runs: same values) instead of reading prefixes a tail CTA wrote
template <bool kAgents>
__global__ void __launch_bounds__(256) per_search_scan(const float *total, double *carry, SearchArgs a, PerAgents g) {
    SACB_PDL_ENTER();
    if (kAgents) {      // this CTA's agent (every agent draws the same B samples: no CTA is idle)
        const int ag = per_agent(g);
        if (g.meta) { a.n = agent_len(g, ag, a.n); a.n_chunks = (int)((a.n + kChunk - 1) / kChunk); }
        a.p_alpha += ag * g.pa_stride;
        a.u = reinterpret_cast<const double *>(reinterpret_cast<const char *>(a.u) + ag * g.u_stride);
        total = ws_at(total, g, ag); carry = ws_at(carry, g, ag);
        a.counters = ws_at(a.counters, g, ag); a.idx_out = ws_at(a.idx_out, g, ag); a.flagged = ws_at(a.flagged, g, ag);
        a.ticket = ws_at(a.ticket, g, ag); a.carry_exact = ws_at(a.carry_exact, g, ag); a.chunk_sum = ws_at(a.chunk_sum, g, ag);
        a.chunk_fine = ws_at(a.chunk_fine, g, ag); a.weights = ws_at(a.weights, g, ag); a.frame = ws_at(a.frame, g, ag);
        a.slots += ag * g.batch_stride; a.idx_copy += ag * g.batch_stride;
        if (a.isw_ws) a.isw_ws += ag * g.isw_stride;
    }
    const float tot = *total;
    const int j = (int)blockIdx.x * 8 + (int)(threadIdx.x >> 5);
    const double uu_pre = j < a.B ? a.u[j] : -1.0;      // in flight during the scan
    __shared__ double s_carry[kCarrySmem];
    __shared__ int s_cnt[2];
    carry_scan(a.chunk_sum, a.chunk_fine, a.n_chunks, s_carry, s_cnt);
    __syncthreads();
    if (blockIdx.x == 0) {      // the global copies (exact pass, statistics)
        for (int i = threadIdx.x; i <= a.n_chunks; i += blockDim.x) carry[i] = s_carry[i];
        if (threadIdx.x == 0) a.counters[0] = s_cnt[0];
    }
    if (!search_group(a, s_carry, s_cnt[0], tot, (int)blockIdx.x, (int)gridDim.x, uu_pre)) return;
    if (threadIdx.x == 0) { a.counters[3] = a.counters[1]; a.counters[1] = 0; }      // flagged count of this call; reset for the next one
}

// ---------------------------------------------------------------------------------------------------------------
// priorities: update (last duplicate wins), push (max over the whole capacity array)
// ---------------------------------------------------------------------------------------------------------------
// one CTA per agent (blockIdx.x), tables / indices / |td| at the given strides from the first agent's
__global__ void __launch_bounds__(1024) per_update_kernel(float *prio, float *p_alpha, const int64_t *idx, const float *td, int B, float alpha, int is_final,
                                                          int64_t tab_stride, int64_t idx_stride, int64_t td_stride) {
    SACB_PDL_ENTER();
    prio += blockIdx.x * tab_stride; p_alpha += blockIdx.x * tab_stride; idx += blockIdx.x * idx_stride; td += blockIdx.x * td_stride;
    extern __shared__ int64_t s_idx[];
    for (int j = threadIdx.x; j < B; j += blockDim.x) s_idx[j] = idx[j];
    __syncthreads();
    for (int j = threadIdx.x; j < B; j += blockDim.x) {
        const int64_t me = s_idx[j];
        int dup = 0;      // no early exit: the loads pipeline instead of one shared-memory round trip per iteration
#pragma unroll 8
        for (int k = 0; k < B; k++) dup |= (k > j && s_idx[k] == me) ? 1 : 0;
        if (!dup) {
            const float p = is_final ? td[j] : (float)((double)td[j] + 1e-6);      // priority.item() + 1e-6, stored as float32
            prio[s_idx[j]] = p;
            p_alpha[s_idx[j]] = powf(p, alpha);
        }
    }
}

// blockIdx.y = agent: its table at x + y * x_stride, its CTA maxima at block_out + y * out_stride
__global__ void __launch_bounds__(1024) max_reduce_kernel(const float *x, int64_t n, float *block_out, int64_t x_stride, int64_t out_stride) {
    __shared__ float s[32];
    x += blockIdx.y * x_stride; block_out += blockIdx.y * out_stride;
    float m = -INFINITY;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = fmaxf(m, x[i]);
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = s[threadIdx.x];
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (threadIdx.x == 0) block_out[blockIdx.x] = m;
    }
}

// src_rows != null: the `count` transitions themselves are moved here too, straight out of the pinned staging block (host memory is
// addressable from the device): the trainer's one-transition push then costs the host one launch, no copy call
__global__ void per_push_kernel(float *prio, float *p_alpha, const float *block_max, int n_blocks, int empty, int64_t pos, int64_t count,
                                int64_t capacity, float alpha, const float4 *src_rows, float4 *ring, int row_vec4) {
    if (src_rows) {      // pos + count <= capacity: a run never crosses the end of the ring
        float4 *dst = ring + pos * row_vec4;
        for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < count * row_vec4; k += (int64_t)gridDim.x * blockDim.x) dst[k] = src_rows[k];
    }
    float m = 1.0f;                                            // `if self.buffer else 1.0`
    if (!empty) { m = block_max[0]; for (int i = 1; i < n_blocks; i++) m = fmaxf(m, block_max[i]); }
    const float pa = powf(m, alpha);
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t slot = (pos + k) % capacity;
        prio[slot] = m; p_alpha[slot] = pa;
    }
}

__global__ void pow_alpha_kernel(const float *prio, float *p_alpha, int64_t n, float alpha) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p_alpha[i] = powf(prio[i], alpha);
}

// ---------------------------------------------------------------------------------------------------------------
// ring gather to a dense staging buffer (host-facing sample / read-back)
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_rows_kernel(const float *ring, int64_t ring_row, const int32_t *slots, int n, float *out) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = blockIdx.x * 8 + warp;
    if (j >= n) return;
    const float4 *src = reinterpret_cast<const float4 *>(ring + (int64_t)slots[j] * ring_row);
    float4 *dst = reinterpret_cast<float4 *>(out + (int64_t)j * ring_row);
    for (int k = lane; k < ring_row / 4; k += 32) dst[k] = __ldcs(src + k);
}

static int64_t per_ws_bytes(sacb_handle h);
// bytes between two agents' sampler workspaces
static int64_t per_ws_stride(sacb_handle h) { return align_up(per_ws_bytes(h), 256); }
static PerWs per_ws_of(sacb_handle h, int agent) {
    PerWs w;
    char *base = (char *)h->per_ws + (int64_t)agent * per_ws_stride(h);
    const int64_t cap = h->cfg.capacity, nch = cap / kChunk + 2, B = h->cfg.max_batch;
    auto take = [&](size_t bytes) { char *p = base; base += align_up((int64_t)bytes, 256); return p; };
    // the same carve-up for every agent, per_ws_stride apart
    w.block_vals = (float *)take(sizeof(float) * 4096);
    w.total = (float *)take(256);
    w.chunk_sum = (double *)take(sizeof(double) * nch);
    w.chunk_carry = (double *)take(sizeof(double) * (nch + 1));
    w.chunk_fine = (int *)take(sizeof(int) * nch);
    w.counters = (int *)take(256);
    w.tickets = (int *)take(sizeof(int) * 3 * kTicketInts);
    w.block_max = (float *)take(sizeof(float) * 128);
    w.cdf_exact = (double *)take(sizeof(double) * cap);
    w.u = (double *)take(sizeof(double) * B);
    w.flagged = (int *)take(sizeof(int) * B);
    w.idx = (int64_t *)take(sizeof(int64_t) * B);
    w.weights = (float *)take(sizeof(float) * B);
    return w;
}
static int64_t per_ws_bytes(sacb_handle h) {
    const int64_t cap = h->cfg.capacity, nch = cap / kChunk + 2, B = h->cfg.max_batch;
    return 4096 * 4 + 256 + 8 * nch + 8 * (nch + 1) + 4 * nch + 256 + 8 * cap + 8 * B + 4 * B + 8 * B + 4 * B + 16 * 256 + 4 * 3 * kTicketInts + 256 + 4 * 128 + 256;
}

int replay_create(sacb_handle h) {
    const sacb_config &c = h->cfg;
    h->ring_row = align_up(2 * c.obs_dim + c.act_dim + 2, 4);
    const int n = c.n_agents;
    h->r_len.assign(n, 0); h->r_pos.assign(n, 0); h->r_head.assign(n, 0); h->per_frame.assign(n, 1);   // frame starts at 1 (replay_buffer.py:31)
    h->per_frame_dirty.assign(n, 1); h->sample_k.assign(n, 0); h->prio_max_valid.assign(n, 0);
    const size_t ring_bytes = sizeof(float) * (size_t)h->ring_row * c.capacity * n;
    if (cudaMalloc(&h->ring, ring_bytes) != cudaSuccess) { cudaGetLastError(); return fail(SACB_ERR_NOMEM, "replay ring does not fit in device memory"); }
    h->stage_rows_cap = std::max<int64_t>(c.max_batch, 4096);
    if (cudaMalloc(&h->stage_rows, sizeof(float) * h->ring_row * h->stage_rows_cap) != cudaSuccess) return fail(SACB_ERR_NOMEM, "staging alloc failed");
    if (c.replay_kind == SACB_REPLAY_PER) {
        if (n != 1 && c.capacity > kPopulationPerCapacity) return fail(SACB_ERR_ARG, "prioritized population: capacity <= 2096128 per agent");
        if (c.max_batch > 1024) return fail(SACB_ERR_ARG, "prioritized replay supports max_batch <= 1024");
        // per agent: prio / p_alpha [n, capacity], sampler workspace [n, per_ws_stride], last-sample indices [n, max_batch]
        const size_t tab = sizeof(float) * c.capacity * n, ws = (size_t)per_ws_stride(h) * n;
        if (cudaMalloc(&h->prio, tab) != cudaSuccess || cudaMalloc(&h->p_alpha, tab) != cudaSuccess ||
            cudaMalloc(&h->per_ws, ws) != cudaSuccess || cudaMalloc(&h->last_idx_dev, sizeof(int64_t) * c.max_batch * n) != cudaSuccess)
            return fail(SACB_ERR_NOMEM, "PER tables do not fit in device memory");
        cudaMemsetAsync(h->prio, 0, tab, h->stream);
        cudaMemsetAsync(h->p_alpha, 0, tab, h->stream);
        cudaMemsetAsync(h->per_ws, 0, ws, h->stream);
    }
    return SACB_OK;
}

void replay_destroy(sacb_handle h) {
    cudaFree(h->ring); cudaFree(h->stage_rows); cudaFree(h->prio); cudaFree(h->p_alpha); cudaFree(h->per_ws); cudaFree(h->last_idx_dev); cudaFree(h->gather_slots); cudaFree(h->ring_meta);
}

// logical index -> physical ring slot.  uniform: deque order (j-th oldest); PER: list position
static inline int64_t physical_slot(sacb_handle h, int agent, int64_t j) {
    if (h->cfg.replay_kind == SACB_REPLAY_PER) return j;
    return (h->r_head[agent] + j) % h->cfg.capacity;
}

// ring geometry for the device index draws: values travel as kernel parameters (no staging buffer to keep alive), <= 128 agents per launch
struct MetaChunk { int64_t v[256]; };
__global__ void set_ring_meta_kernel(int64_t *meta, MetaChunk c, int first, int count) {
    const int i = threadIdx.x;
    if (i < 2 * count) meta[2 * first + i] = c.v[i];
}
int upload_ring_meta(sacb_handle h) {
    if (!h->ring_meta_dirty) return SACB_OK;
    const int n = h->cfg.n_agents;
    if (!h->ring_meta && cudaMalloc(&h->ring_meta, sizeof(int64_t) * 2 * n) != cudaSuccess) return fail(SACB_ERR_NOMEM, "device allocation failed");
    for (int first = 0; first < n; first += 128) {
        MetaChunk c;
        const int count = std::min(128, n - first);
        for (int a = 0; a < count; a++) { c.v[2 * a] = h->r_len[first + a]; c.v[2 * a + 1] = h->r_head[first + a]; }
        set_ring_meta_kernel<<<1, 256, 0, h->stream>>>(h->ring_meta, c, first, count);
        h->kernel_launches++;
    }
    SACB_CUDA(cudaGetLastError());
    h->ring_meta_dirty = false;
    return SACB_OK;
}

int replay_stage_slots(sacb_handle h, const int64_t *idx, int64_t B) {
    const int n = h->cfg.n_agents;
    int32_t *pin = reinterpret_cast<int32_t *>(h->pin);
    if ((int64_t)n * B * (int64_t)sizeof(int32_t) > h->pin_floats * (int64_t)sizeof(float)) return fail(SACB_ERR_ARG, "index set too large");
    if (!h->ev_slots) SACB_CUDA(cudaEventCreateWithFlags(&h->ev_slots, cudaEventDisableTiming));
    if (h->slots_in_flight) SACB_CUDA(cudaEventSynchronize(h->ev_slots));      // the previous copy out of the pinned block (long done)
    for (int a = 0; a < n; a++)
        for (int64_t j = 0; j < B; j++) {
            const int64_t lj = idx[a * B + j];
            if (lj < 0 || lj >= h->r_len[a]) return fail(SACB_ERR_STATE, "replay index out of range");
            pin[a * B + j] = (int32_t)physical_slot(h, a, lj);
        }
    for (int a = 0; a < n; a++)
        SACB_CUDA(cudaMemcpyAsync(h->slots + (int64_t)a * h->cfg.max_batch, pin + a * B, sizeof(int32_t) * B, cudaMemcpyHostToDevice, h->stream));
    SACB_CUDA(cudaEventRecord(h->ev_slots, h->stream));      // no synchronisation on this path: the update is enqueued right behind
    h->slots_in_flight = true;
    return SACB_OK;
}

}  // namespace sacb
using namespace sacb;

extern "C" int sacb_stage_indices(sacb_handle h, const int64_t *idx, int64_t B, int64_t n_steps) {
    if (!h || !idx || B < 1 || B > h->cfg.max_batch || n_steps < 1) return fail(SACB_ERR_ARG, "bad argument");
    const int n = h->cfg.n_agents;
    std::vector<int32_t> slots((size_t)n_steps * n * B);
    for (int64_t s = 0; s < n_steps; s++)
        for (int a = 0; a < n; a++)
            for (int64_t j = 0; j < B; j++) {
                const int64_t lj = idx[(s * n + a) * B + j];
                if (lj < 0 || lj >= h->r_len[a]) return fail(SACB_ERR_STATE, "replay index out of range");
                slots[(s * n + a) * B + j] = (int32_t)physical_slot(h, a, lj);
            }
    if (B != h->cfg.max_batch && n > 1) return fail(SACB_ERR_ARG, "population staging needs B == max_batch");
    cudaFree(h->slots_staged);
    SACB_CUDA(cudaMalloc(&h->slots_staged, slots.size() * sizeof(int32_t)));
    SACB_CUDA(cudaMemcpy(h->slots_staged, slots.data(), slots.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    h->staged_steps = n_steps; h->staged_next = 0; h->staged_B = B;
    return SACB_OK;
}

extern "C" int64_t sacb_len(sacb_handle h, int agent) {
    if (!h || agent < 0 || agent >= h->cfg.n_agents) return -1;
    return h->r_len[agent];
}

extern "C" int sacb_clear_replay(sacb_handle h, int agent) {
    if (!h || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    h->r_len[agent] = h->r_pos[agent] = h->r_head[agent] = 0;
    h->ring_meta_dirty = true;
    h->sample_k[agent] = 0;
    h->prio_max_valid[agent] = 0;
    if (h->prio) {      // this agent's tables only
        const int64_t cap = h->cfg.capacity;
        cudaMemsetAsync(h->prio + agent * cap, 0, sizeof(float) * cap, h->stream); cudaMemsetAsync(h->p_alpha + agent * cap, 0, sizeof(float) * cap, h->stream);
    }
    return SACB_OK;
}

// max(priorities) over the whole capacity array (replay_buffer.py:38) as 128 CTA maxima.  The table only changes through
// update_priorities / set_priorities / clear (a push writes the maximum itself, which leaves it unchanged), so the reduction runs
// right behind those -- off the push -> sample -> update critical path -- and push reuses it while `prio_max_valid`.
// agents [first, first + count), one launch (blockIdx.y = agent)
static void per_refresh_max(sacb_handle h, cudaStream_t st, int first, int count) {
    PerWs w = per_ws_of(h, first);
    const int64_t cap = h->cfg.capacity;
    max_reduce_kernel<<<dim3(128, count), 1024, 0, st>>>(h->prio + first * cap, cap, w.block_max, cap, per_ws_stride(h) / (int64_t)sizeof(float));
    h->kernel_launches++;
    for (int a = first; a < first + count; a++) h->prio_max_valid[a] = 1;
}

// ring = the agent's ring (the push kernel moves pinned rows there itself)
static int per_push_priorities(sacb_handle h, int agent, int64_t pos, int64_t count, bool empty, float *ring, const float *pinned_rows = nullptr) {
    PerWs w = per_ws_of(h, agent);
    const int nb = 128;
    const int64_t cap = h->cfg.capacity;
    if (!empty && !h->prio_max_valid[agent]) per_refresh_max(h, h->stream, agent, 1);
    const int row_vec4 = (int)(h->ring_row / 4);
    const int64_t work = pinned_rows ? std::max<int64_t>(count, count * row_vec4) : count;
    per_push_kernel<<<(int)std::min<int64_t>(64, (work + 255) / 256), 256, 0, h->stream>>>(h->prio + agent * cap, h->p_alpha + agent * cap, w.block_max, nb, empty ? 1 : 0,
                                                                                         pos, count, cap, h->cfg.per_alpha, reinterpret_cast<const float4 *>(pinned_rows),
                                                                                         reinterpret_cast<float4 *>(ring), row_vec4);
    h->kernel_launches++;
    if (empty) h->prio_max_valid[agent] = 0;      // the first push writes 1.0 into an all-zero table: reduce again next time
    SACB_CUDA(cudaGetLastError());
    return SACB_OK;
}

extern "C" int sacb_push(sacb_handle h, int agent, const float *s, const float *a, const float *r, const float *s2, const float *done, int64_t n) {
    if (!h || !s || !a || !r || !s2 || !done || agent < 0 || agent >= h->cfg.n_agents || n < 0) return fail(SACB_ERR_ARG, "bad argument");
    const sacb_config &c = h->cfg;
    const int64_t cap = c.capacity, row = h->ring_row;
    float *ring = h->ring + (int64_t)agent * cap * row;
    const bool per = c.replay_kind == SACB_REPLAY_PER;
    int64_t done_n = 0;
    h->ring_meta_dirty = true;
    while (done_n < n) {
        // next write slot; a contiguous run never crosses the end of the ring
        int64_t slot;
        if (per) slot = h->r_pos[agent];
        else slot = h->r_len[agent] < cap ? (h->r_head[agent] + h->r_len[agent]) % cap : h->r_head[agent];
        const int64_t run = std::min(n - done_n, cap - slot);
        const size_t pitch = sizeof(float) * row, wo = sizeof(float) * c.obs_dim, wa = sizeof(float) * c.act_dim;
        float *dst = ring + slot * row;
        SACB_CUDA(cudaMemcpy2DAsync(dst, pitch, s + done_n * c.obs_dim, wo, wo, run, cudaMemcpyHostToDevice, h->stream));
        SACB_CUDA(cudaMemcpy2DAsync(dst + c.obs_dim, pitch, s2 + done_n * c.obs_dim, wo, wo, run, cudaMemcpyHostToDevice, h->stream));
        SACB_CUDA(cudaMemcpy2DAsync(dst + 2 * c.obs_dim, pitch, a + done_n * c.act_dim, wa, wa, run, cudaMemcpyHostToDevice, h->stream));
        SACB_CUDA(cudaMemcpy2DAsync(dst + 2 * c.obs_dim + c.act_dim, pitch, r + done_n, sizeof(float), sizeof(float), run, cudaMemcpyHostToDevice, h->stream));
        SACB_CUDA(cudaMemcpy2DAsync(dst + 2 * c.obs_dim + c.act_dim + 1, pitch, done + done_n, sizeof(float), sizeof(float), run, cudaMemcpyHostToDevice, h->stream));
        if (per) {
            int rc = per_push_priorities(h, agent, slot, run, h->r_len[agent] == 0, ring);
            if (rc) return rc;
            h->r_pos[agent] = (slot + run) % cap;
            h->r_len[agent] = std::min(cap, h->r_len[agent] + run);
        } else {
            const int64_t grow = std::min(run, cap - h->r_len[agent]);
            h->r_len[agent] += grow;
            h->r_head[agent] = (h->r_head[agent] + (run - grow)) % cap;      // overwritten oldest entries (deque maxlen eviction)
        }
        done_n += run;
    }
    SACB_CUDA(cudaStreamSynchronize(h->stream));     // caller may reuse its buffers
    return SACB_OK;
}

extern "C" int64_t sacb_row_floats(sacb_handle h) { return h ? h->ring_row : -1; }

// host-side helper of ReplayBuffer's index draw (include/sacb200.h): append the first distinct values below n of a word stream
extern "C" int64_t sacb_host_first_distinct(const uint32_t *words, int64_t n_words, uint64_t n, int shift, int64_t *picks, int64_t n_have, int64_t k) {
    if (!words || !picks || n_words < 0 || n_have < 0 || k < n_have || shift < 0 || shift > 31) return -1;
    // open addressing over the picks so far (k is a minibatch size: the table is a few KB and rebuilt per call)
    int64_t cap = 16;
    while (cap < 4 * k) cap <<= 1;
    std::vector<int64_t> table((size_t)cap, -1);
    auto insert = [&](int64_t v) -> bool {      // false: already present
        uint64_t hsh = (uint64_t)v * 0x9E3779B97F4A7C15ull;
        for (int64_t i = (int64_t)(hsh >> 32) & (cap - 1);; i = (i + 1) & (cap - 1)) {
            if (table[(size_t)i] == v) return false;
            if (table[(size_t)i] < 0) { table[(size_t)i] = v; return true; }
        }
    };
    for (int64_t j = 0; j < n_have; j++) insert(picks[j]);
    for (int64_t j = 0; j < n_words && n_have < k; j++) {
        const uint64_t v = words[j] >> shift;
        if (v < n && insert((int64_t)v)) picks[n_have++] = (int64_t)v;
    }
    return n_have;
}

extern "C" int sacb_push_rows(sacb_handle h, int agent, const float *rows, int64_t n) {
    if (!h || !rows || agent < 0 || agent >= h->cfg.n_agents || n < 0) return fail(SACB_ERR_ARG, "bad argument");
    const sacb_config &c = h->cfg;
    const int64_t cap = c.capacity, row = h->ring_row;
    float *ring = h->ring + (int64_t)agent * cap * row;
    const bool per = c.replay_kind == SACB_REPLAY_PER;
    // the trainer's one-transition push (trainer.py:194): staged through pinned memory, nothing on this path waits for the device
    const bool staged = n <= kPinPushRows && h->pin_push;
    if (staged) {
        if (h->push_in_flight) SACB_CUDA(cudaEventSynchronize(h->ev_push));      // the previous copy out of the staging buffer (long done)
        memcpy(h->pin_push, rows, sizeof(float) * row * n);
        rows = h->pin_push;
    }
    int64_t done_n = 0;
    h->ring_meta_dirty = true;
    while (done_n < n) {
        int64_t slot;
        if (per) slot = h->r_pos[agent];
        else slot = h->r_len[agent] < cap ? (h->r_head[agent] + h->r_len[agent]) % cap : h->r_head[agent];
        const int64_t run = std::min(n - done_n, cap - slot);
        const bool by_kernel = per && staged;      // the push kernel moves the rows out of the pinned block itself
        if (!by_kernel) SACB_CUDA(cudaMemcpyAsync(ring + slot * row, rows + done_n * row, sizeof(float) * row * run, cudaMemcpyHostToDevice, h->stream));
        if (per) {
            int rc = per_push_priorities(h, agent, slot, run, h->r_len[agent] == 0, ring, by_kernel ? rows + done_n * row : nullptr);
            if (rc) return rc;
            h->r_pos[agent] = (slot + run) % cap;
            h->r_len[agent] = std::min(cap, h->r_len[agent] + run);
        } else {
            const int64_t grow = std::min(run, cap - h->r_len[agent]);
            h->r_len[agent] += grow;
            h->r_head[agent] = (h->r_head[agent] + (run - grow)) % cap;
        }
        done_n += run;
    }
    if (staged) { SACB_CUDA(cudaEventRecord(h->ev_push, h->stream)); h->push_in_flight = true; }
    else SACB_CUDA(cudaStreamSynchronize(h->stream));      // the caller may reuse its buffer
    return SACB_OK;
}

static int gather_to_host(sacb_handle h, int agent, const int32_t *slots_host, int64_t n, float *s, float *a, float *r, float *s2, float *done) {
    const sacb_config &c = h->cfg;
    const int64_t row = h->ring_row;
    const float *ring = h->ring + (int64_t)agent * c.capacity * row;
    // host-facing reads (`.buffer`, checkpoints, ReplayBuffer.sample of any size) move stage_rows_cap rows per round trip
    if (!h->gather_slots && cudaMalloc(&h->gather_slots, sizeof(int32_t) * h->stage_rows_cap) != cudaSuccess) return fail(SACB_ERR_NOMEM, "device allocation failed");
    // slots_host == null: the slots of the last prioritized sample, already on the device (at most max_batch of them)
    int32_t *slots_dev = slots_host ? h->gather_slots : h->slots + (int64_t)agent * c.max_batch;
    const int64_t chunk = slots_host ? h->stage_rows_cap : std::max<int64_t>(n, 1);
    for (int64_t off = 0; off < n; off += chunk) {
        const int64_t m = std::min<int64_t>(chunk, n - off);
        if (slots_host) SACB_CUDA(cudaMemcpyAsync(slots_dev, slots_host + off, sizeof(int32_t) * m, cudaMemcpyHostToDevice, h->stream));
        gather_rows_kernel<<<(int)((m + 7) / 8), 256, 0, h->stream>>>(ring, row, slots_dev, (int)m, h->stage_rows);
        h->kernel_launches++;
        const size_t pitch = sizeof(float) * row, wo = sizeof(float) * c.obs_dim, wa = sizeof(float) * c.act_dim;
        const float *src = h->stage_rows;
        if (s) SACB_CUDA(cudaMemcpy2DAsync(s + off * c.obs_dim, wo, src, pitch, wo, m, cudaMemcpyDeviceToHost, h->stream));
        if (s2) SACB_CUDA(cudaMemcpy2DAsync(s2 + off * c.obs_dim, wo, src + c.obs_dim, pitch, wo, m, cudaMemcpyDeviceToHost, h->stream));
        if (a) SACB_CUDA(cudaMemcpy2DAsync(a + off * c.act_dim, wa, src + 2 * c.obs_dim, pitch, wa, m, cudaMemcpyDeviceToHost, h->stream));
        if (r) SACB_CUDA(cudaMemcpy2DAsync(r + off, sizeof(float), src + 2 * c.obs_dim + c.act_dim, pitch, sizeof(float), m, cudaMemcpyDeviceToHost, h->stream));
        if (done) SACB_CUDA(cudaMemcpy2DAsync(done + off, sizeof(float), src + 2 * c.obs_dim + c.act_dim + 1, pitch, sizeof(float), m, cudaMemcpyDeviceToHost, h->stream));
        SACB_CUDA(cudaStreamSynchronize(h->stream));
    }
    return SACB_OK;
}

extern "C" int sacb_read_transitions(sacb_handle h, int agent, const int64_t *idx, int64_t n, float *s, float *a, float *r, float *s2, float *done) {
    if (!h || !idx || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    std::vector<int32_t> slots(n);
    for (int64_t j = 0; j < n; j++) {
        if (idx[j] < 0 || idx[j] >= h->r_len[agent]) return fail(SACB_ERR_STATE, "replay index out of range");
        slots[j] = (int32_t)physical_slot(h, agent, idx[j]);
    }
    return gather_to_host(h, agent, slots.data(), n, s, a, r, s2, done);
}

extern "C" int sacb_sample_uniform(sacb_handle h, int agent, const int64_t *idx, int64_t B, float *s, float *a, float *r, float *s2, float *done) {
    if (!h || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    if (B > h->r_len[agent]) return fail(SACB_ERR_STATE, "Sample larger than population or is negative");   // random.sample's ValueError
    if (!idx) return fail(SACB_ERR_ARG, "indices required (draw them with random.sample(range(len), B))");
    return sacb_read_transitions(h, agent, idx, B, s, a, r, s2, done);
}

// ---- PER --------------------------------------------------------------------------------------------------------
namespace sacb {
static int64_t *per_frame_dev(sacb_handle h, int agent) { return reinterpret_cast<int64_t *>(per_ws_of(h, agent).counters + 8); }

// create / sacb_per_set_frame: the device copy of every agent's frame counter follows the host's
int upload_per_frame(sacb_handle h, cudaStream_t st) {
    bool any = false;
    for (int a = 0; a < h->cfg.n_agents; a++) {
        if (!h->per_frame_dirty[a]) continue;
        SACB_CUDA(cudaMemcpyAsync(per_frame_dev(h, a), &h->per_frame[a], sizeof(int64_t), cudaMemcpyHostToDevice, st));
        any = true;
    }
    if (!any) return SACB_OK;
    SACB_CUDA(cudaStreamSynchronize(st));
    for (int a = 0; a < h->cfg.n_agents; a++) h->per_frame_dirty[a] = 0;
    return SACB_OK;
}

int per_sample_launch(sacb_handle h, cudaStream_t st, const double *u, int64_t B, int64_t *k_out, int first, int count) {
    if (!h || h->cfg.replay_kind != SACB_REPLAY_PER) return fail(SACB_ERR_ARG, "handle has no prioritized buffer");
    if (first < 0 || count < 1 || first + count > h->cfg.n_agents) return fail(SACB_ERR_ARG, "agent index out of range");
    int64_t n = h->r_len[first], k;
    if (count == 1) {
        if (n < 1) return fail(SACB_ERR_STATE, "cannot sample from an empty buffer");
        k = std::min<int64_t>(B, n);                                 // n_samples = min(batch_size, len)  (replay_buffer.py:50)
    } else {      // every agent's minibatch has B rows (the batched update program): len >= B everywhere; grids sized for the longest agent
        for (int a = first; a < first + count; a++) {
            if (h->r_len[a] < B) return fail(SACB_ERR_STATE, "population sample: every agent's buffer must hold at least B transitions");
            n = std::max(n, h->r_len[a]);
        }
        k = B;
    }
    if (k > h->cfg.max_batch) return fail(SACB_ERR_ARG, "batch size exceeds max_batch");
    PerWs w = per_ws_of(h, 0);      // agent 0's pointers: the kernels add each agent's stride
    const bool pdl = h->use_pdl != 0;
    int64_t *frame_dev = per_frame_dev(h, 0);
    if (int rc = upload_per_frame(h, st)) return rc;
    if (count > 1) { if (int rc = upload_ring_meta(h)) return rc; }      // each agent's length, read by the kernels
    for (int a = first; a < first + count; a++) h->per_frame[a] += 1;    // host mirror (statistics, `frame`); the kernels read and advance the device copy
    const int64_t mb = h->cfg.max_batch;
    if (u) {      // host-drawn uniforms (np.random.random_sample inside np.random.choice): through pinned memory, no pageable staging
        if (!h->pin_u) {
            if (cudaMallocHost(&h->pin_u, sizeof(double) * mb * h->cfg.n_agents) != cudaSuccess || cudaEventCreateWithFlags(&h->ev_u, cudaEventDisableTiming) != cudaSuccess)
                return fail(SACB_ERR_NOMEM, "pinned allocation failed");
        }
        if (h->u_in_flight) SACB_CUDA(cudaEventSynchronize(h->ev_u));      // the previous call's search kernel has read the block (long done)
        // the search kernel reads them from here (host memory is addressable from the device): no copy call.  Row of agent a: pin_u + a * max_batch
        for (int a = first; a < first + count; a++) memcpy(h->pin_u + a * mb, u + (a - first) * k, sizeof(double) * k);
    }
    const double *u_dev = u ? h->pin_u : w.u;
    const int depth = top_depth_of(n);
    if (depth > 11) return fail(SACB_ERR_ARG, "capacity too large for the summation heap");
    const float *pa = h->p_alpha;
    int *tickets = w.tickets;
    const int n_chunks = (int)((n + kChunk - 1) / kChunk);
    SearchArgs sa;
    sa.p_alpha = pa; sa.n = n; sa.u = u_dev; sa.B = (int)k; sa.counters = w.counters; sa.idx_out = w.idx; sa.flagged = w.flagged;
    sa.ticket = tickets + 2 * kTicketInts; sa.carry_exact = w.cdf_exact; sa.chunk_sum = w.chunk_sum; sa.chunk_fine = w.chunk_fine; sa.n_chunks = n_chunks;
    sa.weights = w.weights; sa.slots = h->slots; sa.isw_ws = h->ws + h->L.isw; sa.idx_copy = h->last_idx_dev;
    sa.frame = frame_dev; sa.beta_start = (double)h->cfg.per_beta_start; sa.one_minus_start = 1.0 - (double)h->cfg.per_beta_start; sa.beta_frames = (double)h->cfg.per_beta_frames;
    const int64_t ws_stride = per_ws_stride(h);
    const PerAgents g{count > 1 ? h->ring_meta : nullptr, first, h->cfg.capacity, ws_stride, u ? (int64_t)sizeof(double) * mb : ws_stride, mb, h->L.ws_size};
    // no serial tails while the chunk prefixes fit into shared memory (DESIGN.md section 4 records the one- and two-launch forms measured against this)
    const bool no_tails = n_chunks + 1 <= kCarrySmem;
    if (!no_tails && h->cfg.n_agents != 1) return fail(SACB_ERR_ARG, "prioritized population: capacity <= 2096128 per agent");
    const bool agents = h->cfg.n_agents > 1;      // population handles: the kernels with the agent offsets
    SACB_CUDA(launch_pdl(agents ? per_sum<true> : per_sum<false>, dim3((2 << depth) - 1, count), dim3(256), 0, st, pdl, pa, n, depth, w.block_vals, w.total, tickets + 0,
                         w.u, u ? 0 : (int)k, h->cfg.seed, (const int64_t *)frame_dev, no_tails ? 0 : 1, g));
    if (no_tails) {
        SACB_CUDA(launch_pdl(agents ? per_chunk_notail<true> : per_chunk_notail<false>, dim3((n_chunks + 7) / 8, count), dim3(256), 0, st, pdl, pa, n, depth, (const float *)w.block_vals, w.total,
                             w.chunk_sum, w.chunk_fine, g));
        SACB_CUDA(launch_pdl(agents ? per_search_scan<true> : per_search_scan<false>, dim3((int)((k + 7) / 8), count), dim3(256), 0, st, pdl, (const float *)w.total, w.chunk_carry, sa, g));
    } else {
        SACB_CUDA(launch_pdl(per_chunk, dim3((n_chunks + 7) / 8), dim3(256), 0, st, pdl, pa, n, (const float *)w.total, w.chunk_sum, w.chunk_fine,
                             n_chunks, w.chunk_carry, w.counters, tickets + kTicketInts));
        SACB_CUDA(launch_pdl(per_search, dim3((int)((k + 7) / 8)), dim3(256), 0, st, pdl, (const float *)w.total, (const double *)w.chunk_carry, sa));
    }
    h->kernel_launches += 3;
    if (u) { SACB_CUDA(cudaEventRecord(h->ev_u, st)); h->u_in_flight = true; }      // behind the last kernel of the call
    for (int a = first; a < first + count; a++) h->sample_k[a] = k;
    if (k_out) *k_out = k;
    return SACB_OK;
}

// priorities <- |td| + 1e-6 of the last update for agents [first, first + count): one CTA per agent, then their CTA maxima
int per_writeback_launch(sacb_handle h, cudaStream_t st, int64_t B, bool pdl_ok, int first, int count) {
    const int64_t cap = h->cfg.capacity, mb = h->cfg.max_batch, wss = h->L.ws_size;
    SACB_CUDA(launch_pdl(per_update_kernel, dim3(count), dim3(1024), sizeof(int64_t) * B, st, h->use_pdl != 0 && pdl_ok, h->prio + first * cap,
                         h->p_alpha + first * cap, (const int64_t *)(h->last_idx_dev + first * mb), (const float *)(h->ws + first * wss + h->L.td), (int)B,
                         h->cfg.per_alpha, 0, cap, mb, wss));
    h->kernel_launches++;
    per_refresh_max(h, st, first, count);      // for the next push; same stream, behind the write-back
    return SACB_OK;
}
}  // namespace sacb

static bool bad_per_agent(sacb_handle h, int agent) { return !h || agent < 0 || agent >= h->cfg.n_agents || h->cfg.replay_kind != SACB_REPLAY_PER; }

extern "C" int sacb_per_sample(sacb_handle h, int agent, const double *u, int64_t B, int64_t *idx_out, float *weights_out,
                               float *s, float *a, float *r, float *s2, float *done) {
    if (!h || h->cfg.replay_kind != SACB_REPLAY_PER) return fail(SACB_ERR_ARG, "handle has no prioritized buffer");
    if (agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "agent index out of range");
    int64_t k = 0;
    int rc = per_sample_launch(h, h->stream, u, B, &k, agent, 1);
    if (rc) return rc;
    PerWs w = per_ws_of(h, agent);
    if (idx_out) SACB_CUDA(cudaMemcpyAsync(idx_out, w.idx, sizeof(int64_t) * k, cudaMemcpyDeviceToHost, h->stream));
    if (weights_out) SACB_CUDA(cudaMemcpyAsync(weights_out, w.weights, sizeof(float) * k, cudaMemcpyDeviceToHost, h->stream));
    if (s || a || r || s2 || done) return gather_to_host(h, agent, nullptr, k, s, a, r, s2, done);
    if (idx_out || weights_out) SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

extern "C" int sacb_per_sample_all(sacb_handle h, const double *u, int64_t B, int64_t *idx_out, float *weights_out) {
    if (!h || h->cfg.replay_kind != SACB_REPLAY_PER) return fail(SACB_ERR_ARG, "handle has no prioritized buffer");
    if (B < 1 || B > h->cfg.max_batch) return fail(SACB_ERR_ARG, "batch size out of range");
    const int n = h->cfg.n_agents;
    for (int a = 0; a < n; a++)
        if (h->r_len[a] < B) return fail(SACB_ERR_STATE, "population sample: every agent's buffer must hold at least B transitions");
    int rc = per_sample_launch(h, h->stream, u, B, nullptr, 0, n);
    if (rc) return rc;
    // the results sit at the same offset of every agent's workspace: one strided copy each
    PerWs w = per_ws_of(h, 0);
    const size_t pitch = (size_t)per_ws_stride(h);
    if (idx_out) SACB_CUDA(cudaMemcpy2DAsync(idx_out, sizeof(int64_t) * B, w.idx, pitch, sizeof(int64_t) * B, n, cudaMemcpyDeviceToHost, h->stream));
    if (weights_out) SACB_CUDA(cudaMemcpy2DAsync(weights_out, sizeof(float) * B, w.weights, pitch, sizeof(float) * B, n, cudaMemcpyDeviceToHost, h->stream));
    if (idx_out || weights_out) SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

static int per_update_impl(sacb_handle h, int agent, const int64_t *idx, const float *prio, int64_t B, int is_final);
extern "C" int sacb_per_update(sacb_handle h, int agent, const int64_t *idx, const float *prio, int64_t B) { return per_update_impl(h, agent, idx, prio, B, 0); }
extern "C" int sacb_per_update_final(sacb_handle h, int agent, const int64_t *idx, const float *prio, int64_t B) { return per_update_impl(h, agent, idx, prio, B, 1); }
extern "C" int sacb_per_update_from_td(sacb_handle h, int agent, int64_t B) {
    if (bad_per_agent(h, agent)) return fail(SACB_ERR_ARG, "bad argument");
    if (B < 1 || B > h->cfg.max_batch) return fail(SACB_ERR_ARG, "batch size out of range");
    if (h->sample_k[agent] != B) return fail(SACB_ERR_STATE, "sacb_per_update_from_td: the last prioritized sample does not hold B rows");
    return per_writeback_launch(h, h->stream, B, true, agent, 1);
}
static int per_update_impl(sacb_handle h, int agent, const int64_t *idx, const float *prio, int64_t B, int is_final) {
    if (bad_per_agent(h, agent) || !prio) return fail(SACB_ERR_ARG, "bad argument");
    if (B < 1 || B > h->cfg.max_batch) return fail(SACB_ERR_ARG, "batch size out of range");
    PerWs w = per_ws_of(h, agent);
    const int64_t cap = h->cfg.capacity;
    const int64_t *idx_dev = h->last_idx_dev + agent * h->cfg.max_batch;
    if (idx) {
        for (int64_t j = 0; j < B; j++) if (idx[j] < 0 || idx[j] >= cap) return fail(SACB_ERR_STATE, "priority index out of range");
        SACB_CUDA(cudaMemcpyAsync(w.idx, idx, sizeof(int64_t) * B, cudaMemcpyHostToDevice, h->stream));
        idx_dev = w.idx;
    }
    SACB_CUDA(cudaMemcpyAsync(w.weights, prio, sizeof(float) * B, cudaMemcpyHostToDevice, h->stream));
    per_update_kernel<<<1, 1024, sizeof(int64_t) * B, h->stream>>>(h->prio + agent * cap, h->p_alpha + agent * cap, idx_dev, w.weights, (int)B, h->cfg.per_alpha,
                                                                   is_final, cap, h->cfg.max_batch, 0);
    h->kernel_launches++;
    h->prio_max_valid[agent] = 0;
    SACB_CUDA(cudaGetLastError());
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

extern "C" int sacb_per_get_priorities(sacb_handle h, int agent, float *prio, int64_t n) {
    if (bad_per_agent(h, agent) || !h->prio || n > h->cfg.capacity) return fail(SACB_ERR_ARG, "bad argument");
    SACB_CUDA(cudaMemcpyAsync(prio, h->prio + agent * h->cfg.capacity, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

extern "C" int sacb_per_set_priorities(sacb_handle h, int agent, const float *prio, const float *p_alpha, int64_t n) {
    if (bad_per_agent(h, agent) || !h->prio || n > h->cfg.capacity || !prio) return fail(SACB_ERR_ARG, "bad argument");
    h->sample_k[agent] = 0;      // a minibatch drawn from the old table is stale
    h->prio_max_valid[agent] = 0;
    float *pr = h->prio + agent * h->cfg.capacity, *pa = h->p_alpha + agent * h->cfg.capacity;
    SACB_CUDA(cudaMemcpyAsync(pr, prio, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    if (p_alpha) SACB_CUDA(cudaMemcpyAsync(pa, p_alpha, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    else { pow_alpha_kernel<<<256, 256, 0, h->stream>>>(pr, pa, n, h->cfg.per_alpha); h->kernel_launches++; }
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    return SACB_OK;
}

extern "C" int sacb_per_get_stats(sacb_handle h, int agent, sacb_per_stats *out) {
    if (bad_per_agent(h, agent) || !h->prio || !out) return fail(SACB_ERR_ARG, "bad argument");
    PerWs w = per_ws_of(h, agent);
    int counters[4] = {0, 0, 0, 0};
    float tot = 0.f; double last = 0.0;
    const int64_t n = std::max<int64_t>(1, h->r_len[agent]);
    const int n_chunks = (int)((n + kChunk - 1) / kChunk);
    SACB_CUDA(cudaMemcpyAsync(counters, w.counters, sizeof(int) * 4, cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaMemcpyAsync(&tot, w.total, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaMemcpyAsync(&last, w.chunk_carry + n_chunks, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    SACB_CUDA(cudaStreamSynchronize(h->stream));
    out->frame = h->per_frame[agent]; out->pos = h->r_pos[agent]; out->len = h->r_len[agent];
    out->n_fine = counters[0]; out->n_flagged = counters[3]; out->n_exact_fallbacks = counters[2];
    out->total_f32 = tot; out->cdf_last = last;
    return SACB_OK;
}

extern "C" int sacb_per_set_frame(sacb_handle h, int agent, int64_t frame) {
    if (!h || agent < 0 || agent >= h->cfg.n_agents) return fail(SACB_ERR_ARG, "bad argument");
    h->per_frame[agent] = frame;
    h->per_frame_dirty[agent] = 1;
    return SACB_OK;
}
