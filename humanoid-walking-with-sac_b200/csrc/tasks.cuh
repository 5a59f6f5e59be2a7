// Non-GEMM tile tasks of the SAC update program (weight shadows, gather, sampling, losses, bias / output-layer
// optimiser steps).  Each body reads its own argument struct of Task's union (common.cuh), which the host builder (program.cu)
// fills.  Matrices that feed a GEMM are pair matrices (bf16 hi/lo planes, common.cuh).
#pragma once
#include "gemm.cuh"
#include "sample.cuh"

namespace sacb {

constexpr int kShadowRows = 64;      // weight rows per T_SHADOW tile (4 per warp)

// T_SHADOW: one warp per row.  Runs at the start of every step, so weights written from outside the update (load_state_dict
// through the aliased torch tensors, checkpoint loads, the data-parallel apply kernel) are always picked up.
__device__ __forceinline__ void task_shadow(const ShadowArgs &t, int tile, const Program &P, int agent) {
    const int rows = t.rows, cols = t.cols;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const Pm dst = resolve_pm(t.dst, P.bases, agent);
    const float *src0 = resolve(t.src, P.bases, agent) + t.col0;
    const bool even = ((t.src_ld | t.col0) & 1) == 0;     // every row starts 8 B aligned in src and 4 B aligned in dst
    constexpr int kR = kShadowRows / (kThreads / 32);    // rows per warp, handled together: kR independent loads in flight per trip
    const int r0 = tile * kShadowRows + warp;
    constexpr int kU = 4;                                // column chunks handled together: kR * kU independent loads in flight per trip
    for (int c0 = 2 * lane; c0 < cols; c0 += 64 * kU) {
        float2 x[kR][kU];
#pragma unroll
        for (int i = 0; i < kR; i++) {
            const int r = r0 + i * (kThreads / 32);
#pragma unroll
            for (int u = 0; u < kU; u++) {
                const int c = c0 + 64 * u;
                x[i][u] = make_float2(0.f, 0.f);
                if (r < rows && c < cols) {
                    const float *src = src0 + (int64_t)r * t.src_ld + c;
                    if (even) x[i][u] = __ldcg(reinterpret_cast<const float2 *>(src));
                    else { x[i][u].x = ldcg(src); if (c + 1 < cols) x[i][u].y = ldcg(src + 1); }
                }
            }
        }
#pragma unroll
        for (int i = 0; i < kR; i++) {
            const int r = r0 + i * (kThreads / 32);
            if (r >= rows) continue;
#pragma unroll
            for (int u = 0; u < kU; u++) {
                const int c = c0 + 64 * u;
                if (c >= cols) continue;
                if (c + 1 >= cols) x[i][u].y = 0.f;
                uint32_t hi, lo;
                split_pack2(x[i][u].x, x[i][u].y, hi, lo);
                __nv_bfloat16 *q = dst.hi + (int64_t)r * dst.ld + c;
                *reinterpret_cast<uint32_t *>(q) = hi;
                *reinterpret_cast<uint32_t *>(q + dst.plane) = lo;
            }
        }
    }
}

// T_GATHER: ring row = [s | s2 | a | r | d] (16 B aligned)
//   X rows [0,B) <- (s2, .)   rows [B,2B) <- (s, a)   rows [2B,3B) <- (s, .)
// four rows per tile, four warps per sampled row: one warp per destination row (the fourth moves r and d).  A lane forms
// pairs of neighbouring destination columns (one 4-byte store per bf16 plane); ring reads are coalesced streaming loads,
// 8 in flight per lane.
// Device index draw of the uniform ring (production mode, no host in the loop): minibatch row b of update `step` reads the
// transition at logical position perm(b), perm = a keyed bijection of [0, n) -- B DISTINCT positions, i.e. sampling without
// replacement like random.sample (replay_buffer.py:15).  The bijection works on the next power of two (rounds of odd multiply /
// add / xor-shift, each a bijection of k-bit integers, keyed by Philox(seed; step, agent)) and cycle-walks back into [0, n).
__device__ __forceinline__ uint32_t draw_position(uint32_t b, uint32_t n, uint64_t seed, uint32_t agent, uint32_t step) {
    uint32_t key[4] = {step, agent, 0x1d5a7b1eu, 0u};
    philox4x32(key, (uint32_t)seed, (uint32_t)(seed >> 32));
    uint32_t k2[4] = {step, agent, 0x1d5a7b1fu, 1u};
    philox4x32(k2, (uint32_t)seed, (uint32_t)(seed >> 32));
    const int bits = n <= 2 ? 1 : 32 - __clz(n - 1);
    const uint32_t mask = bits >= 32 ? 0xFFFFFFFFu : ((1u << bits) - 1u);
    const int sh = max(1, bits / 2);
    uint32_t x = b;
    do {
#pragma unroll
        for (int r = 0; r < 4; r++) {
            x = (x * (key[r] | 1u) + k2[r]) & mask;
            x ^= x >> sh;
        }
    } while (x >= n);
    return x;
}

__device__ __forceinline__ void task_gather(const GatherArgs &t, int tile, const Program &P, int agent, const float *scalars, uint64_t seed) {
    const int B = t.B, obs = t.obs, act = t.act;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = tile * 4 + (warp >> 2), part = warp & 3;
    if (b >= B) return;
    int slot;
    if (t.device_draw) {      // indices drawn here (the four warps of a row compute the same slot); recorded for the host / tests
        const int64_t n = P.ring_meta[2 * agent], head = P.ring_meta[2 * agent + 1];
        const uint32_t step = (uint32_t)__float_as_int(ldcg(scalars + SC_N_UPDATES));
        slot = (int)((head + draw_position((uint32_t)b, (uint32_t)n, seed, (uint32_t)agent, step)) % t.capacity);
        if (part == 3 && lane == 2) const_cast<int32_t *>(P.slots)[(int64_t)agent * P.slots_stride + b] = slot;
    } else {
        slot = P.slots[(int64_t)agent * P.slots_stride + b];
    }
    const float *row = P.ring + agent * P.ring_agent_stride + (int64_t)slot * P.ring_row;
    if (part == 3) {
        if (lane == 0) resolve(t.r, P.bases, agent)[b] = __ldcs(row + 2 * obs + act);
        if (lane == 1) resolve(t.d, P.bases, agent)[b] = __ldcs(row + 2 * obs + act + 1);
        return;
    }
    const Pm X = resolve_pm(t.x, P.bases, agent);
    const int xrow = part == 0 ? b : (part == 1 ? B + b : 2 * B + b);
    const int ncols = part == 1 ? obs + act : obs;
    auto src = [&](int c) -> float {       // destination column -> ring element
        if (part == 0) return __ldcs(row + obs + c);
        return __ldcs(row + (c < obs ? c : obs + c));      // c >= obs: action column (c - obs) sits at 2*obs + (c - obs)
    };
    __nv_bfloat16 *q = X.hi + (int64_t)xrow * X.ld;
    constexpr int kU = 4;
    for (int c0 = 2 * lane; c0 < ncols; c0 += 64 * kU) {
        float x0[kU], x1[kU];
#pragma unroll
        for (int u = 0; u < kU; u++) {
            const int c = c0 + 64 * u;
            x0[u] = c < ncols ? src(c) : 0.f;
            x1[u] = c + 1 < ncols ? src(c + 1) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < kU; u++) {
            const int c = c0 + 64 * u;
            if (c >= ncols) continue;
            uint32_t hi, lo;
            split_pack2(x0[u], x1[u], hi, lo);
            *reinterpret_cast<uint32_t *>(q + c) = hi;
            *reinterpret_cast<uint32_t *>(q + c + X.plane) = lo;
        }
    }
}

// T_SAMPLE: one warp per sampled row
__device__ __forceinline__ void task_sample(const SampleArgs &t, int tile, const Program &P, int agent, const float *scalars, uint64_t seed) {
    const int B = t.B, A = t.A, obs = t.obs;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = tile * (kThreads / 32) + warp;
    if (j >= 2 * B) return;
    const float *head = resolve(t.head, P.bases, agent) + (int64_t)j * 2 * A;
    float *eps = resolve(t.eps, P.bases, agent);
    const Pm X = resolve_pm(t.x, P.bases, agent);
    const int xrow = j < B ? j : 2 * B + (j - B);
    const uint32_t step = (uint32_t)__float_as_int(ldcg(scalars + SC_N_UPDATES));
    float lp = 0.f;
    for (int a = lane; a < A; a += 32) {
        float e;
        if (t.device_eps) {   // production mode: draw on device and keep the draw for the backward pass
            e = philox_normal(seed, (uint32_t)agent, step, (uint32_t)j, (uint32_t)a);
            eps[(int64_t)j * A + a] = e;
        } else {
            e = ldcg(eps + (int64_t)j * A + a);
        }
        const SampleElem s = sample_elem(ldcg(head + a), ldcg(head + A + a), e, t.scale, t.bias);
        pm_store(X, xrow, obs + a, s.action);
        lp += s.logp;
    }
    lp = warp_sum(lp);
    if (lane == 0) resolve(t.logp, P.bases, agent)[j] = lp;
}

// dot product of one PM activation row with an fp32 weight vector (H % 8 == 0): 8 elements per lane per trip
__device__ __forceinline__ float row_dot(const Pm &h, const float *w, int64_t row, int n, int lane) {
    float s = 0.f;
    for (int j = lane * 8; j < n; j += 256) {
        float hv[8];
        pm_load8(h, row, j, hv);
        const float4 w0 = __ldcg(reinterpret_cast<const float4 *>(w + j)), w1 = __ldcg(reinterpret_cast<const float4 *>(w + j + 4));
        s += hv[0] * w0.x + hv[1] * w0.y + hv[2] * w0.z + hv[3] * w0.w + hv[4] * w1.x + hv[5] * w1.y + hv[6] * w1.z + hv[7] * w1.w;
    }
    return warp_sum(s);
}

// dL/dh of the last hidden layer of a critic: dq[b] * w_out[n] * relu'(h[b,n]), written as a PM row (H % 8 == 0)
__device__ __forceinline__ void write_dh_last(const Pm &dh, const Pm &h, const float *w_out, int64_t row, int n, int lane, float dq) {
    for (int j = lane * 8; j < n; j += 256) {
        const uint4 hh = __ldcg(reinterpret_cast<const uint4 *>(h.hi + row * h.ld + j));     // sign of the activation: hi plane
        const uint32_t hw[4] = {hh.x, hh.y, hh.z, hh.w};
        const float4 w0 = __ldcg(reinterpret_cast<const float4 *>(w_out + j)), w1 = __ldcg(reinterpret_cast<const float4 *>(w_out + j + 4));
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float g0 = bf16_bits_to_float(hw[i] & 0xFFFFu) > 0.f ? dq * wv[2 * i] : 0.f;
            const float g1 = bf16_bits_to_float(hw[i] >> 16) > 0.f ? dq * wv[2 * i + 1] : 0.f;
            split_pack2(g0, g1, hi[i], lo[i]);
        }
        __nv_bfloat16 *q = dh.hi + row * dh.ld + j;
        *reinterpret_cast<uint4 *>(q) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4 *>(q + dh.plane) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

// four rows at once (throughput programs): the loads of all four rows of a trip are in flight together, the weights are read once
__device__ __forceinline__ void row_dot4(const Pm &h, const float *w, const int64_t (&row)[4], const bool (&on)[4], int n, int lane, float (&out)[4]) {
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j = lane * 8; j < n; j += 256) {
        uint4 hh[4], ll[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            hh[i] = ll[i] = make_uint4(0u, 0u, 0u, 0u);
            if (on[i]) {
                const __nv_bfloat16 *q = h.hi + row[i] * h.ld + j;
                hh[i] = __ldcg(reinterpret_cast<const uint4 *>(q));
                ll[i] = __ldcg(reinterpret_cast<const uint4 *>(q + h.plane));
            }
        }
        const float4 w0 = __ldcg(reinterpret_cast<const float4 *>(w + j)), w1 = __ldcg(reinterpret_cast<const float4 *>(w + j + 4));
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint32_t hw[4] = {hh[i].x, hh[i].y, hh[i].z, hh[i].w}, lw[4] = {ll[i].x, ll[i].y, ll[i].z, ll[i].w};
            float hv[8];
#pragma unroll
            for (int c = 0; c < 4; c++) {      // same value reconstruction and the same order of the 8 products as row_dot / pm_load8
                hv[2 * c] = bf16_bits_to_float(hw[c] & 0xFFFFu) + bf16_bits_to_float(lw[c] & 0xFFFFu);
                hv[2 * c + 1] = bf16_bits_to_float(hw[c] >> 16) + bf16_bits_to_float(lw[c] >> 16);
            }
            s[i] += hv[0] * wv[0] + hv[1] * wv[1] + hv[2] * wv[2] + hv[3] * wv[3] + hv[4] * wv[4] + hv[5] * wv[5] + hv[6] * wv[6] + hv[7] * wv[7];
        }
    }
#pragma unroll
    for (int i = 0; i < 4; i++) out[i] = warp_sum(s[i]);
}
__device__ __forceinline__ void write_dh_last4(const Pm &dh, const Pm &h, const float *w_out, const int64_t (&row)[4], const bool (&on)[4], int n, int lane, const float (&dq)[4]) {
    for (int j = lane * 8; j < n; j += 256) {
        uint4 hh[4];
#pragma unroll
        for (int i = 0; i < 4; i++) hh[i] = on[i] ? __ldcg(reinterpret_cast<const uint4 *>(h.hi + row[i] * h.ld + j)) : make_uint4(0u, 0u, 0u, 0u);
        const float4 w0 = __ldcg(reinterpret_cast<const float4 *>(w_out + j)), w1 = __ldcg(reinterpret_cast<const float4 *>(w_out + j + 4));
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int i = 0; i < 4; i++) {
            if (!on[i]) continue;
            const uint32_t hw[4] = {hh[i].x, hh[i].y, hh[i].z, hh[i].w};
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const float g0 = bf16_bits_to_float(hw[c] & 0xFFFFu) > 0.f ? dq[i] * wv[2 * c] : 0.f;
                const float g1 = bf16_bits_to_float(hw[c] >> 16) > 0.f ? dq[i] * wv[2 * c + 1] : 0.f;
                split_pack2(g0, g1, hi[c], lo[c]);
            }
            __nv_bfloat16 *q = dh.hi + row[i] * dh.ld + j;
            *reinterpret_cast<uint4 *>(q) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4 *>(q + dh.plane) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
    }
}

// The two loss tasks work on R batch rows per tile: R = 4 (latency programs: 4 warps per row, one per network, 64
// tiles at B = 256) or R = 16 (throughput programs: a warp takes one network for 4 rows, all of their loads in flight together;
// four times fewer dependent round trips per row).  Warp w handles the pairs (row, net) = (w / 4 + 4 j, w % 4), j < R / 4.
constexpr int kLossRows = 4, kLossRowsMax = 16;

// T_TARGET_LOSS: Bellman target + critic MSE terms + dL/dq   (sac_imp.py:92-105).
// Warp (row, k) forms the output-layer dot product of net k for its rows, one thread per row then does the scalar arithmetic,
// the warps of nets 2, 3 (q1, q2) finally write dL/dh of the last hidden layer.
__device__ __forceinline__ void task_target_loss(const TargetLossArgs &t, int tile, const Program &P, int agent, const float *scalars, float *smem) {
    const int B = t.B, H = t.H, R = t.R, nj = R >> 2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int k = warp & 3, r_w = warp >> 2;
    float *sq = smem, *sd = smem + 4 * kLossRowsMax, *sl = sd + 2 * kLossRowsMax;      // dots [R][4 nets], dq [R][2], loss terms [R][2]
    const Pm h = resolve_pm(t.h[k], P.bases, agent);
    const float *w = resolve(t.w_out[k], P.bases, agent);
    // the row's scalars are fetched by its scalar thread BEFORE the dot products, so their latency hides behind them
    float pre_bias[4] = {0.f, 0.f, 0.f, 0.f}, pre_alpha = 0.f, pre_gamma = 0.f, pre_logp = 0.f, pre_r = 0.f, pre_d = 0.f, pre_w = 1.f;
    if ((int)threadIdx.x < R && tile * R + (int)threadIdx.x < B) {
        const int br = tile * R + threadIdx.x;
        for (int j = 0; j < 4; j++) pre_bias[j] = ldcg(resolve(t.b_out[j], P.bases, agent));
        const int n_upd = __float_as_int(ldcg(scalars + SC_N_UPDATES));
        pre_alpha = ldcg(scalars + SC_ALPHA0 + (n_upd & 1));
        pre_gamma = ldcg(scalars + SC_GAMMA);
        const float *isw = resolve(t.is_weights, P.bases, agent);
        pre_logp = ldcg(resolve(t.logp_next, P.bases, agent) + br);
        pre_r = ldcg(resolve(t.r, P.bases, agent) + br);
        pre_d = ldcg(resolve(t.d, P.bases, agent) + br);
        if (isw) pre_w = ldcg(isw + br);
    }
    int64_t rows4[4];
    bool on4[4];
#pragma unroll
    for (int j = 0; j < 4; j++) { rows4[j] = tile * R + r_w + 4 * j; on4[j] = j < nj && rows4[j] < B; }
    if (nj == 4) {
        float q4[4];
        row_dot4(h, w, rows4, on4, H, lane, q4);
        if (lane == 0) for (int j = 0; j < 4; j++) sq[(r_w + 4 * j) * 4 + k] = on4[j] ? q4[j] : 0.f;
    } else {
        const int b = tile * R + r_w;
        const float q = b < B ? row_dot(h, w, b, H, lane) : 0.f;
        if (lane == 0) sq[r_w * 4 + k] = q;
    }
    __syncthreads();
    if ((int)threadIdx.x < R) {
        const int r = threadIdx.x, br = tile * R + r;
        float l1 = 0.f, l2 = 0.f, dq1 = 0.f, dq2 = 0.f;
        if (br < B) {
            float qq[4];
            for (int j = 0; j < 4; j++) qq[j] = sq[r * 4 + j] + pre_bias[j];
            const float alpha = pre_alpha;
            const float qn = fminf(qq[0], qq[1]);
            const float vt = qn - alpha * pre_logp;                                   // sac_imp.py:97
            const float yy = pre_r + (1.f - pre_d) * pre_gamma * vt;                   // :98
            const float wgt = pre_w;
            const float e1 = qq[2] - yy, e2 = qq[3] - yy;
            dq1 = 2.f * wgt * e1 / (float)B;                                                                          // d mean((q-y)^2) / dq
            dq2 = 2.f * wgt * e2 / (float)B;
            resolve(t.y, P.bases, agent)[br] = yy;
            resolve(t.dq[0], P.bases, agent)[br] = dq1;
            resolve(t.dq[1], P.bases, agent)[br] = dq2;
            resolve(t.td, P.bases, agent)[br] = fabsf(e1);
            l1 = wgt * e1 * e1; l2 = wgt * e2 * e2;
        }
        sd[2 * r] = dq1; sd[2 * r + 1] = dq2; sl[2 * r] = l1; sl[2 * r + 1] = l2;
    }
    __syncthreads();
    if (k >= 2) {
        const Pm dh = resolve_pm(t.dh[k - 2], P.bases, agent);
        if (nj == 4) {
            float dq4[4];
            for (int j = 0; j < 4; j++) dq4[j] = sd[2 * (r_w + 4 * j) + (k - 2)];
            write_dh_last4(dh, h, w, rows4, on4, H, lane, dq4);
        } else if (on4[0]) {
            write_dh_last(dh, h, w, rows4[0], H, lane, sd[2 * r_w + (k - 2)]);
        }
    }
    if ((int)threadIdx.x < nj) {      // partials per group of kLossRows rows, whatever R is: T_FINISH adds the same sequence of numbers
        const int sub = threadIdx.x;
        float s1 = 0.f, s2 = 0.f;
        for (int i = kLossRows * sub; i < kLossRows * (sub + 1); i++) { s1 += sl[2 * i]; s2 += sl[2 * i + 1]; }
        float *part = resolve(t.partials, P.bases, agent);
        part[2 * (tile * nj + sub)] = s1; part[2 * (tile * nj + sub) + 1] = s2;
    }
    __syncthreads();
}

// T_ACTOR_LOSS: policy-loss terms and min-Q routing (sac_imp.py:117-121).  Same tiling: the warps of "nets" 0, 1 form the two dot
// products, those of 2, 3 write dL/dh of the last hidden layer of q1, q2.
__device__ __forceinline__ void task_actor_loss(const ActorLossArgs &t, int tile, const Program &P, int agent, const float *scalars, float *smem) {
    const int B = t.B, H = t.H, R = t.R, nj = R >> 2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int k = warp & 3, r_w = warp >> 2;
    float *sq = smem, *sd = smem + 4 * kLossRowsMax, *sl = sd + 2 * kLossRowsMax;
    const Pm h = resolve_pm(t.h[k & 1], P.bases, agent);
    const float *w = resolve(t.w_out[k & 1], P.bases, agent);
    float pre_b1 = 0.f, pre_b2 = 0.f, pre_alpha = 0.f, pre_ent = 0.f, pre_logp = 0.f;      // fetched before the dot products (latency hidden)
    if ((int)threadIdx.x < R && tile * R + (int)threadIdx.x < B) {
        pre_b1 = ldcg(resolve(t.b_out[0], P.bases, agent)); pre_b2 = ldcg(resolve(t.b_out[1], P.bases, agent));
        const int n_upd = __float_as_int(ldcg(scalars + SC_N_UPDATES));
        pre_alpha = ldcg(scalars + SC_ALPHA0 + (n_upd & 1));
        pre_ent = ldcg(scalars + SC_TARGET_ENTROPY);
        pre_logp = ldcg(resolve(t.logp, P.bases, agent) + tile * R + threadIdx.x);
    }
    int64_t rows4[4];
    bool on4[4];
#pragma unroll
    for (int j = 0; j < 4; j++) { rows4[j] = tile * R + r_w + 4 * j; on4[j] = j < nj && rows4[j] < B; }
    if (k < 2) {
        if (nj == 4) {
            float q4[4];
            row_dot4(h, w, rows4, on4, H, lane, q4);
            if (lane == 0) for (int j = 0; j < 4; j++) sq[(r_w + 4 * j) * 4 + k] = on4[j] ? q4[j] : 0.f;
        } else {
            const int b = tile * R + r_w;
            const float q = b < B ? row_dot(h, w, b, H, lane) : 0.f;
            if (lane == 0) sq[r_w * 4 + k] = q;
        }
    }
    __syncthreads();
    if ((int)threadIdx.x < R) {
        const int r = threadIdx.x, br = tile * R + r;
        float pl = 0.f, ent = 0.f, d1 = 0.f, d2 = 0.f;
        if (br < B) {
            const float q1 = sq[r * 4] + pre_b1, q2 = sq[r * 4 + 1] + pre_b2;
            const float alpha = pre_alpha;
            const float l = pre_logp;
            pl = alpha * l - fminf(q1, q2);                                          // sac_imp.py:119-121
            const float sel = q1 < q2 ? 1.f : (q1 == q2 ? 0.5f : 0.f);               // torch.minimum backward
            d1 = -sel / (float)B;
            d2 = -(1.f - sel) / (float)B;
            ent = l + pre_ent;
        }
        sd[2 * r] = d1; sd[2 * r + 1] = d2; sl[2 * r] = pl; sl[2 * r + 1] = ent;
    }
    __syncthreads();
    if (k >= 2) {
        const Pm dh = resolve_pm(t.dh[k - 2], P.bases, agent);
        if (nj == 4) {
            float dq4[4];
            for (int j = 0; j < 4; j++) dq4[j] = sd[2 * (r_w + 4 * j) + (k - 2)];
            write_dh_last4(dh, h, w, rows4, on4, H, lane, dq4);
        } else if (on4[0]) {
            write_dh_last(dh, h, w, rows4[0], H, lane, sd[2 * r_w + (k - 2)]);
        }
    }
    if ((int)threadIdx.x < nj) {
        const int sub = threadIdx.x;
        float s1 = 0.f, s2 = 0.f;
        for (int i = kLossRows * sub; i < kLossRows * (sub + 1); i++) { s1 += sl[2 * i]; s2 += sl[2 * i + 1]; }
        float *part = resolve(t.partials, P.bases, agent);
        part[2 * (tile * nj + sub)] = s1; part[2 * (tile * nj + sub) + 1] = s2;
    }
    __syncthreads();
}

// T_SAMPLE_BWD: closed form of SURVEY 3.3, one thread per (row, action) element
__device__ __forceinline__ void task_sample_bwd(const SampleBwdArgs &t, int tile, const Program &P, int agent, const float *scalars) {
    const int B = t.B, A = t.A;
    const int idx = tile * kThreads + threadIdx.x;
    if (idx >= B * A) return;
    const int b = idx / A, a = idx % A;
    const int n_upd = __float_as_int(ldcg(scalars + SC_N_UPDATES));
    const float alpha = ldcg(scalars + SC_ALPHA0 + (n_upd & 1));
    const float *head = resolve(t.head, P.bases, agent) + (int64_t)b * 2 * A;
    const float eps = ldcg(resolve(t.eps, P.bases, agent) + idx);
    const SampleElem s = sample_elem(ldcg(head + a), ldcg(head + A + a), eps, t.scale, t.bias);
    const float da = ldcg(resolve(t.da[0], P.bases, agent) + idx) + ldcg(resolve(t.da[1], P.bases, agent) + idx);
    const float sc = t.scale, omy2 = 1.f - s.y * s.y, aB = alpha / (float)B;
    const float g_u = da * sc * omy2 + aB * (2.f * sc * s.y * omy2) / (sc * omy2 + kSquashEps);
    const Pm g = resolve_pm(t.g_head, P.bases, agent);
    pm_store(g, b, a, g_u);
    pm_store(g, b, A + a, (g_u * s.std * eps - aB) * s.in_range);
}

// Column sums over batch rows for a tile of kColsumCols = 64 columns: a thread owns 8 consecutive columns (one 16-byte load per
// bf16 plane and row) of row lane tid / 8, rows lane, lane + 64, ... (4 rows in flight); the four row lanes of a warp are combined
// with shuffles, the 16 warps through shared memory in warp order: a fixed summation order.  Result valid for threadIdx.x < 64.
constexpr int kColsumCols = 64;
constexpr int kColsumSmem = (kThreads / 32) * kColsumCols;      // floats of shared memory
// kDeep = false (the two-CTAs-per-SM builds, 64 registers): at most 4 rows in flight per thread, the second resident CTA supplies the rest
template <bool kDeep, class F>
__device__ __forceinline__ float colsum64(int r0, int r1, float *smem, F load8) {
    const int cg = threadIdx.x & 7, rl = threadIdx.x >> 3, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; j++) acc[j] = 0.f;
    int b = r0 + rl;
    for (; kDeep && b + 7 * 64 < r1; b += 8 * 64) {      // long batches: 8 rows (16 loads of 16 bytes) in flight per thread
        float v[8][8];
#pragma unroll
        for (int u = 0; u < 8; u++) load8(b + 64 * u, cg * 8, v[u]);
#pragma unroll
        for (int u = 0; u < 8; u++)
#pragma unroll
            for (int j = 0; j < 8; j++) acc[j] += v[u][j];
    }
    for (; b + 3 * 64 < r1; b += 4 * 64) {
        float v[4][8];
#pragma unroll
        for (int u = 0; u < 4; u++) load8(b + 64 * u, cg * 8, v[u]);
#pragma unroll
        for (int u = 0; u < 4; u++)
#pragma unroll
            for (int j = 0; j < 8; j++) acc[j] += v[u][j];
    }
    for (; b < r1; b += 64) {
        float v[8];
        load8(b, cg * 8, v);
#pragma unroll
        for (int j = 0; j < 8; j++) acc[j] += v[j];
    }
#pragma unroll
    for (int j = 0; j < 8; j++) {
        acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 8);
        acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 16);
    }
    if (lane < 8) {
#pragma unroll
        for (int j = 0; j < 8; j++) smem[warp * kColsumCols + cg * 8 + j] = acc[j];
    }
    __syncthreads();
    float tot = 0.f;
    if (threadIdx.x < kColsumCols)
        for (int w = 0; w < kThreads / 32; w++) tot += smem[w * kColsumCols + threadIdx.x];
    __syncthreads();
    return tot;
}

// Adam on one element whose optimizer state was fetched before the column sum (the two latencies overlap); same arithmetic as adam_element
struct PreState { float w, m, v, wt; };
__device__ __forceinline__ PreState prefetch_state(bool on, const float *w, const float *m, const float *v, const float *wt) {
    PreState s{0.f, 0.f, 0.f, 0.f};
    if (on) { s.w = __ldcg(w); s.m = __ldcg(m); s.v = __ldcg(v); if (wt) s.wt = __ldcg(wt); }
    return s;
}
__device__ __forceinline__ void adam_prefetched(float g, PreState s, float *w, float *m, float *v, float *wt, float ss, float bs, float tau) {
    const float mm = s.m + (1.0f - kBeta1) * (g - s.m);
    const float vv = s.v * kBeta2 + (1.0f - kBeta2) * g * g;
    const float denom = sqrtf(vv) / bs + kAdamEps;
    const float ww = s.w - ss * (mm / denom);
    *m = mm; *v = vv; *w = ww;
    if (wt) *wt = s.wt * (1.0f - tau) + ww * tau;
}
// gradient of a column-sum task: exported (optionally accumulated over row chunks with atomics: data-parallel programs, whose
// gradient slab is zeroed at the start of the step) and / or applied
__device__ __forceinline__ void colsum_finish(float g, bool chunked, float *ge, int apply, PreState st, float *w, float *m, float *v, float *wt,
                                              float ss, float bs, float tau) {
    if (ge) { if (chunked) atomicAdd(ge, g); else *ge = g; }
    if (apply) adam_prefetched(g, st, w, m, v, wt, ss, bs, tau);
}

// T_OUT_ADAM tiles: [row chunk][64-column tile] for the weight gradient, then one bias tile per row chunk
template <bool kDeep = true>
__device__ __forceinline__ void task_out_adam(const OutAdamArgs &t, int tile, const Program &P, int agent, const float *scalars, float *smem) {
    const int B = t.B, H = t.H, R = t.chunk_rows, n_ct = cdiv(H, kColsumCols), n_rc = cdiv(B, R);
    const float *dq = resolve(t.dq, P.bases, agent);
    // the Adam factors and the Polyak rate (one L2 line): ahead of the column sum, where their latency hides; the light build
    // (kDeep = false, 64 registers) loads them behind it instead, as task_bias_adam does -- holding them across it costs that build spills
    float ss = 0.f, bs = 0.f, tau = 0.f;
    if constexpr (kDeep) { adam_factors_cached(scalars, t.w.step_slot, ss, bs); tau = __ldcg(scalars + SC_TAU); }
    if (tile >= n_ct * n_rc) {      // bias tile of row chunk tile - n_ct * n_rc: db = sum_b dq[b] (32 lane partials, then the warp tree)
        const int rc = tile - n_ct * n_rc, r0 = rc * R, r1 = min(B, r0 + R);
        if (threadIdx.x < 32) {
            float gb = 0.f;
            for (int b = r0 + threadIdx.x; b < r1; b += 32) gb += ldcg(dq + b);
            gb = warp_sum(gb);
            if (threadIdx.x == 0) {
                const AdamArgs &a = t.b;
                if constexpr (!kDeep) { adam_factors_cached(scalars, a.step_slot, ss, bs); tau = __ldcg(scalars + SC_TAU); }
                float *w = resolve(a.w, P.bases, agent), *m = resolve(a.m, P.bases, agent), *v = resolve(a.v, P.bases, agent);
                float *wt = resolve(a.wt, P.bases, agent), *ge = resolve(a.gexp, P.bases, agent);
                colsum_finish(gb, n_rc > 1, ge, a.apply, prefetch_state(a.apply != 0, w, m, v, wt), w, m, v, wt, ss, bs, tau);
            }
        }
        return;
    }
    const int ct = tile % n_ct, rc = tile / n_ct, r0 = rc * R, r1 = min(B, r0 + R);
    const int n = ct * kColsumCols + threadIdx.x;
    const Pm h = resolve_pm(t.h, P.bases, agent);
    const bool owner = threadIdx.x < kColsumCols && n < H;
    const AdamArgs &a = t.w;
    float *w = resolve(a.w, P.bases, agent) + n, *m = resolve(a.m, P.bases, agent) + n, *v = resolve(a.v, P.bases, agent) + n;
    float *wt = resolve(a.wt, P.bases, agent), *ge = resolve(a.gexp, P.bases, agent);
    const PreState st = prefetch_state(owner && a.apply, w, m, v, wt ? wt + n : nullptr);
    const int c0 = ct * kColsumCols;
    const float g = colsum64<kDeep>(r0, r1, smem, [&](int b, int c, float (&out)[8]) {
        if (c0 + c < h.ld) {
            pm_load8(h, b, c0 + c, out);
            const float d = ldcg(dq + b);
#pragma unroll
            for (int j = 0; j < 8; j++) out[j] *= d;
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) out[j] = 0.f;
        }
    });
    if (owner) {
        if constexpr (!kDeep) { adam_factors_cached(scalars, a.step_slot, ss, bs); tau = __ldcg(scalars + SC_TAU); }
        colsum_finish(g, n_rc > 1, ge ? ge + n : nullptr, a.apply, st, w, m, v, wt ? wt + n : nullptr, ss, bs, tau);
    }
}

// T_BIAS_ADAM tiles: [row chunk][64-column tile]
template <bool kDeep = true>
__device__ __forceinline__ void task_bias_adam(const ColsumAdamArgs &t, int tile, const Program &P, int agent, const float *scalars, float *smem) {
    const int B = t.B, N = t.N, R = t.chunk_rows, n_ct = cdiv(N, kColsumCols), n_rc = cdiv(B, R);
    const int ct = tile % n_ct, rc = tile / n_ct, r0 = rc * R, r1 = min(B, r0 + R);
    const int n = ct * kColsumCols + threadIdx.x;
    const Pm dh = resolve_pm(t.src, P.bases, agent);
    const bool owner = threadIdx.x < kColsumCols && n < N;
    const AdamArgs &a = t.adam;
    float *w = resolve(a.w, P.bases, agent) + n, *m = resolve(a.m, P.bases, agent) + n, *v = resolve(a.v, P.bases, agent) + n;
    float *bt = resolve(a.wt, P.bases, agent), *ge = resolve(a.gexp, P.bases, agent);
    const PreState st = prefetch_state(owner && a.apply, w, m, v, bt ? bt + n : nullptr);
    const int c0 = ct * kColsumCols;
    const float g = colsum64<kDeep>(r0, r1, smem, [&](int b, int c, float (&out)[8]) {
        if (c0 + c < dh.ld) pm_load8(dh, b, c0 + c, out);
        else {
#pragma unroll
            for (int j = 0; j < 8; j++) out[j] = 0.f;
        }
    });
    if (owner) {
        float ss, bs;
        adam_factors_cached(scalars, a.step_slot, ss, bs);
        const float tau = __ldcg(scalars + SC_TAU);
        colsum_finish(g, n_rc > 1, ge ? ge + n : nullptr, a.apply, st, w, m, v, bt ? bt + n : nullptr, ss, bs, tau);
    }
}

// ---- opt-in LayerNorm variant (no counterpart in the reference: DESIGN.md) --------------------------------------------------------
// One warp per row, the row (H <= 1024 values, H % 8 == 0) held in registers: 8 consecutive elements per lane and trip.
constexpr int kLnRows = kThreads / 32, kLnMaxH = 1024, kLnTrips = kLnMaxH / 256;
__device__ __forceinline__ void pm_store8(const Pm &p, int64_t row, int col, const float (&x)[8]) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int i = 0; i < 4; i++) split_pack2(x[2 * i], x[2 * i + 1], hi[i], lo[i]);
    __nv_bfloat16 *q = p.hi + row * p.ld + col;
    *reinterpret_cast<uint4 *>(q) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4 *>(q + p.plane) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}
__device__ __forceinline__ void load8f(const float *p, float (&out)[8]) {
    const float4 a = __ldcg(reinterpret_cast<const float4 *>(p)), b = __ldcg(reinterpret_cast<const float4 *>(p + 4));
    out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w; out[4] = b.x; out[5] = b.y; out[6] = b.z; out[7] = b.w;
}
// T_LN_FWD: h = relu((z - mean) * rstd * gamma + beta), mean / biased variance over the H columns of the row (torch.nn.LayerNorm)
__device__ __forceinline__ void task_ln_fwd(const LnFwdArgs &t, int tile, const Program &P, int agent) {
    const int rows = t.rows, H = t.H, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = tile * kLnRows + warp;
    if (row >= rows) return;      // warp-uniform
    const float *z = resolve(t.z, P.bases, agent) + (int64_t)row * H, *gam = resolve(t.gamma, P.bases, agent), *bet = resolve(t.beta, P.bases, agent);
    float v[kLnTrips][8];
    float s = 0.f;
#pragma unroll
    for (int u = 0; u < kLnTrips; u++) {
        const int j = u * 256 + lane * 8;
        if (j < H) {
            load8f(z + j, v[u]);
#pragma unroll
            for (int i = 0; i < 8; i++) s += v[u][i];
        }
    }
    const float mean = warp_sum(s) / (float)H;
    float q = 0.f;
#pragma unroll
    for (int u = 0; u < kLnTrips; u++)
        if (u * 256 + lane * 8 < H) {
#pragma unroll
            for (int i = 0; i < 8; i++) { const float d = v[u][i] - mean; q += d * d; }
        }
    const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)H + t.eps);
    const Pm h = resolve_pm(t.h, P.bases, agent);
#pragma unroll
    for (int u = 0; u < kLnTrips; u++) {
        const int j = u * 256 + lane * 8;
        if (j < H) {
            float g[8], b[8], y[8];
            load8f(gam + j, g); load8f(bet + j, b);
#pragma unroll
            for (int i = 0; i < 8; i++) y[i] = fmaxf((v[u][i] - mean) * rstd * g[i] + b[i], 0.f);
            pm_store8(h, row, j, y);
        }
    }
    if (lane == 0) { float *st = resolve(t.stats, P.bases, agent) + 2 * (int64_t)row; st[0] = mean; st[1] = rstd; }
}
// T_LN_BWD: dpre = gradient at the LayerNorm output (ReLU mask already applied by the producer) -> dz = gradient at the Linear output:
//   g = dpre * gamma ; xhat = (z - mean) * rstd ; dz = rstd * (g - mean_j(g) - xhat * mean_j(g * xhat)) ; gg = dpre * xhat (its column
//   sums over the batch are dgamma, those of dpre are dbeta: T_BIAS_ADAM tasks)
__device__ __forceinline__ void task_ln_bwd(const LnBwdArgs &t, int tile, const Program &P, int agent) {
    const int rows = t.rows, H = t.H, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = tile * kLnRows + warp;
    if (row >= rows) return;
    const float *z = resolve(t.z, P.bases, agent) + (int64_t)row * H, *gam = resolve(t.gamma, P.bases, agent);
    const float *st = resolve(t.stats, P.bases, agent) + 2 * (int64_t)row;
    const float mean = ldcg(st), rstd = ldcg(st + 1);
    const Pm dpre = resolve_pm(t.dpre, P.bases, agent), dz = resolve_pm(t.dz, P.bases, agent);
    const bool want_gg = !is_null(t.gg.base);
    float g[kLnTrips][8], xh[kLnTrips][8];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int u = 0; u < kLnTrips; u++) {
        const int j = u * 256 + lane * 8;
        if (j < H) {
            float d[8], zz[8], gm[8];
            pm_load8(dpre, row, j, d); load8f(z + j, zz); load8f(gam + j, gm);
#pragma unroll
            for (int i = 0; i < 8; i++) { xh[u][i] = (zz[i] - mean) * rstd; g[u][i] = d[i] * gm[i]; s1 += g[u][i]; s2 += g[u][i] * xh[u][i]; }
            if (want_gg) {
                float gg[8];
#pragma unroll
                for (int i = 0; i < 8; i++) gg[i] = d[i] * xh[u][i];
                pm_store8(resolve_pm(t.gg, P.bases, agent), row, j, gg);
            }
        }
    }
    const float m1 = warp_sum(s1) / (float)H, m2 = warp_sum(s2) / (float)H;
#pragma unroll
    for (int u = 0; u < kLnTrips; u++) {
        const int j = u * 256 + lane * 8;
        if (j < H) {
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; i++) o[i] = rstd * (g[u][i] - m1 - xh[u][i] * m2);
            pm_store8(dz, row, j, o);
        }
    }
}

// T_FINISH (one thread): finalise the loss scalars from the per-tile partials (fixed order), the temperature step
// (sac_imp.py:128-135) and the optimizer step counters (+1 each, sac_imp.py:109,113,125,134).
__device__ __forceinline__ void task_finish(const FinishArgs &t, const Program &P, int agent, float *scalars, float *smem) {
    const int nt = t.n_part;
    const float Bf = t.B;
    const float *cp = resolve(t.critic_part, P.bases, agent), *ap = resolve(t.actor_part, P.bases, agent);
    // the agent's scalar block is read ONCE into shared memory, edited there and written back at the end: the serial part below
    // would otherwise be a chain of ~8 dependent L2 round trips
    __shared__ float sc[32];
    if (threadIdx.x < 32) sc[threadIdx.x] = ldcg(scalars + threadIdx.x);
    // deterministic two-level sum: 128 threads each add a contiguous run of tile partials in tile order (one tile
    // each while nt <= 128), thread 0 then adds the 128 run sums in order
    constexpr int kRuns = kThreads / 4;
    if ((int)threadIdx.x < kRuns) {
        const int c = cdiv(nt, kRuns), i0 = threadIdx.x * c, i1 = min(nt, i0 + c);
        float a1 = 0.f, a2 = 0.f, b1 = 0.f, b2 = 0.f;
        int i = i0;
        for (; i + 7 < i1; i += 8) {      // large batches: eight partial pairs in flight (same order of the additions)
            float2 c8[8], d8[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                c8[u] = cp ? __ldcg(reinterpret_cast<const float2 *>(cp) + i + u) : make_float2(0.f, 0.f);
                d8[u] = ap ? __ldcg(reinterpret_cast<const float2 *>(ap) + i + u) : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 8; u++) { if (cp) { a1 += c8[u].x; a2 += c8[u].y; } if (ap) { b1 += d8[u].x; b2 += d8[u].y; } }
        }
        for (; i < i1; i++) {
            if (cp) { a1 += ldcg(cp + 2 * i); a2 += ldcg(cp + 2 * i + 1); }
            if (ap) { b1 += ldcg(ap + 2 * i); b2 += ldcg(ap + 2 * i + 1); }
        }
        smem[threadIdx.x] = a1; smem[kRuns + threadIdx.x] = a2; smem[2 * kRuns + threadIdx.x] = b1; smem[3 * kRuns + threadIdx.x] = b2;
    }
    __syncthreads();
    // threads 32..35: the step counter of one optimizer each (+1, sac_imp.py:109,113,125,134) and its next bias corrections
    // from the host-built table with the agent's learning rate, formed while thread 0 works
    const int k = (int)threadIdx.x - 32;
    int new_step = 0;
    float2 fac = make_float2(0.f, 0.f);
    const bool bump = k >= 0 && k < 4 && t.bump[k];      // SC_STEP_POLICY, SC_STEP_Q1, SC_STEP_Q2, SC_STEP_ALPHA are consecutive
    if (bump) {
        new_step = __float_as_int(sc[SC_STEP_POLICY + k]) + 1;
        const AdamBias b = P.adam_table[min(new_step, kAdamTable - 1)];
        fac = make_float2(adam_step_size(sc[SC_LR], b.bc1), b.bc2_sqrt);
    }
    if (threadIdx.x == 0) {
        if (cp) {
            float s1 = 0.f, s2 = 0.f;
            for (int i = 0; i < kRuns; i++) { s1 += smem[i]; s2 += smem[kRuns + i]; }
            sc[SC_LOSS_Q1] = s1 / Bf; sc[SC_LOSS_Q2] = s2 / Bf;
        }
        if (ap) {
            float s1 = 0.f, s2 = 0.f;
            for (int i = 0; i < kRuns; i++) { s1 += smem[2 * kRuns + i]; s2 += smem[3 * kRuns + i]; }
            sc[SC_LOSS_PI] = s1 / Bf;
            const int n_upd = __float_as_int(sc[SC_N_UPDATES]);
            float alpha_next = sc[SC_ALPHA0 + (n_upd & 1)];
            if (t.auto_entropy) {
                const float la = sc[SC_LOG_ALPHA];
                const float g = -(s2 / Bf);                                      // d(-mean(log_alpha*(logp+H_t)))/dlog_alpha
                sc[SC_LOSS_ALPHA] = la * g;
                float *gexp = resolve(t.alpha_grad, P.bases, agent);
                if (gexp) *gexp = g;
                if (t.apply) {      // adam_element on the shared-memory copy (same arithmetic)
                    const float ss = sc[SC_FAC0 + 2 * (SC_STEP_ALPHA - SC_STEP_POLICY)], bs = sc[SC_FAC0 + 2 * (SC_STEP_ALPHA - SC_STEP_POLICY) + 1];
                    float mm = sc[SC_LOG_ALPHA_M], vv = sc[SC_LOG_ALPHA_V];
                    mm = mm + (1.0f - kBeta1) * (g - mm);
                    vv = vv * kBeta2 + (1.0f - kBeta2) * g * g;
                    const float denom = sqrtf(vv) / bs + kAdamEps;
                    sc[SC_LOG_ALPHA] = la - ss * (mm / denom);
                    sc[SC_LOG_ALPHA_M] = mm; sc[SC_LOG_ALPHA_V] = vv;
                }
                alpha_next = expf(sc[SC_LOG_ALPHA]);                            // self.alpha = self.log_alpha.exp()
            }
            if (t.apply) sc[SC_ALPHA0 + ((n_upd + 1) & 1)] = alpha_next;
        }
        if (t.bump_updates) {
            sc[SC_N_UPDATES] = __int_as_float(__float_as_int(sc[SC_N_UPDATES]) + 1);
            const int pos = __float_as_int(sc[SC_HIST_POS]);
            float *hist = resolve(t.loss_hist, P.bases, agent) + 4 * (pos % kLossHist);
            hist[0] = sc[SC_LOSS_Q1]; hist[1] = sc[SC_LOSS_Q2]; hist[2] = sc[SC_LOSS_PI]; hist[3] = sc[SC_LOSS_ALPHA];
            sc[SC_HIST_POS] = __int_as_float(pos + 1);
        }
        sc[SC_ERROR_FLAG] = __int_as_float(*reinterpret_cast<volatile int *>(P.error_flag));      // watchdog flags of the earlier stages
    }
    __syncthreads();      // thread 0 has read the current bias corrections
    if (bump) {
        sc[SC_STEP_POLICY + k] = __int_as_float(new_step);
        sc[SC_FAC0 + 2 * k] = fac.x; sc[SC_FAC0 + 2 * k + 1] = fac.y;
    }
    __syncthreads();
    if (threadIdx.x < 32) scalars[threadIdx.x] = sc[threadIdx.x];
    static_assert(SC_ERROR_FLAG == SC_LOSS_Q1 + 4, "losses and the flag are contiguous");
    if (P.host_losses && agent == 0 && threadIdx.x < 5) P.host_losses[threadIdx.x] = sc[SC_LOSS_Q1 + threadIdx.x];
}

}  // namespace sacb
