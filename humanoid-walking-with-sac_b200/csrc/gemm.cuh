// GEMM tile workers of the SAC update program.
//   gemm_tile_tc   : TMA -> shared memory (SWIZZLE_128B) -> tcgen05.mma kind::f16 on bf16 hi/lo operand pairs,
//                    fp32 accumulator in TMEM, fused epilogues (bias+ReLU, ReLU mask, Adam+Polyak+shadow refresh)
//   gemm_tile_ffma : fp32 FFMA tile on the same pair-matrix operands (checker of the tensor-core tile, strict mode)
// Both compute  C[M,N] = epilogue( A[M,K] * B[N,K]^T )  for one output tile of a Task.
#pragma once
#include "common.cuh"

namespace sacb {

__device__ __forceinline__ float ldcg(const float *p) { return __ldcg(p); }

// ---- bf16 pair helpers --------------------------------------------------------------------------------------
__device__ __forceinline__ float bf16_bits_to_float(uint32_t b16) { return __uint_as_float(b16 << 16); }
// x -> (hi, lo) with hi = bf16_rn(x), lo = bf16_rn(x - hi)
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16 &hi, __nv_bfloat16 &lo) {
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
__device__ __forceinline__ float pm_load(const Pm &p, int64_t row, int col) {
    const __nv_bfloat16 *q = p.hi + row * p.ld + col;
    return __bfloat162float(q[0]) + __bfloat162float(q[p.plane]);
}
__device__ __forceinline__ void pm_store(const Pm &p, int64_t row, int col, float x) {
    __nv_bfloat16 hi, lo;
    split_bf16(x, hi, lo);
    __nv_bfloat16 *q = p.hi + row * p.ld + col;
    q[0] = hi; q[p.plane] = lo;
}
// two floats -> packed bf16x2 hi word and lo word (element 0 in the low half)
__device__ __forceinline__ void split_pack2(float x0, float x1, uint32_t &hi, uint32_t &lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
    const float2 hf = __bfloat1622float2(h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x0 - hf.x, x1 - hf.y);
    hi = *reinterpret_cast<const uint32_t *>(&h);
    lo = *reinterpret_cast<const uint32_t *>(&l);
}
// 8 consecutive elements of a PM row (16 B per plane, 16 B aligned) -> floats
__device__ __forceinline__ void pm_load8(const Pm &p, int64_t row, int col, float (&out)[8]) {
    const __nv_bfloat16 *q = p.hi + row * p.ld + col;
    const uint4 h = __ldcg(reinterpret_cast<const uint4 *>(q));
    const uint4 l = __ldcg(reinterpret_cast<const uint4 *>(q + p.plane));
    const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        out[2 * i] = bf16_bits_to_float(hw[i] & 0xFFFFu) + bf16_bits_to_float(lw[i] & 0xFFFFu);
        out[2 * i + 1] = bf16_bits_to_float(hw[i] >> 16) + bf16_bits_to_float(lw[i] >> 16);
    }
}

// ---- resolved (per agent) epilogue arguments ------------------------------------------------------------------
struct EpiR {
    int epi, M, N;
    float *C; int ldc;
    Pm Cpm;
    const float *bias;
    Pm mask;
    float *w, *m, *v, *wt, *gexp;
    Pm shadow, shadow2, shadow_t;
    int shadow2_col0;
    int apply;
    float step_size, bc2_sqrt, inv_bc2_sqrt, tau;
};

// Adam bias corrections for step t (torch/optim/adam.py::_single_tensor_adam): python floats = double.  Double-precision
// pow is slow on this part, so it runs once per optimizer per update (T_FINISH) and the tiles read the cached pair.
__host__ inline AdamBias adam_bias(int step_before) {
    const double t = (double)(step_before + 1);
    AdamBias b;
    b.bc1 = 1.0 - pow((double)0.9, t);
    b.bc2_sqrt = (float)sqrt(1.0 - pow((double)0.999, t));
    b.pad = 0.f;
    return b;
}
// step size from the table entry: one correctly rounded float64 division, on the host and on the device alike
__host__ __device__ __forceinline__ float adam_step_size(float lr, double bc1) { return (float)((double)lr / bc1); }
__device__ __forceinline__ void adam_factors_cached(const float *scalars, int step_slot, float &step_size, float &bc2_sqrt) {
    const float2 f = __ldcg(reinterpret_cast<const float2 *>(scalars + SC_FAC0 + 2 * (step_slot - SC_STEP_POLICY)));
    step_size = f.x; bc2_sqrt = f.y;
}
// host side: the factors for the agent's own learning rate (SC_LR of the same block)
__host__ inline void adam_factors_store(float *scalars, int step_slot, int step) {
    const AdamBias b = adam_bias(step);
    scalars[SC_FAC0 + 2 * (step_slot - SC_STEP_POLICY)] = adam_step_size(scalars[SC_LR], b.bc1);
    scalars[SC_FAC0 + 2 * (step_slot - SC_STEP_POLICY) + 1] = b.bc2_sqrt;
}
// device side: the bias corrections come from the host-built table (float64 pow is very slow on this part)
__device__ __forceinline__ void adam_factors_store(float *scalars, int step_slot, int step, const AdamBias *table) {
    const AdamBias b = table[min(step, kAdamTable - 1)];
    scalars[SC_FAC0 + 2 * (step_slot - SC_STEP_POLICY)] = adam_step_size(scalars[SC_LR], b.bc1);
    scalars[SC_FAC0 + 2 * (step_slot - SC_STEP_POLICY) + 1] = b.bc2_sqrt;
}

// one Adam element update (+ Polyak, sac_imp.py:146-152); returns the new weight
__device__ __forceinline__ float adam_element(float g, float *w, float *m, float *v, float *wt, float *gexp, int apply,
                                              float step_size, float bc2_sqrt, float tau) {
    if (gexp) *gexp = g;
    if (!apply) return __ldcg(w);
    float mm = __ldcg(m), vv = __ldcg(v), ww = __ldcg(w);
    mm = mm + (1.0f - kBeta1) * (g - mm);                 // exp_avg.lerp_(grad, 1 - beta1)
    vv = vv * kBeta2 + (1.0f - kBeta2) * g * g;          // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float denom = sqrtf(vv) / bc2_sqrt + kAdamEps;
    ww = ww - step_size * (mm / denom);
    *m = mm; *v = vv; *w = ww;
    if (wt) *wt = __ldcg(wt) * (1.0f - tau) + ww * tau;  // target <- target*(1-tau) + param*tau
    return ww;
}

__device__ __forceinline__ void epilogue_element(const EpiR &e, int m, int n, float acc) {
    if (m >= e.M || n >= e.N) return;
    switch (e.epi) {
        case EPI_F32: e.C[(int64_t)m * e.ldc + n] = acc + (e.bias ? ldcg(e.bias + n) : 0.f); break;
        case EPI_BIAS_RELU: pm_store(e.Cpm, m, n, fmaxf(acc + ldcg(e.bias + n), 0.f)); break;
        case EPI_MASK: pm_store(e.Cpm, m, n, __bfloat162float(e.mask.hi[(int64_t)m * e.mask.ld + n]) > 0.f ? acc : 0.f); break;
        case EPI_ADAM: {
            const int64_t o = (int64_t)m * e.N + n;
            const float w1 = adam_element(acc, e.w + o, e.m + o, e.v + o, e.wt ? e.wt + o : nullptr, e.gexp ? e.gexp + o : nullptr,
                                          e.apply, e.step_size, e.bc2_sqrt, e.tau);
            if (e.shadow.hi && e.apply) pm_store(e.shadow, m, n, w1);
            if (e.shadow2.hi && e.apply && n >= e.shadow2_col0) pm_store(e.shadow2, m, n - e.shadow2_col0, w1);
        } break;
    }
}

__device__ __forceinline__ EpiR resolve_epilogue(const Task &t, const AgentBases &b, int agent, const float *scalars) {
    EpiR e;
    e.epi = t.epi; e.M = t.M; e.N = t.N;
    e.C = resolve(t.C, b, agent); e.ldc = t.ldc;
    e.Cpm = resolve_pm(t.Cpm, b, agent);
    e.bias = resolve(t.bias, b, agent);
    e.mask = resolve_pm(t.mask, b, agent);
    e.w = e.m = e.v = e.wt = e.gexp = nullptr; e.apply = 0; e.step_size = e.bc2_sqrt = e.inv_bc2_sqrt = 0.f; e.tau = 0.f;
    e.shadow.hi = nullptr; e.shadow.ld = 0; e.shadow.plane = 0;
    e.shadow2 = e.shadow; e.shadow_t = e.shadow; e.shadow2_col0 = 0;
    if (t.epi == EPI_ADAM) {
        e.w = resolve(t.adam.w, b, agent); e.m = resolve(t.adam.m, b, agent); e.v = resolve(t.adam.v, b, agent);
        e.wt = resolve(t.adam.wt, b, agent); e.gexp = resolve(t.adam.gexp, b, agent);
        e.shadow = resolve_pm(t.adam.shadow, b, agent);
        e.shadow2 = resolve_pm(t.adam.shadow2, b, agent); e.shadow2_col0 = t.adam.shadow2_col0;
        e.shadow_t = resolve_pm(t.adam.shadow_t, b, agent);
        e.apply = t.adam.apply; e.tau = __ldcg(scalars + SC_TAU);
        adam_factors_cached(scalars, t.adam.step_slot, e.step_size, e.bc2_sqrt);
        e.inv_bc2_sqrt = 1.0f / e.bc2_sqrt;
    }
    return e;
}

// value of the logical operand at (r, k); caller guarantees in-bounds
__device__ __forceinline__ float operand_at(const Pm &p, int mn_major, int r, int k) {
    return mn_major ? pm_load(p, k, r) : pm_load(p, r, k);
}

// ============================================================================================================
// fp32 FFMA tile: 64 x 64 x 16, 256 worker threads, 4x4 outputs per thread
// ============================================================================================================
__device__ __forceinline__ void gemm_tile_ffma(const Task &t, int tile, const AgentBases &bases, int agent,
                                               const float *scalars, float *smem) {
    const Pm A = resolve_pm(t.A.pm, bases, agent), B = resolve_pm(t.B.pm, bases, agent);
    const int a_mn = t.A.mn_major, b_mn = t.B.mn_major;
    const EpiR epi = resolve_epilogue(t, bases, agent, scalars);
    const int tm = tile / t.tiles_n, tn = tile % t.tiles_n;
    const int m0 = tm * kSM, n0 = tn * kSN;
    float(*As)[kSM + 4] = reinterpret_cast<float(*)[kSM + 4]>(smem);
    float(*Bs)[kSN + 4] = reinterpret_cast<float(*)[kSN + 4]>(smem + kSK * (kSM + 4));
    const int tid = threadIdx.x, ty = (tid >> 4) & 15, tx = tid & 15;
    const bool worker = tid < 256;       // 16 x 16 threads x (4 x 4) outputs; the other warps only help with the loads
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < t.K; k0 += kSK) {
#pragma unroll
        for (int e = 0; e < kSM * kSK / kThreads; e++) {
            const int idx = tid + e * kThreads;
            int r, k;
            if (!a_mn) { r = idx >> 4; k = idx & 15; } else { k = idx >> 6; r = idx & 63; }
            As[k][r] = (m0 + r < t.M && k0 + k < t.K) ? operand_at(A, a_mn, t.A.r0 + m0 + r, k0 + k) : 0.f;
            if (!b_mn) { r = idx >> 4; k = idx & 15; } else { k = idx >> 6; r = idx & 63; }
            Bs[k][r] = (n0 + r < t.N && k0 + k < t.K) ? operand_at(B, b_mn, t.B.r0 + n0 + r, k0 + k) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kSK && worker; k++) {
            const float4 a = *reinterpret_cast<const float4 *>(&As[k][ty * 4]);
            const float4 b = *reinterpret_cast<const float4 *>(&Bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
    if (worker) {
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) epilogue_element(epi, m0 + ty * 4 + i, n0 + tx * 4 + j, acc[i][j]);
    }
}

// ============================================================================================================
// tcgen05 tile
// ============================================================================================================
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy writes (st.global / st.shared) -> visible to the async proxy (TMA, tensor core)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
// same, shared memory only (does not wait for outstanding global stores)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// bounded wait: try_wait suspends the thread in hardware (no issue-slot burning spin next to the TMA / MMA warps) and
// returns after a system-defined time limit; a lost arrival surfaces as an error after ~1 s, never as a hung GPU box
__device__ __forceinline__ bool mbar_wait(uint64_t *bar, uint32_t parity, int *error_flag) {
    const uint32_t addr = smem_u32(bar);
    long long t0 = 0;
#pragma unroll 1
    for (uint32_t it = 0;; ++it) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) return true;
        if (it == 0) t0 = clock64();
        else if (clock64() - t0 > 2000000000ll) break;
    }
    if (error_flag) atomicExch(error_flag, 1);
    return false;
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA: one box of a 4-D tensor {cols, rows, plane, agent} -> shared memory, completion counted on `bar`
__device__ __forceinline__ void tma_load_4d(const CUtensorMap *tm, uint64_t *bar, uint32_t smem_dst, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

__device__ __forceinline__ bool elect_one() {      // one lane of a converged warp
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}

// UMMA shared-memory descriptor (cute/arch/mma_sm100_desc.hpp::SmemDescriptor), SWIZZLE_128B, version 1:
// start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | layout_type=2 [61,64)
//   K-major : rows of 128 B (64 bf16 of K); SBO = 1024 B between 8-row groups; LBO unused (1)
//   MN-major: rows of 128 B (64 bf16 of M/N) indexed by k; SBO = 1024 B between 8-k groups; LBO = bytes between
//             64-wide M/N groups
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor (UMMA::InstrDescriptor): c_format F32=1 [4,6) | a_format BF16=1 [7,10) | b_format BF16=1 [10,13)
// | a_major [15] | b_major [16] (0 = K, 1 = MN) | N>>3 [17,23) | M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

// per-CTA state that survives across tiles (persistent kernel): pipeline position and TMEM base
struct TcState {
    uint32_t tmem_base;
    uint32_t g;            // k-blocks issued so far (stage = g % kTStages, phase = (g / kTStages) & 1)
    uint32_t accum_uses;   // completed tiles (parity of the accumulator barrier)
    uint8_t *tiles;        // 1024-aligned operand ring: kTStages x (A: hi 16 KB | lo 16 KB ; B: hi 8 KB | lo 8 KB)
    uint64_t *full_bar;    // [kTStages]  TMA -> MMA warp: the k-block landed in shared memory
    uint64_t *empty_bar;   // [kTStages]  tcgen05.commit -> TMA warp: the MMAs that read the slot are done
    uint64_t *accum_bar;   //             tcgen05.commit -> everyone: the accumulator tile is complete
    unsigned long long *trace;   // optional per-CTA timestamps (profiling aid)
    const CUtensorMap *tmA, *tmB; // descriptors of the current task in GLOBAL memory (the task's other fields are read from a smem copy)
    // K blocks of the next tile whose B operand was requested ahead of its A operand (tc_prefetch_b): their `full` barriers are
    // armed with the whole K block's bytes already
    uint32_t b_pre;
};

__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_nctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }

// ---- main loop of one output tile: warp 0 = TMA producer, warp 1 = MMA issuer ----------------------------------
// smem stage: A region 32 KB then B region 16 KB (a 64-row / 32-column task fills only the front of its region).
//   K-major  A: one box {64 k, bm rows, 2 planes}             -> [hi bm*128 B][lo bm*128 B]
//   MN-major A: bm/64 boxes {64 m, 64 k, 2 planes} (m groups) -> [hi g0 8K][lo g0 8K]([hi g1 8K][lo g1 8K])
//   K-major  B: one box {64 k, bn rows, 2 planes}             -> [hi bn*128 B][lo bn*128 B]
//   MN-major B: one box {64 n, 64 k, 2 planes} (bn = 64 only) -> [hi 8 KB][lo 8 KB]
// TMEM accumulator: bm = 128 -> tile row r in lane r; bm = 64 -> tile row r in lane (r % 16) + 32 * (r / 16)
// (cute::UMMA::tmem_frg_1sm, M_MMA == 64: the upper half of every 32-lane subpartition stays unused).
__device__ __forceinline__ void trace_stamp(unsigned long long *trace, int slot) {
    unsigned long long ts;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts));
    trace[(size_t)blockIdx.x * kTraceSlots + slot] = ts;
}

// The B operand of a forward / dX GEMM is a weight shadow that nothing the tile waits for writes, while its A operand (activations,
// gradients) is what the tile waits for: the first K blocks of B are requested here, from the current ring position, so that after
// the wait only the A halves still have to cross the SM's L2 port -- the tile is bound by exactly that ingest.  Caller: a chained
// launch, before the cluster barrier that ends the previous layer (the previous tile's epilogue is done with the ring by then).
__device__ __forceinline__ void tc_prefetch_b(const Task &t, const Task *tg, int tile, int agent, TcState &st, int *error_flag) {
    st.b_pre = 0;
    if ((threadIdx.x >> 5) != 0) return;
    const int nkb = cdiv(t.K, kTK), n_pre = min(nkb, kTStages);
    if (elect_one()) {
        const int n0 = (tile % t.tiles_n) * t.bn, nb = t.B.r0 + n0;
        const uint32_t tiles = smem_u32(st.tiles);
        for (int kb = 0; kb < n_pre; kb++) {
            const uint32_t g = st.g + kb, s = g % kTStages;
            mbar_wait(&st.empty_bar[s], ((g / kTStages) & 1) ^ 1, error_flag);
            mbar_arrive_expect_tx(&st.full_bar[s], (uint32_t)(t.bm + t.bn) * (kTK * 2 * 2));      // A + B bytes: the A loads follow in tc_mainloop
            const uint32_t sb = tiles + s * kTcStageBytes + kTcABytes;
            if (!t.B.mn_major) tma_load_4d(&tg->tmB, &st.full_bar[s], sb, kb * kTK, nb, 0, agent);
            else tma_load_4d(&tg->tmB, &st.full_bar[s], sb, nb, kb * kTK, 0, agent);
        }
    }
    __syncwarp();
    st.b_pre = (uint32_t)n_pre;      // uniform over warp 0 (the only warp that reads it)
}

// returns the number of K-blocks accumulated (0: the tile is zero)
__device__ __forceinline__ int tc_mainloop(const Task &t, int m0, int n0, int agent, TcState &st, int *error_flag, bool traced) {
    const int warp = threadIdx.x >> 5;
    if (traced && threadIdx.x == 0) trace_stamp(st.trace, 12);
    const int nkb = cdiv(t.K, kTK);
    const uint32_t tiles = smem_u32(st.tiles);
    const int a_mn = t.A.mn_major, b_mn = t.B.mn_major;
    const uint32_t g0 = st.g, nst = (uint32_t)kTStages;
    if (warp == 0) {
        if (elect_one()) {
            for (int kb = 0; kb < nkb; kb++) {
                const uint32_t g = g0 + kb, s = g % nst;
                const bool pre = (uint32_t)kb < st.b_pre;      // B requested and the barrier armed ahead (tc_prefetch_b)
                if (!pre) mbar_wait(&st.empty_bar[s], ((g / nst) & 1) ^ 1, error_flag);
                if (traced && kb < 16) trace_stamp(st.trace, 16 + kb);
                if (!pre) mbar_arrive_expect_tx(&st.full_bar[s], (uint32_t)(t.bm + t.bn) * (kTK * 2 * 2));      // both planes of both operand tiles
                const uint32_t sa = tiles + s * kTcStageBytes, sb = sa + kTcABytes;
                const int k0 = kb * kTK, ma = t.A.r0 + m0, nb = t.B.r0 + n0;
                if (!a_mn) {
                    tma_load_4d(st.tmA, &st.full_bar[s], sa, k0, ma, 0, agent);        // box rows = bm (descriptor)
                } else {
                    tma_load_4d(st.tmA, &st.full_bar[s], sa, ma, k0, 0, agent);
                    if (t.bm > 64) tma_load_4d(st.tmA, &st.full_bar[s], sa + kTcABytes / 2, ma + 64, k0, 0, agent);
                }
                if (pre) continue;
                if (!b_mn) tma_load_4d(st.tmB, &st.full_bar[s], sb, k0, nb, 0, agent);
                else tma_load_4d(st.tmB, &st.full_bar[s], sb, nb, k0, 0, agent);
            }
        }
        __syncwarp();
        st.b_pre = 0;
    } else if (warp == 1) {
        const uint32_t idesc = make_idesc(t.bm, t.bn, a_mn, b_mn);
        // byte offsets inside a stage: lo plane of each operand (K-major: after the `rows` 128 B rows of the hi plane; MN-major:
        // after the 64 k-rows of a 64-wide group), and the step of one UMMA_K (16 bf16)
        const uint32_t a_lo = a_mn ? kTcABytes / 4 : (uint32_t)t.bm * 128u, b_lo = b_mn ? kTcBBytes / 2 : (uint32_t)t.bn * 128u;
        const uint32_t a_lbo = a_mn ? kTcABytes / 2 : 16, b_lbo = 16;
        const uint32_t a_kstep = a_mn ? 2048 : 32, b_kstep = b_mn ? 2048 : 32;
        for (int kb = 0; kb < nkb; kb++) {
            const uint32_t g = g0 + kb, s = g % nst;
            mbar_wait(&st.full_bar[s], (g / nst) & 1, error_flag);
            tc_fence_after();
            if (traced && kb < 16 && (threadIdx.x & 31) == 0) trace_stamp(st.trace, 32 + kb);
            if (elect_one()) {
                const uint32_t sa = tiles + s * kTcStageBytes, sb = sa + kTcABytes;
#pragma unroll
                for (int kk = 0; kk < kTK / 16; kk++) {
                    const uint64_t da_hi = make_desc(sa + kk * a_kstep, a_lbo), da_lo = make_desc(sa + a_lo + kk * a_kstep, a_lbo);
                    const uint64_t db_hi = make_desc(sb + kk * b_kstep, b_lbo), db_lo = make_desc(sb + b_lo + kk * b_kstep, b_lbo);
                    // small terms first: a_lo*b_hi + a_hi*b_lo, then a_hi*b_hi
                    umma_bf16(st.tmem_base, da_lo, db_hi, idesc, (kb | kk) ? 1u : 0u);
                    umma_bf16(st.tmem_base, da_hi, db_lo, idesc, 1u);
                    umma_bf16(st.tmem_base, da_hi, db_hi, idesc, 1u);
                }
                umma_commit(&st.empty_bar[s]);                 // implies tcgen05.fence::before_thread_sync
                if (kb == nkb - 1) umma_commit(st.accum_bar);
            }
            __syncwarp();
        }
    }
    st.g += nkb;
    return nkb;
}

// ---- epilogue ----------------------------------------------------------------------------------------------------
// Phase 1: every warp copies its TMEM quadrant (32 rows x 16 columns, one row per lane) into a shared-memory staging
// tile (the operand ring is idle by then).  Phase 2: thread t owns 4 consecutive columns of rows t/16 + 32*i, so a warp
// touches 2 x 256 contiguous bytes of every fp32 array (w, m, v, target) and 2 x 128 B of every bf16 plane: fully
// coalesced 128-bit accesses instead of one row per lane.
constexpr int kCsLd = kTN + 4;      // fp32 row stride of the staging tile: 16 B aligned, conflict-free for 128-bit accesses
static_assert(kTM * kCsLd * 4 <= kTcStageBytes, "staging tile must fit into one operand stage");

__device__ __forceinline__ void store_pm4(const Pm &p, int m, int n, int N, const float (&x)[4]) {
    __nv_bfloat16 *q = p.hi + (int64_t)m * p.ld + n;
    if (n + 3 < N) {        // ld % 8 == 0, plane % 8 == 0, n % 4 == 0  ->  8 B aligned
        uint32_t h0, l0, h1, l1;
        split_pack2(x[0], x[1], h0, l0);
        split_pack2(x[2], x[3], h1, l1);
        *reinterpret_cast<uint2 *>(q) = make_uint2(h0, h1);
        *reinterpret_cast<uint2 *>(q + p.plane) = make_uint2(l0, l1);
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (n + j < N) { __nv_bfloat16 h, l; split_bf16(x[j], h, l); q[j] = h; q[j + p.plane] = l; }
    }
}

constexpr int kAdamRowGroups = 2;      // pass A of the Adam epilogue handles 4 / kAdamRowGroups of a thread's rows at a time
// Adam (+ Polyak, + shadow refresh) on one weight element; g = gradient
struct AdamOut { float m, v, w, t; };
__device__ __forceinline__ AdamOut adam_math(const EpiR &e, float g, float w, float m, float v, float wt) {
    AdamOut o;
    o.m = m + (1.0f - kBeta1) * (g - m);                                  // exp_avg.lerp_(grad, 1 - beta1)
    o.v = v * kBeta2 + (1.0f - kBeta2) * g * g;                           // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    float sq;      // sqrt.approx (MUFU, <= 1 ulp) instead of the IEEE subroutine call: 7 % of an Adam stage's issue slots went into its call / return
    asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(o.v));
    o.w = w - e.step_size * __fdividef(o.m, sq * e.inv_bc2_sqrt + kAdamEps);     // <= 3 ulp from the IEEE form
    o.t = wt * (1.0f - e.tau) + o.w * e.tau;                              // target <- target*(1-tau) + param*tau  (sac_imp.py:146-152)
    return o;
}

// EPI_ADAM phase 2.  The weight matrix is contiguous [M, N] fp32 (it is aliased by the torch parameter), so when N % 4 != 0
// a row starts at any 4-byte phase.
//   pass A: per row the 16 threads take 4-column groups that start at the first 16-byte aligned column of THAT row inside
//           the tile (a0 = 0..3): every w / m / v / target access is an aligned 128-bit access, all loads before any store
//   pass B: the columns no aligned group covers (a0 leading ones, <= 3 trailing ones), one element per thread
//   both passes leave the new weights in the staging tile; pass C writes the bf16 pair shadows from there with the
//   tile-aligned mapping (the shadow rows are padded to 16 B)
__device__ __forceinline__ void adam_epilogue_tile(const EpiR &e, float *Cs, int m0, int n0, int bm) {
    const int tid = threadIdx.x;     // rows [bm, 128) of the staging tile belong to no tile of this CTA (64-row tiles)
    const int ncols = min(kTN, e.N - n0);      // valid columns of this tile (> 0)
#pragma unroll 1
    for (int half = 0; half < kAdamRowGroups; half++) {   // ---- pass A, kAdamRows rows of a thread at a time (register budget)
        const int j16 = tid & 15, r0 = tid >> 4;
        constexpr int R = 4 / kAdamRowGroups;
        int mrow[R], c[R];
        bool vec[R];
        float4 w[R], mm[R], vv[R], wt[R];
#pragma unroll
        for (int ii = 0; ii < R; ii++) {
            const int i = half * R + ii;
            mrow[ii] = m0 + 32 * i + r0;
            const int a0 = (4 - (int)(((int64_t)mrow[ii] * e.N + n0) & 3)) & 3;
            c[ii] = a0 + 4 * j16;
            vec[ii] = mrow[ii] < e.M && c[ii] + 3 < ncols && 32 * i + r0 < bm;
            w[ii] = mm[ii] = vv[ii] = wt[ii] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (vec[ii] && e.apply) {
                const int64_t o = (int64_t)mrow[ii] * e.N + n0 + c[ii];
                w[ii] = __ldcg(reinterpret_cast<const float4 *>(e.w + o));
                mm[ii] = __ldcg(reinterpret_cast<const float4 *>(e.m + o));
                vv[ii] = __ldcg(reinterpret_cast<const float4 *>(e.v + o));
                if (e.wt) wt[ii] = __ldcg(reinterpret_cast<const float4 *>(e.wt + o));
            }
        }
#pragma unroll
        for (int ii = 0; ii < R; ii++) {
            const int i = half * R + ii;
            if (!vec[ii]) continue;
            float *cs = Cs + (32 * i + r0) * kCsLd + c[ii];
            const int64_t o = (int64_t)mrow[ii] * e.N + n0 + c[ii];
            const float g[4] = {cs[0], cs[1], cs[2], cs[3]};
            if (e.gexp) *reinterpret_cast<float4 *>(e.gexp + o) = make_float4(g[0], g[1], g[2], g[3]);
            if (!e.apply) continue;
            const AdamOut a = adam_math(e, g[0], w[ii].x, mm[ii].x, vv[ii].x, wt[ii].x), b = adam_math(e, g[1], w[ii].y, mm[ii].y, vv[ii].y, wt[ii].y);
            const AdamOut cc = adam_math(e, g[2], w[ii].z, mm[ii].z, vv[ii].z, wt[ii].z), d = adam_math(e, g[3], w[ii].w, mm[ii].w, vv[ii].w, wt[ii].w);
            *reinterpret_cast<float4 *>(e.m + o) = make_float4(a.m, b.m, cc.m, d.m);
            *reinterpret_cast<float4 *>(e.v + o) = make_float4(a.v, b.v, cc.v, d.v);
            *reinterpret_cast<float4 *>(e.w + o) = make_float4(a.w, b.w, cc.w, d.w);
            if (e.wt) *reinterpret_cast<float4 *>(e.wt + o) = make_float4(a.t, b.t, cc.t, d.t);
            cs[0] = a.w; cs[1] = b.w; cs[2] = cc.w; cs[3] = d.w;
        }
    }
    if (e.N % 4 != 0 || ncols < kTN) {   // ---- pass B (warp-uniform condition): thread (row = tid / 4, q = tid % 4)
        const int row = tid >> 2, q = tid & 3, m = m0 + row;
        if (m < e.M && row < bm) {
            const int a0 = (4 - (int)(((int64_t)m * e.N + n0) & 3)) & 3;
            const int nv = ncols > a0 ? (ncols - a0) >> 2 : 0, tail0 = a0 + 4 * nv;
            int col[2];
            int cnt = 0;
            if (q < min(a0, ncols)) col[cnt++] = q;                 // leading columns [0, a0)
            if (tail0 + q < ncols) col[cnt++] = tail0 + q;         // trailing columns [tail0, ncols)
            float w[2], mm[2], vv[2], wt[2];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                w[u] = mm[u] = vv[u] = wt[u] = 0.f;
                if (u < cnt && e.apply) {
                    const int64_t o = (int64_t)m * e.N + n0 + col[u];
                    w[u] = __ldcg(e.w + o); mm[u] = __ldcg(e.m + o); vv[u] = __ldcg(e.v + o);
                    if (e.wt) wt[u] = __ldcg(e.wt + o);
                }
            }
#pragma unroll
            for (int u = 0; u < 2; u++) {
                if (u >= cnt) continue;
                const int64_t o = (int64_t)m * e.N + n0 + col[u];
                float *cs = Cs + row * kCsLd + col[u];
                const float g = *cs;
                if (e.gexp) e.gexp[o] = g;
                if (!e.apply) continue;
                const AdamOut r = adam_math(e, g, w[u], mm[u], vv[u], wt[u]);
                e.m[o] = r.m; e.v[o] = r.v; e.w[o] = r.w;
                if (e.wt) e.wt[o] = r.t;
                *cs = r.w;
            }
        }
    }
    if (!e.apply || (!e.shadow.hi && !e.shadow2.hi)) return;
    __syncthreads();                     // ---- pass C: the staging tile now holds the new weights
    {
        const int c4 = (tid & 15) * 4, r0 = tid >> 4;
        if (c4 >= ncols) return;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int m = m0 + 32 * i + r0;
            if (m >= e.M || 32 * i + r0 >= bm) continue;
            const float4 v4 = *reinterpret_cast<const float4 *>(Cs + (32 * i + r0) * kCsLd + c4);
            const float w1[4] = {v4.x, v4.y, v4.z, v4.w};
            const int n = n0 + c4;
            if (e.shadow.hi) store_pm4(e.shadow, m, n, e.N, w1);
            if (e.shadow2.hi && n + 3 >= e.shadow2_col0) {
                if (n >= e.shadow2_col0 && ((n - e.shadow2_col0) & 3) == 0) {
                    store_pm4(e.shadow2, m, n - e.shadow2_col0, e.N - e.shadow2_col0, w1);
                } else {
#pragma unroll
                    for (int j = 0; j < 4; j++)
                        if (n + j >= e.shadow2_col0 && n + j < e.N) pm_store(e.shadow2, m, n + j - e.shadow2_col0, w1[j]);
                }
            }
        }
    }
}

// auxiliary operands of R rows (m[i]) x 4 columns starting at n: the bias (column only) or the sign source of the ReLU mask.
// They do not depend on the accumulator, so the tensor-core epilogue fetches them BEFORE it waits for the main loop.
template <int EPI, int R>
__device__ __forceinline__ void epilogue_aux4(const EpiR &e, const int (&m)[R], int n, float (&aux)[R][4]) {
#pragma unroll
    for (int i = 0; i < R; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) aux[i][j] = 0.f;
    if (n >= e.N) return;
    const bool full = n + 3 < e.N;
    if (EPI == EPI_MASK) {
#pragma unroll
        for (int i = 0; i < R; i++) {       // sign of the stored activation (hi plane)
            if (m[i] >= e.M) continue;
            const __nv_bfloat16 *q = e.mask.hi + (int64_t)m[i] * e.mask.ld + n;
            if (full) {
                const uint2 a = __ldcg(reinterpret_cast<const uint2 *>(q));
                aux[i][0] = bf16_bits_to_float(a.x & 0xFFFFu); aux[i][1] = bf16_bits_to_float(a.x >> 16);
                aux[i][2] = bf16_bits_to_float(a.y & 0xFFFFu); aux[i][3] = bf16_bits_to_float(a.y >> 16);
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) aux[i][j] = (n + j < e.N) ? __bfloat162float(q[j]) : 0.f;
            }
        }
    } else if (e.bias) {                    // the bias depends on the column only (arena vectors are 16 B aligned, n % 4 == 0)
        if (full) {
            const float4 b4 = __ldcg(reinterpret_cast<const float4 *>(e.bias + n));
            aux[0][0] = b4.x; aux[0][1] = b4.y; aux[0][2] = b4.z; aux[0][3] = b4.w;
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++) aux[0][j] = (n + j < e.N) ? ldcg(e.bias + n + j) : 0.f;
        }
#pragma unroll
        for (int i = 1; i < R; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) aux[i][j] = aux[0][j];
    }
}

// R rows (m[i]) x 4 columns starting at n; acc[i] = the staged accumulators, aux = epilogue_aux4 of the same rows / columns.
template <int EPI, int R>
__device__ __forceinline__ void epilogue_rows4(const EpiR &e, const int (&m)[R], int n, const float4 (&acc4)[R], const float (&aux)[R][4]) {
    if (n >= e.N) return;
    const bool full = n + 3 < e.N;
    float acc[R][4];
#pragma unroll
    for (int i = 0; i < R; i++) { acc[i][0] = acc4[i].x; acc[i][1] = acc4[i].y; acc[i][2] = acc4[i].z; acc[i][3] = acc4[i].w; }
#pragma unroll
    for (int i = 0; i < R; i++) {
        if (m[i] >= e.M) continue;
        float out[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (EPI == EPI_F32) out[j] = acc[i][j] + aux[i][j];
            else if (EPI == EPI_BIAS_RELU) out[j] = fmaxf(acc[i][j] + aux[i][j], 0.f);
            else out[j] = aux[i][j] > 0.f ? acc[i][j] : 0.f;
        }
        if (EPI == EPI_F32) {
            float *c = e.C + (int64_t)m[i] * e.ldc + n;
            if (full && (e.ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(c) & 15) == 0)) {
                *reinterpret_cast<float4 *>(c) = make_float4(out[0], out[1], out[2], out[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) if (n + j < e.N) c[j] = out[j];
            }
        } else {
            store_pm4(e.Cpm, m[i], n, e.N, out);
        }
    }
}

template <int EPI>
__device__ __forceinline__ void tc_epilogue(const EpiR &epi, int m0, int n0, int bm, int bn, TcState &st, int nkb_mine, int *error_flag, bool traced) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *Cs = reinterpret_cast<float *>(st.tiles);      // staging tile [kTM][kCsLd] over operand stage 0 (all MMAs have retired)
    // phase-2 mapping: bn / 4 threads cover a row (4 columns each); the 512 threads cover 32 (bn = 64) or 64 (bn = 32) rows per
    // pass, four passes.  The rows' auxiliary operands (bias / activation signs) are fetched now, under the main loop.
    const int ct = bn >> 2, rs = kThreads / ct;
    const int c4 = (tid % ct) * 4, r0 = tid / ct;
    int m[4];
    float aux[4][4];
    if (EPI != EPI_ADAM) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int row = rs * i + r0;
            m[i] = row < bm ? m0 + row : 0x7fffffff;      // rows beyond the tile are skipped like rows beyond M
        }
        epilogue_aux4<EPI, 4>(epi, m, n0 + c4, aux);
    }
    {   // phase 1: warp w owns TMEM lanes 32*(w%4).., column group w/4.  A 64-row tile keeps 16 rows in the lower half of each
        // 32-lane subpartition; a 32-column tile has only two column groups.
        const bool half_m = bm == 64;
        const int row = half_m ? (warp & 3) * 16 + lane : (warp & 3) * 32 + lane, colh = (warp >> 2) * 16;
        const bool cols_live = colh < bn;      // warp-uniform
        float v[16];
        if (nkb_mine > 0) {
            mbar_wait(st.accum_bar, st.accum_uses & 1, error_flag);
            st.accum_uses++;
            if (traced && tid == 64) trace_stamp(st.trace, 6);
            tc_fence_after();
            if (cols_live) tmem_ld16(st.tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)colh, v);
        } else {      // K = 0: a zero tile
#pragma unroll
            for (int j = 0; j < 16; j++) v[j] = 0.f;
        }
        if (cols_live && (!half_m || lane < 16)) {
            float4 *dst = reinterpret_cast<float4 *>(Cs + row * kCsLd + colh);
#pragma unroll
            for (int j = 0; j < 4; j++) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
    }
    tc_fence_before();
    __syncthreads();     // staging complete; all TMEM reads retired (the next tile's first MMA may overwrite the accumulator)
    if (traced && tid == 64) trace_stamp(st.trace, 7);
    if (EPI == EPI_ADAM) {
        adam_epilogue_tile(epi, Cs, m0, n0, bm);
    } else {   // phase 2: the staged accumulators of the thread's rows meet the prefetched auxiliary operands
        float4 acc[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int row = rs * i + r0;
            acc[i] = m[i] != 0x7fffffff ? *reinterpret_cast<const float4 *>(Cs + row * kCsLd + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (traced && tid == 64 && acc[0].x != 12345.678f) trace_stamp(st.trace, 13);
        epilogue_rows4<EPI, 4>(epi, m, n0 + c4, acc, aux);
    }
    if (traced && tid == 64) trace_stamp(st.trace, 8);
    fence_proxy_async_smem();   // generic-proxy accesses of the staging tile are ordered before the next TMA write into it
    __syncthreads();
}

}  // namespace tc

// t = shared-memory copy of the task (fields), tg = the task in global memory (TMA descriptors)
template <uint32_t kEpis = kAllEpis>
__device__ __forceinline__ void gemm_tile_tc(const Task &t, const Task *tg, int tile, const AgentBases &bases, int agent,
                                             const float *scalars, tc::TcState &st, int *error_flag, bool first_tile) {
    using namespace tc;
    st.tmA = &tg->tmA; st.tmB = &tg->tmB;
    const int tm = tile / t.tiles_n, tn = tile % t.tiles_n;
    const int m0 = tm * t.bm, n0 = tn * t.bn;
    const bool traced = st.trace && first_tile;      // the CTA's first tile of the stage
    const int nkb_mine = tc_mainloop(t, m0, n0, agent, st, error_flag, traced);
    auto stamp = [&](int slot) { if (traced && threadIdx.x == 0) trace_stamp(st.trace, slot); };
    stamp(2);
    const EpiR epi = resolve_epilogue(t, bases, agent, scalars);
    switch (t.epi) {
        case EPI_F32: if constexpr ((kEpis & tb(EPI_F32)) != 0) tc_epilogue<EPI_F32>(epi, m0, n0, t.bm, t.bn, st, nkb_mine, error_flag, traced); break;
        case EPI_BIAS_RELU: if constexpr ((kEpis & tb(EPI_BIAS_RELU)) != 0) tc_epilogue<EPI_BIAS_RELU>(epi, m0, n0, t.bm, t.bn, st, nkb_mine, error_flag, traced); break;
        case EPI_MASK: if constexpr ((kEpis & tb(EPI_MASK)) != 0) tc_epilogue<EPI_MASK>(epi, m0, n0, t.bm, t.bn, st, nkb_mine, error_flag, traced); break;
        default: if constexpr ((kEpis & tb(EPI_ADAM)) != 0) tc_epilogue<EPI_ADAM>(epi, m0, n0, t.bm, t.bn, st, nkb_mine, error_flag, traced); break;
    }
    stamp(3);
}

}  // namespace sacb
