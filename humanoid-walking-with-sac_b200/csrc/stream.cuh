// Throughput form of a GEMM stage (population of agents, large-batch data parallel): stages whose tiles outnumber the SMs.
//
// One resident CTA per SM walks its share of the stage's output tiles with the three roles decoupled, so that operand ingest,
// tensor-core issue and the epilogue of consecutive tiles overlap (in the latency form -- gemm.cuh, one tile per CTA -- they run
// one after the other, which is right when a stage has at most one tile per SM):
//   warp 0        TMA producer : runs ahead across tile boundaries, bounded only by the 3 x 64 KB operand ring
//   warp 1        MMA issuer   : tcgen05.mma (bf16x3) into one of TWO 128-column TMEM accumulators
//   warp 2        TMEM allocation / release
//   warps 4..11   epilogue     : tcgen05.ld -> staging tile -> coalesced fused epilogue of tile i while tile i+1 is accumulated
// Output tile 128 x 256 / 128 x 128 / 128 x 64 (chosen per stage by the builder): per 64-deep K block a CTA pulls 96 / 64 / 48 KB for
// 4.2 / 2.1 / 1.05 MFLOP of products -- 43.7 / 32.8 / 21.8 FLOP per operand byte against the chip-wide L2 -> SMEM limit (the 128 x 128
// tile already issues its MMAs at the tensor peak, profiles/r02_tcgen05_rate_by_shape.txt; what holds a large-batch stage at 46-52 %
// tensor-pipe activity is operand delivery: 7.6 TB/s of L2 -> SM traffic, profiles/r02_summary.md).  The 192 KB operand ring is cut
// into as many slots as the stage's widest tile allows: 2 x 96 KB, 3 x 64 KB or 4 x 48 KB.
// Tiles are assigned round-robin (tile = blockIdx.x + i * gridDim.x): every role derives the same sequence on its own.
// Same arithmetic per output element as the latency form (same K order, same three products), so results are bit-identical.
#pragma once
#include "gemm.cuh"

#ifndef SACB_STATE_DEPTH
#define SACB_STATE_DEPTH 2
#endif
namespace sacb {
namespace stream {

constexpr int kThreads = 384;                 // 12 warps
constexpr int kEpiWarp0 = 4, kEpiThreads = 256;
constexpr int kBM = 128, kBN = 128, kBNMax = 256, kBK = 64, kMaxStages = 4;
constexpr int kABytes = kBM * kBK * 2 * 2;    // hi + lo planes: 32 KB
constexpr int kGroupBytes = 64 * kBK * 2 * 2; // one 64-wide group of an MN-major operand, hi + lo: 16 KB ([hi 8 KB][lo 8 KB])
constexpr int kRingBytes = 192 * 1024;
constexpr int kStagingBytes = kBM * tc::kCsLd * 4;                // 128 x 68 floats = 34 KB: 64 columns of the tile at a time
constexpr int kMiscBytes = 1024;                                  // barriers, TMEM base, stage table
constexpr int kSmemBytes = kRingBytes + kStagingBytes + kMiscBytes;   // 232448 = the 227 KB a CTA can have: no static shared memory
constexpr int kAccCols = kBNMax, kTmemCols = 2 * kAccCols;      // two accumulators of up to 256 columns: all 512 TMEM columns
// Optimizer-state landing zone of the Adam epilogue (stages that step weights): the last 64 KB of the ring, two buffers of
// [w | m | v | target][2 rows][256 threads] float4 filled with cp.async -- the state of the NEXT two-row group of a thread is in flight
// (no registers held) while the current group is stepped.  Such a stage runs on a 128 KB operand ring.
constexpr int kStateBufBytes = 4 * 2 * kEpiThreads * 16;         // 32 KB
constexpr int kStateDepth = SACB_STATE_DEPTH;                      // two-row groups of a thread in flight
constexpr int kStateBytes = kStateDepth * kStateBufBytes;
constexpr int kRingBytesAdam = kRingBytes - kStateBytes;          // 128 KB

struct Misc {                 // lives behind the staging tile
    uint64_t full[kMaxStages], empty[kMaxStages], acc_full[2], acc_empty[2];
    uint32_t tmem_base;
    int32_t n_tiles, n_tasks, task_begin;
    int32_t slot_bytes, n_slots;      // ring geometry of this stage: slots of (128 + widest bn) x 256 B
    int32_t adam_state;               // the stage steps weights: the tail of the ring is the optimizer-state landing zone
    int32_t tile_begin[kMaxStageTasks];
};
static_assert(sizeof(Misc) <= kMiscBytes, "misc block");

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory"); }

__device__ __forceinline__ void tmem_alloc_cols(uint32_t *dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}

// the tile a work item denotes; every role calls this with the same arguments
struct TileRef { const Task *tg; int agent, m0, n0, bm, bn, kb0, nkb; };
__device__ __forceinline__ TileRef locate(const Program &P, const Misc &mi, int wi) {
    TileRef r;
    r.agent = wi / mi.n_tiles;
    const int tis = wi % mi.n_tiles;
    int k = 0;
    while (k + 1 < mi.n_tasks && tis >= mi.tile_begin[k + 1]) k++;
    r.tg = &P.tasks[mi.task_begin + k];
    int tile = tis - mi.tile_begin[k];
    r.bm = r.tg->bm; r.bn = r.tg->bn;
    const int tn = r.tg->tiles_n, per = r.tg->tiles_m * tn;
    // split K (gradient-export GEMMs of large batches): tile = [chunk][tm][tn], the chunks of an output tile are accumulated into the
    // zeroed gradient slab with atomics by their epilogues
    const int chunk = r.tg->kb_per_chunk, nkb_all = cdiv(r.tg->K, kBK);
    r.kb0 = 0; r.nkb = nkb_all;
    if (chunk > 0) { r.kb0 = (tile / per) * chunk; r.nkb = max(0, min(nkb_all - r.kb0, chunk)); tile %= per; }
    r.m0 = (tile / tn) * r.bm; r.n0 = (tile % tn) * r.bn;
    return r;
}

// ---- Adam (+ Polyak, + shadow refresh) on 64 columns of the tile held in the staging tile, 256 epilogue threads.
// pass A: per row the 16 threads take the 4-column groups that start at the first 16-byte aligned column of THAT row (the fp32
//         matrices are contiguous [M, N]: a row starts at any 4-byte phase when N % 4 != 0), all loads of two rows before any store
// pass B: the columns no aligned group covers, one element per thread
// Shadows (of the stepped weights, of the action block of a critic's fc1, of the Polyak target) are written straight from the
// registers that hold the new values: 8-byte stores per plane where the group is 4-column aligned in the shadow, else per element.
__device__ __forceinline__ void shadow_store4(const Pm &p, int m, int n, int N, const float (&x)[4]) {
    if (!p.hi) return;
    if ((n & 3) == 0) { tc::store_pm4(p, m, n, N, x); return; }
#pragma unroll
    for (int j = 0; j < 4; j++) if (n + j < N) pm_store(p, m, n + j, x[j]);
}
__device__ __forceinline__ void shadow2_store4(const EpiR &e, int m, int n, const float (&x)[4]) {      // columns >= shadow2_col0 only
    if (!e.shadow2.hi || n + 3 < e.shadow2_col0) return;
    if (n >= e.shadow2_col0 && ((n - e.shadow2_col0) & 3) == 0) { tc::store_pm4(e.shadow2, m, n - e.shadow2_col0, e.N - e.shadow2_col0, x); return; }
#pragma unroll
    for (int j = 0; j < 4; j++) if (n + j >= e.shadow2_col0 && n + j < e.N) pm_store(e.shadow2, m, n + j - e.shadow2_col0, x[j]);
}
// one two-row group of a thread: rows r0 + 16 (2 grp + ii), the aligned 4-column group c[ii] of each
struct AdamGroup { int mrow[2], c[2]; bool vec[2]; };
__device__ __forceinline__ AdamGroup adam_group(const EpiR &e, int m0, int n0, int ncols, int et, int grp) {
    AdamGroup g;
    const int j16 = et & 15, r0 = et >> 4;
#pragma unroll
    for (int ii = 0; ii < 2; ii++) {
        g.mrow[ii] = m0 + r0 + 16 * (2 * grp + ii);
        const int a0 = (4 - (int)(((int64_t)g.mrow[ii] * e.N + n0) & 3)) & 3;
        g.c[ii] = a0 + 4 * j16;
        g.vec[ii] = g.mrow[ii] < e.M && g.c[ii] + 3 < ncols;
    }
    return g;
}
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(tc::smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
// request the optimizer state of group `grp` of the pass at columns n0 into landing buffer `buf` (one commit group, always)
__device__ __forceinline__ void adam_issue(const EpiR &e, float4 *state, int m0, int n0, int et, int grp, int buf) {
    const int ncols = min(64, e.N - n0);
    if (e.apply && ncols > 0) {
        const AdamGroup g = adam_group(e, m0, n0, ncols, et, grp);
        float4 *dst = state + (size_t)buf * (kStateBufBytes / 16) + et;
#pragma unroll
        for (int ii = 0; ii < 2; ii++) {
            if (!g.vec[ii]) continue;
            const int64_t o = (int64_t)g.mrow[ii] * e.N + n0 + g.c[ii];
            cp_async16(dst + (0 * 2 + ii) * kEpiThreads, e.w + o);
            cp_async16(dst + (1 * 2 + ii) * kEpiThreads, e.m + o);
            cp_async16(dst + (2 * 2 + ii) * kEpiThreads, e.v + o);
            if (e.wt) cp_async16(dst + (3 * 2 + ii) * kEpiThreads, e.wt + o);
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}
// `state` = the landing zone when the stage has one (then groups 0 and 1 of this pass were requested by the caller), else null:
// plain loads, two rows of a thread at a time
__device__ __forceinline__ void adam_epilogue(const EpiR &e, const float *Cs, float4 *state, int m0, int n0, int et, bool accumulate) {
    const int ncols = min(64, e.N - n0);
    if (ncols <= 0) {      // uniform over the epilogue threads; the caller's two requests still have to retire
        if (state) asm volatile("cp.async.wait_group 0;" ::: "memory");
        return;
    }
#pragma unroll 1
    for (int grp = 0; grp < 4; grp++) {         // pass A, two rows of a thread at a time
        const AdamGroup g = adam_group(e, m0, n0, ncols, et, grp);
        float4 w[2], mm[2], vv[2], wt[2];
        if (state) {      // groups grp and grp + 1 are in flight: wait for the older one, then put group grp + 2 behind them
            // groups grp .. min(grp + kStateDepth - 1, 3) are in flight: wait for the oldest
            const int younger = min(kStateDepth - 1, 3 - grp);
            if (younger >= 2) asm volatile("cp.async.wait_group 2;" ::: "memory");
            else if (younger == 1) asm volatile("cp.async.wait_group 1;" ::: "memory");
            else asm volatile("cp.async.wait_group 0;" ::: "memory");
            const float4 *src = state + (size_t)(grp % kStateDepth) * (kStateBufBytes / 16) + et;
#pragma unroll
            for (int ii = 0; ii < 2; ii++) {
                w[ii] = mm[ii] = vv[ii] = wt[ii] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g.vec[ii] && e.apply) {      // a thread reads back exactly what it requested: no barrier
                    w[ii] = src[(0 * 2 + ii) * kEpiThreads]; mm[ii] = src[(1 * 2 + ii) * kEpiThreads]; vv[ii] = src[(2 * 2 + ii) * kEpiThreads];
                    if (e.wt) wt[ii] = src[(3 * 2 + ii) * kEpiThreads];
                }
            }
            if (grp + kStateDepth < 4) adam_issue(e, state, m0, n0, et, grp + kStateDepth, grp % kStateDepth);      // the buffer just read
        } else {
#pragma unroll
            for (int ii = 0; ii < 2; ii++) {
                w[ii] = mm[ii] = vv[ii] = wt[ii] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g.vec[ii] && e.apply) {
                    const int64_t o = (int64_t)g.mrow[ii] * e.N + n0 + g.c[ii];
                    w[ii] = __ldcg(reinterpret_cast<const float4 *>(e.w + o));
                    mm[ii] = __ldcg(reinterpret_cast<const float4 *>(e.m + o));
                    vv[ii] = __ldcg(reinterpret_cast<const float4 *>(e.v + o));
                    if (e.wt) wt[ii] = __ldcg(reinterpret_cast<const float4 *>(e.wt + o));
                }
            }
        }
#pragma unroll
        for (int ii = 0; ii < 2; ii++) {
            if (!g.vec[ii]) continue;
            const int row = (et >> 4) + 16 * (2 * grp + ii);
            const float *cs = Cs + row * tc::kCsLd + g.c[ii];
            const int64_t o = (int64_t)g.mrow[ii] * e.N + n0 + g.c[ii];
            const float gr[4] = {cs[0], cs[1], cs[2], cs[3]};
            if (e.gexp) {
                if (accumulate) atomicAdd(reinterpret_cast<float4 *>(e.gexp + o), make_float4(gr[0], gr[1], gr[2], gr[3]));      // one 16-byte reduction at L2
                else *reinterpret_cast<float4 *>(e.gexp + o) = make_float4(gr[0], gr[1], gr[2], gr[3]);
            }
            if (!e.apply) continue;
            const tc::AdamOut a = tc::adam_math(e, gr[0], w[ii].x, mm[ii].x, vv[ii].x, wt[ii].x), b = tc::adam_math(e, gr[1], w[ii].y, mm[ii].y, vv[ii].y, wt[ii].y);
            const tc::AdamOut cc = tc::adam_math(e, gr[2], w[ii].z, mm[ii].z, vv[ii].z, wt[ii].z), d = tc::adam_math(e, gr[3], w[ii].w, mm[ii].w, vv[ii].w, wt[ii].w);
            *reinterpret_cast<float4 *>(e.m + o) = make_float4(a.m, b.m, cc.m, d.m);
            *reinterpret_cast<float4 *>(e.v + o) = make_float4(a.v, b.v, cc.v, d.v);
            *reinterpret_cast<float4 *>(e.w + o) = make_float4(a.w, b.w, cc.w, d.w);
            if (e.wt) *reinterpret_cast<float4 *>(e.wt + o) = make_float4(a.t, b.t, cc.t, d.t);
            const float w1[4] = {a.w, b.w, cc.w, d.w};
            const int n = n0 + g.c[ii];
            shadow_store4(e.shadow, g.mrow[ii], n, e.N, w1);
            shadow2_store4(e, g.mrow[ii], n, w1);
            if (e.wt && e.shadow_t.hi) { const float t1[4] = {a.t, b.t, cc.t, d.t}; shadow_store4(e.shadow_t, g.mrow[ii], n, e.N, t1); }
        }
    }
    if (e.N % 4 != 0 || ncols < 64) {           // pass B: the columns no aligned group covers; thread (row = et / 4 (+ 64), q = et % 4)
        // at most two such columns per row half and thread: all (<= 16) scalar loads of the thread are issued before the first step, one
        // exposed round trip instead of four (a critic's fc1 has 365 columns: every row of every pass comes through here)
        int64_t off[4];
        int rowc[4], coln[4];
        float sw[4], sm[4], sv[4], st[4];
        int cnt = 0;
#pragma unroll
        for (int hb = 0; hb < 2; hb++) {
            const int row = (et >> 2) + 64 * hb, q = et & 3, m = m0 + row;
            const bool live = m < e.M;
            const int a0 = (4 - (int)(((int64_t)m * e.N + n0) & 3)) & 3;
            const int nv = ncols > a0 ? (ncols - a0) >> 2 : 0, tail0 = a0 + 4 * nv;
            const int cand[2] = {q, tail0 + q};
            const bool on[2] = {live && q < min(a0, ncols), live && tail0 + q < ncols};
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int k = 2 * hb + u;
                off[k] = -1; rowc[k] = row; coln[k] = cand[u];
                sw[k] = sm[k] = sv[k] = st[k] = 0.f;
                if (on[u]) {
                    off[k] = (int64_t)m * e.N + n0 + cand[u];
                    if (e.apply) { sw[k] = __ldcg(e.w + off[k]); sm[k] = __ldcg(e.m + off[k]); sv[k] = __ldcg(e.v + off[k]); if (e.wt) st[k] = __ldcg(e.wt + off[k]); }
                    cnt++;
                }
            }
        }
        if (cnt) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (off[k] < 0) continue;
                const int64_t o = off[k];
                const float g = Cs[rowc[k] * tc::kCsLd + coln[k]];
                if (e.gexp) { if (accumulate) atomicAdd(e.gexp + o, g); else e.gexp[o] = g; }
                if (!e.apply) continue;
                const tc::AdamOut r = tc::adam_math(e, g, sw[k], sm[k], sv[k], st[k]);
                e.m[o] = r.m; e.v[o] = r.v; e.w[o] = r.w;
                if (e.wt) e.wt[o] = r.t;
                const int m = m0 + rowc[k], n = n0 + coln[k];
                if (e.shadow.hi) pm_store(e.shadow, m, n, r.w);
                if (e.shadow2.hi && n >= e.shadow2_col0) pm_store(e.shadow2, m, n - e.shadow2_col0, r.w);
                if (e.wt && e.shadow_t.hi) pm_store(e.shadow_t, m, n, r.t);
            }
        }
    }
}

// L2 prefetch of the optimizer state one 64-column pass of an Adam tile will stream (w, m, v, target: 4 x 128 x 64 floats), issued
// by the epilogue warps at the start of the tile, so that the load phases of its passes find their operands in L2 instead of paying
// DRAM latency four times per pass.  (Prefetching a whole pass AHEAD was measured slower -- 1.36 -> 1.63 ms on the heaviest Adam
// stage of a 128-agent population: the stage is DRAM-throughput bound, earlier prefetches only get evicted.)
__device__ __forceinline__ void adam_prefetch(const EpiR &e, int m0, int n0c, int et) {
    if (!e.apply || n0c >= e.N) return;
    constexpr int kLines = 3;      // 64 floats = 2 lines, + 1: rows start at any 4-byte phase
    for (int i = et; i < kBM * kLines; i += kEpiThreads) {
        const int row = i / kLines, l = i % kLines, m = m0 + row;
        if (m >= e.M || n0c + l * 32 >= e.N + 32) continue;
        const int64_t o = (int64_t)m * e.N + n0c + l * 32;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(e.w + o));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(e.m + o));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(e.v + o));
        if (e.wt) asm volatile("prefetch.global.L2 [%0];" ::"l"(e.wt + o));
    }
}

template <int EPI>
__device__ __forceinline__ void plain_epilogue(const EpiR &epi, const float *Cs, int m0, int n0c, int et, const float (&aux)[8][4]) {
    const int c4 = (et & 15) * 4, r0 = et >> 4;
#pragma unroll
    for (int half = 0; half < 2; half++) {
        int m[4];
        float4 acc[4];
        float ax[4][4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int row = r0 + 16 * (4 * half + i);
            m[i] = m0 + row;
            acc[i] = *reinterpret_cast<const float4 *>(Cs + row * tc::kCsLd + c4);
#pragma unroll
            for (int j = 0; j < 4; j++) ax[i][j] = aux[4 * half + i][j];
        }
        tc::epilogue_rows4<EPI, 4>(epi, m, n0c + c4, acc, ax);
    }
}

template <int EPI>
__device__ __forceinline__ void plain_aux(const EpiR &epi, int m0, int n0c, int et, float (&aux)[8][4]) {
    const int c4 = (et & 15) * 4, r0 = et >> 4;
#pragma unroll
    for (int half = 0; half < 2; half++) {
        int m[4];
        float ax[4][4];
#pragma unroll
        for (int i = 0; i < 4; i++) m[i] = m0 + r0 + 16 * (4 * half + i);
        tc::epilogue_aux4<EPI, 4>(epi, m, n0c + c4, ax);
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) aux[4 * half + i][j] = ax[i][j];
    }
}

// epilogue of one tile: per 64-column pass TMEM -> staging tile (phase 1), fused epilogue from the staging tile (phase 2).
// The first pass's bias / mask operands and the L2 prefetch of the Adam state are issued BEFORE the wait on the accumulator.
template <int EPI>
__device__ __forceinline__ void epilogue_tile(const EpiR &epi, float *Cs, float4 *state, uint32_t acc_addr, const TileRef &r, int et, uint64_t *acc_full, uint32_t parity,
                                              uint64_t *acc_empty, int *err) {
    const int ew = et >> 5, lane = et & 31, q = ew & 3, hcol = (ew >> 2) * 32;
    const int passes = r.bn >> 6;      // 64 columns of the tile at a time: 1, 2 or 4 passes
    float aux[8][4];
    uint32_t mask_bits[4] = {0u, 0u, 0u, 0u};
    if (EPI == EPI_ADAM) {
        for (int p = state ? 1 : 0; p < passes; p++) adam_prefetch(epi, r.m0, r.n0 + 64 * p, et);
        if (state) for (int g0 = 0; g0 < kStateDepth; g0++) adam_issue(epi, state, r.m0, r.n0, et, g0, g0);      // first pass: under the main loop
    } else if (EPI == EPI_MASK) {
        // the ReLU-mask operand (sign of the stored activation) of ALL passes is fetched now and kept as one bit per element:
        // no global load sits between the accumulator and the stores any more (the mask loads paced the dX stages: an epilogue
        // whose second pass started with an exposed L2 / DRAM round trip)
        // (the 16 loads of two passes are issued back to back from clamped addresses and only then unpacked: written with the
        //  row / column guards around each load the compiler serialised them, eight L2 round trips per pass -- ncu source view;
        //  a 256-column tile fetches its second pair of passes the same way right behind the first)
        const int c4 = (et & 15) * 4, r0 = et >> 4;
        auto fetch2 = [&](int pb, uint32_t &bits_a, uint32_t &bits_b) {
            uint2 raw[2][8];
#pragma unroll
            for (int p = 0; p < 2; p++)
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const int row = min(r.m0 + r0 + 16 * i, epi.M - 1), col = min(r.n0 + 64 * (pb + p) + c4, epi.N - 4);      // EPI_MASK outputs are hidden-width: N % 8 == 0
                    raw[p][i] = (pb + p < passes) ? __ldcg(reinterpret_cast<const uint2 *>(epi.mask.hi + (int64_t)row * epi.mask.ld + col)) : make_uint2(0u, 0u);
                }
#pragma unroll
            for (int p = 0; p < 2; p++) {
                uint32_t bits = 0u;
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const bool ok = pb + p < passes && r.m0 + r0 + 16 * i < epi.M && r.n0 + 64 * (pb + p) + c4 < epi.N;
                    const uint32_t w[2] = {raw[p][i].x, raw[p][i].y};
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const uint32_t h = (w[j >> 1] >> (16 * (j & 1))) & 0xFFFFu;      // bf16 bits of the stored activation: > 0 <=> sign clear, not zero
                        const bool pos = ok && (h & 0x8000u) == 0u && (h & 0x7FFFu) != 0u && (h & 0x7FFFu) <= 0x7F80u;
                        bits |= (pos ? 1u : 0u) << (4 * i + j);
                    }
                }
                if (p == 0) bits_a = bits; else bits_b = bits;
            }
        };
        fetch2(0, mask_bits[0], mask_bits[1]);
        if (passes > 2) fetch2(2, mask_bits[2], mask_bits[3]);      // CTA-uniform
    } else {
        plain_aux<EPI>(epi, r.m0, r.n0, et, aux);
    }
    tc::mbar_wait(acc_full, parity, err);
    tc::tc_fence_after();
    for (int pass = 0; pass < passes; pass++) {
        const bool last = pass == passes - 1;
        const int n0c = r.n0 + 64 * pass;
        if (n0c >= epi.N) {      // ragged N: nothing to store from this pass, but the accumulator still has to be released
            if (last) { tc::tc_fence_before(); if (lane == 0) mbar_arrive(acc_empty); }
            if (EPI == EPI_ADAM && state) {      // keep the request pipeline in step: retire this pass's (empty) groups, request the next pass's
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                if (!last) for (int g0 = 0; g0 < kStateDepth; g0++) adam_issue(epi, state, r.m0, n0c + 64, et, g0, g0);
            }
            continue;
        }
        if (EPI == EPI_MASK) {
            const uint32_t mb = pass == 0 ? mask_bits[0] : (pass == 1 ? mask_bits[1] : (pass == 2 ? mask_bits[2] : mask_bits[3]));
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) aux[i][j] = ((mb >> (4 * i + j)) & 1u) ? 1.f : 0.f;
        } else if (EPI != EPI_ADAM && pass > 0) {
            plain_aux<EPI>(epi, r.m0, n0c, et, aux);
        }
        {
            float v[16];
            float4 *dst = reinterpret_cast<float4 *>(Cs + (q * 32 + lane) * tc::kCsLd + hcol);
            const uint32_t taddr = acc_addr + ((uint32_t)(q * 32) << 16) + (uint32_t)(64 * pass + hcol);
            tc::tmem_ld16(taddr, v);
#pragma unroll
            for (int j = 0; j < 4; j++) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            tc::tmem_ld16(taddr + 16, v);
#pragma unroll
            for (int j = 0; j < 4; j++) dst[4 + j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
        if (last) {      // every TMEM read of this warp has retired (tcgen05.wait::ld inside tmem_ld16): the accumulator may be reused
            tc::tc_fence_before();
            if (lane == 0) mbar_arrive(acc_empty);
        }
        epi_bar();
        if (EPI == EPI_ADAM) {
            adam_epilogue(epi, Cs, state, r.m0, n0c, et, r.tg->kb_per_chunk > 0);
            // the next pass's first two groups: in flight across the barrier and the next TMEM -> staging copy
            if (state && !last) for (int g0 = 0; g0 < kStateDepth; g0++) adam_issue(epi, state, r.m0, n0c + 64, et, g0, g0);
        } else plain_epilogue<EPI>(epi, Cs, r.m0, n0c, et, aux);
        epi_bar();        // the staging tile is free for the next pass / tile
    }
}

// the kernel body; P.tasks of the stage are all T_GEMM with bm = 128 and bn in {64, 128, 256}
__device__ __forceinline__ void gemm_stage(const Program &P, const Stage &stage, uint8_t *smem) {
    uint8_t *ring = smem;                                              // 1024-aligned (checked by the caller)
    float *Cs = reinterpret_cast<float *>(smem + kRingBytes);
    Misc &mi = *reinterpret_cast<Misc *>(smem + kRingBytes + kStagingBytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 32) {
        for (int i = 0; i < kMaxStages; i++) { tc::mbar_init(&mi.full[i], 1); tc::mbar_init(&mi.empty[i], 1); }
        for (int i = 0; i < 2; i++) { tc::mbar_init(&mi.acc_full[i], 1); tc::mbar_init(&mi.acc_empty[i], kEpiThreads / 32); }
        tc::fence_barrier_init();
    }
    if (warp == 2) tmem_alloc_cols(&mi.tmem_base, kTmemCols);
    if (threadIdx.x >= 64 && threadIdx.x < 64 + kMaxStageTasks) mi.tile_begin[threadIdx.x - 64] = stage.tile_begin[threadIdx.x - 64];
    if (threadIdx.x == 96) {
        mi.n_tiles = stage.n_tiles; mi.n_tasks = stage.task_end - stage.task_begin; mi.task_begin = stage.task_begin;
        int bn_max = 64, steps = 0;      // the producer runs ahead across tile boundaries: one slot size per stage, that of its widest tile
        for (int k = stage.task_begin; k < stage.task_end; k++) {
            bn_max = max(bn_max, __ldg(&P.tasks[k].bn));
            // a short K loop (K = batch of a population's agents): the tile is bound by its Adam epilogue; a long one (large batch) by its
            // main loop, which keeps the whole ring
            if (__ldg(&P.tasks[k].epi) == EPI_ADAM && __ldg(&P.tasks[k].adam.apply)) steps |= __ldg(&P.tasks[k].K) <= 16 * kBK ? 1 : 2;
        }
        mi.slot_bytes = kABytes + bn_max * (kBK * 2 * 2);
        mi.adam_state = (steps == 1 && mi.slot_bytes <= kRingBytesAdam) ? 1 : 0;      // (the builder keeps weight-stepping tiles at 128 columns)
        mi.n_slots = min(kMaxStages, (mi.adam_state ? kRingBytesAdam : kRingBytes) / mi.slot_bytes);
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const uint32_t tmem = mi.tmem_base, n_slots = (uint32_t)mi.n_slots, slot_bytes = (uint32_t)mi.slot_bytes;
    const int total = mi.n_tiles * P.n_agents;
    int *err = P.error_flag;

    if (warp == 0) {                       // ---------------------------------------------------------------- TMA producer
        if (tc::elect_one()) {
            uint32_t g = 0;
            for (int wi = blockIdx.x; wi < total; wi += gridDim.x) {
                const TileRef r = locate(P, mi, wi);
                const Task &t = *r.tg;
                const int a_mn = t.A.mn_major, b_mn = t.B.mn_major, nkb = r.nkb;
                const int ma = t.A.r0 + r.m0, nb = t.B.r0 + r.n0;
                const uint32_t bytes = (uint32_t)(r.bm + r.bn) * (kBK * 2 * 2);
                for (int kb = 0; kb < nkb; kb++, g++) {
                    const uint32_t s = g % n_slots;
                    tc::mbar_wait(&mi.empty[s], ((g / n_slots) & 1) ^ 1, err);
                    tc::mbar_arrive_expect_tx(&mi.full[s], bytes);
                    const uint32_t sa = tc::smem_u32(ring) + s * slot_bytes, sb = sa + kABytes;
                    const int k0 = (r.kb0 + kb) * kBK;
                    if (!a_mn) {
                        tc::tma_load_4d(&t.tmA, &mi.full[s], sa, k0, ma, 0, r.agent);
                    } else {
                        tc::tma_load_4d(&t.tmA, &mi.full[s], sa, ma, k0, 0, r.agent);
                        tc::tma_load_4d(&t.tmA, &mi.full[s], sa + kABytes / 2, ma + 64, k0, 0, r.agent);
                    }
                    if (!b_mn) {
                        tc::tma_load_4d(&t.tmB, &mi.full[s], sb, k0, nb, 0, r.agent);
                    } else {      // one box per 64-wide group of columns
                        for (int j = 0; j < r.bn; j += 64) tc::tma_load_4d(&t.tmB, &mi.full[s], sb + (j >> 6) * kGroupBytes, nb + j, k0, 0, r.agent);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {                // ---------------------------------------------------------------- MMA issuer
        uint32_t g = 0, it = 0;
        for (int wi = blockIdx.x; wi < total; wi += gridDim.x, it++) {
            const TileRef r = locate(P, mi, wi);
            const Task &t = *r.tg;
            const int a_mn = t.A.mn_major, b_mn = t.B.mn_major, nkb = r.nkb;
            const uint32_t buf = it & 1, use = it >> 1;
            tc::mbar_wait(&mi.acc_empty[buf], (use & 1) ^ 1, err);      // the epilogue has drained this accumulator
            tc::tc_fence_after();
            const uint32_t idesc = tc::make_idesc(r.bm, r.bn, a_mn, b_mn), d = tmem + buf * kAccCols;
            const uint32_t a_lo = a_mn ? kGroupBytes / 2 : (uint32_t)r.bm * 128u, b_lo = b_mn ? kGroupBytes / 2 : (uint32_t)r.bn * 128u;
            const uint32_t a_lbo = a_mn ? kGroupBytes : 16, b_lbo = b_mn ? kGroupBytes : 16;
            const uint32_t a_kstep = a_mn ? 2048 : 32, b_kstep = b_mn ? 2048 : 32;
            for (int kb = 0; kb < nkb; kb++, g++) {
                const uint32_t s = g % n_slots;
                tc::mbar_wait(&mi.full[s], (g / n_slots) & 1, err);
                tc::tc_fence_after();
                if (tc::elect_one()) {
                    const uint32_t sa = tc::smem_u32(ring) + s * slot_bytes, sb = sa + kABytes;
#pragma unroll
                    for (int kk = 0; kk < kBK / 16; kk++) {
                        const uint64_t da_hi = tc::make_desc(sa + kk * a_kstep, a_lbo), da_lo = tc::make_desc(sa + a_lo + kk * a_kstep, a_lbo);
                        const uint64_t db_hi = tc::make_desc(sb + kk * b_kstep, b_lbo), db_lo = tc::make_desc(sb + b_lo + kk * b_kstep, b_lbo);
                        tc::umma_bf16(d, da_lo, db_hi, idesc, (kb | kk) ? 1u : 0u);      // same order of the three products as the latency tile
                        tc::umma_bf16(d, da_hi, db_lo, idesc, 1u);
                        tc::umma_bf16(d, da_hi, db_hi, idesc, 1u);
                    }
                    tc::umma_commit(&mi.empty[s]);
                    if (kb == nkb - 1) tc::umma_commit(&mi.acc_full[buf]);
                }
                __syncwarp();
            }
        }
    } else if (warp >= kEpiWarp0) {        // ---------------------------------------------------------------- epilogue
        const int et = threadIdx.x - kEpiWarp0 * 32;
        float4 *state = mi.adam_state ? reinterpret_cast<float4 *>(ring + kRingBytesAdam) : nullptr;
        uint32_t it = 0;
        for (int wi = blockIdx.x; wi < total; wi += gridDim.x, it++) {
            const TileRef r = locate(P, mi, wi);
            const Task &t = *r.tg;
            const float *scalars = resolve(P.scalars, P.bases, r.agent);
            const EpiR epi = resolve_epilogue(t, P.bases, r.agent, scalars);
            const uint32_t buf = it & 1, use = it >> 1;
            const uint32_t acc = tmem + buf * kAccCols;
            if (wi + (int)gridDim.x < total) {      // the NEXT tile's ReLU-mask rows -> L2 while this tile is finished (one line per thread)
                const TileRef nr = locate(P, mi, wi + gridDim.x);
                if (nr.tg->epi == EPI_MASK) {
                    const Pm mk = resolve_pm(nr.tg->mask, P.bases, nr.agent);
                    const int lines = (nr.bn * 2 + 127) / 128;
                    for (int i = et; i < kBM * lines; i += kEpiThreads) {
                        const int row = nr.m0 + i / lines, col = nr.n0 + (i % lines) * 64;
                        if (row < nr.tg->M && col < nr.tg->N) asm volatile("prefetch.global.L2 [%0];" ::"l"(mk.hi + (int64_t)row * mk.ld + col));
                    }
                }
            }
            switch (epi.epi) {
                case EPI_F32: epilogue_tile<EPI_F32>(epi, Cs, nullptr, acc, r, et, &mi.acc_full[buf], use & 1, &mi.acc_empty[buf], err); break;
                case EPI_BIAS_RELU: epilogue_tile<EPI_BIAS_RELU>(epi, Cs, nullptr, acc, r, et, &mi.acc_full[buf], use & 1, &mi.acc_empty[buf], err); break;
                case EPI_MASK: epilogue_tile<EPI_MASK>(epi, Cs, nullptr, acc, r, et, &mi.acc_full[buf], use & 1, &mi.acc_empty[buf], err); break;
                default: epilogue_tile<EPI_ADAM>(epi, Cs, (state && epi.apply) ? state : nullptr, acc, r, et, &mi.acc_full[buf], use & 1, &mi.acc_empty[buf], err); break;
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 2) tc::tmem_dealloc(tmem, kTmemCols);
}

}  // namespace stream
}  // namespace sacb
