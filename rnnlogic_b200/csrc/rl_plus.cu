// rnnlogic_b200 -- PredictorPlus kernels: candidate compaction, rule-embedding aggregation
// (sum / PNA statistics), scatter of candidate scores into the logit matrix, and the backward into
// the rule embeddings.  Reference: src/predictors.py:210-271, src/layers.py:63-77 / 89-126.
//
// A candidate is a (query, entity) cell with a non-zero total path count (predictors.py:239).
// Candidates are numbered slot-major, entity-major, lane-minor; the order is internal (every
// per-candidate op of the reference is row-wise or an order-free reduction).
#include "rl_device.cuh"

#define HC 16   // hidden-dim chunk kept in registers per pass

// ------------------------------------------------------------------------------------------
// pass 1: nzmask[S][N] (bit b <=> sum_rule count != 0) and cand_cnt[S*N] = popcount
// ------------------------------------------------------------------------------------------
template <typename CT>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_plus_mask(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, uint32_t *__restrict__ nzmask,
            int32_t *__restrict__ cand_cnt)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.y;
    const int ew = blockIdx.x * WARPS_PER_BLOCK + warp;
    const int N = g.num_entities, W = g.rank_words;
    if (ew >= W) return;
    const int q = s.slot_head[slot];
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    const int h = s.lane_h[slot * RL_LANES + lane];
    const bool has_zr = r.zr_ptr[q + 1] > r.zr_ptr[q];
    WordItems wi = load_word_items(fr, s, W, slot, ew);
    uint32_t todo = wi.present;
    if (has_zr) todo |= __reduce_or_sync(FULL, (h >= 0 && (h >> 5) == ew) ? (1u << (h & 31)) : 0u);
    uint32_t my_bits = 0;                                   // lane i keeps the word of entity ew*32+i
    while (todo) {
        const int i = __ffs(todo) - 1;
        todo &= todo - 1;
        bool any = false;
        if ((wi.present >> i) & 1u) for_entity_items<CT>(wi, r, arena, i, [&](CT c, int) { any |= (c != 0); });
        if (has_zr && h == ew * 32 + i) any = true;
        const uint32_t bits = __ballot_sync(FULL, any);
        if (lane == i) my_bits = bits;
    }
    const int e1 = min(32, N - ew * 32);
    if (lane < e1) {
        nzmask[(size_t)slot * N + ew * 32 + lane] = my_bits;
        cand_cnt[(size_t)slot * N + ew * 32 + lane] = __popc(my_bits);
    }
}

// ------------------------------------------------------------------------------------------
// pass 2: per-candidate aggregates.  out[C][H] = sum_rule fp32(count) * emb[rule]  (layers.py:68-72);
// PNA additionally sum of count*emb^2, min / max of emb over rules with count != 0 and their
// arg-rules (layers.py:94-99), and degree = sum count + 1 (layers.py:92).
// ------------------------------------------------------------------------------------------
template <typename CT, bool PNA>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_plus_features(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, const uint32_t *__restrict__ nzmask,
                const int64_t *__restrict__ cand_off, const int32_t *__restrict__ q_off,
                const int32_t *__restrict__ rule_local, const float *__restrict__ emb, int H,
                float *__restrict__ out_sum, float *__restrict__ out_sq, float *__restrict__ out_min,
                float *__restrict__ out_max, int32_t *__restrict__ arg_min, int32_t *__restrict__ arg_max,
                float *__restrict__ degree, int64_t *__restrict__ cand_query)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.y;
    const int ew = blockIdx.x * WARPS_PER_BLOCK + warp;           // entity word: 32 entities, one coalesced mask read
    const int N = g.num_entities;
    if (ew >= g.rank_words) return;
    const int e_lane = ew * 32 + lane;
    const uint32_t my_bits = e_lane < N ? nzmask[(size_t)slot * N + e_lane] : 0u;
    uint32_t cand_ents = __ballot_sync(FULL, my_bits != 0u);
    if (cand_ents == 0u) return;
    const int q = s.slot_head[slot];
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    const int h = s.lane_h[slot * RL_LANES + lane];
    WordItems wi = load_word_items(fr, s, g.rank_words, slot, ew);
  while (cand_ents) {
    const int ei = __ffs(cand_ents) - 1;
    cand_ents &= cand_ents - 1;
    const int e = ew * 32 + ei;
    const uint32_t bits = __shfl_sync(FULL, my_bits, ei);
    const bool mine = (bits >> lane) & 1u;
    const long long idx = cand_off[(size_t)slot * N + e] + __popc(bits & ((1u << lane) - 1u));
    for (int h0 = 0; h0 < H; h0 += HC) {
        double a1[HC], a2[PNA ? HC : 1];
        float mn[PNA ? HC : 1], mx[PNA ? HC : 1];
        int amn[PNA ? HC : 1], amx[PNA ? HC : 1];
        double deg = 1.0;
#pragma unroll
        for (int k = 0; k < HC; ++k) {
            a1[k] = 0.0;
            if (PNA) { a2[k] = 0.0; mn[k] = INFINITY; mx[k] = -INFINITY; amn[k] = -1; amx[k] = -1; }
        }
        auto add = [&](float cf, int rule) {
            const int lr = rule_local[rule];
            const float *er = emb + (size_t)lr * H + h0;
            deg += (double)cf;
#pragma unroll
            for (int k = 0; k < HC; ++k) {
                if (h0 + k < H) {
                    const float ev = __ldg(er + k);
                    a1[k] += (double)cf * (double)ev;
                    if (PNA) {
                        a2[k] += (double)cf * (double)(ev * ev);
                        if (cf != 0.f) {
                            if (ev < mn[k]) { mn[k] = ev; amn[k] = lr; }
                            if (ev > mx[k]) { mx[k] = ev; amx[k] = lr; }
                        }
                    }
                }
            }
        };
        if ((wi.present >> ei) & 1u)
            for_entity_items<CT>(wi, r, arena, ei, [&](CT c, int t) { add((float)c, r.node_term_rule[t]); });
        if (h == e)                                            // empty-body rules: count = one_hot(h)
            for (int t = r.zr_ptr[q]; t < r.zr_ptr[q + 1]; ++t) add(1.f, r.zr_rule[t]);
        if (mine) {
#pragma unroll
            for (int k = 0; k < HC; ++k) {
                if (h0 + k < H) {
                    out_sum[idx * H + h0 + k] = (float)a1[k];
                    if (PNA) {
                        out_sq[idx * H + h0 + k] = (float)a2[k];
                        out_min[idx * H + h0 + k] = mn[k];
                        out_max[idx * H + h0 + k] = mx[k];
                        arg_min[idx * H + h0 + k] = amn[k];
                        arg_max[idx * H + h0 + k] = amx[k];
                    }
                }
            }
            if (h0 == 0) {
                if (degree) degree[idx] = (float)deg;
                cand_query[idx] = (int64_t)q_off[slot] + lane;
            }
        }
    }
  }
}

// ------------------------------------------------------------------------------------------
// candidate scores -> logits (predictors.py:257-269), and the reverse gather for the backward
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_plus_scatter(int N, const uint32_t *__restrict__ nzmask, const int64_t *__restrict__ cand_off,
               const float *__restrict__ zc, const float *__restrict__ bias, const float *__restrict__ extra,
               int fill_neg_inf, float *__restrict__ Z)
{
    const int slot = blockIdx.y;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * RL_LANES) return;
    const int e = (int)(i >> 5), lane = (int)(i & 31);
    const uint32_t bits = nzmask[(size_t)slot * N + e];
    float z = 0.f;
    if ((bits >> lane) & 1u) z = zc[cand_off[(size_t)slot * N + e] + __popc(bits & ((1u << lane) - 1u))];
    else if (fill_neg_inf) z = -INFINITY;
    if (bias) z += bias[e];
    if (extra) z += extra[(size_t)slot * N * RL_LANES + i];
    Z[(size_t)slot * N * RL_LANES + i] = z;
}

__global__ void __launch_bounds__(256)
k_plus_gather(int N, const uint32_t *__restrict__ nzmask, const int64_t *__restrict__ cand_off,
              const float *__restrict__ G, float *__restrict__ dz)
{
    const int slot = blockIdx.y;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * RL_LANES) return;
    const int e = (int)(i >> 5), lane = (int)(i & 31);
    const uint32_t bits = nzmask[(size_t)slot * N + e];
    if ((bits >> lane) & 1u)
        dz[cand_off[(size_t)slot * N + e] + __popc(bits & ((1u << lane) - 1u))] = G[(size_t)slot * N * RL_LANES + i];
}

// ------------------------------------------------------------------------------------------
// backward into the rule embeddings: gA[rule][h] += sum_cells fp32(count) * dA[cell][h]
// (and gB from dB for the PNA squared-sum branch).  Block per (slot, rule end).
// ------------------------------------------------------------------------------------------
// One warp per item (non-zero row of a rule-end node): for every query lane with a non-zero count,
// lanes 0..H-1 add count * dA[cell][h] into gA[rule][h] of every rule ending at the item's node.
#define PLUS_ITEM_BLOCKS 96
template <typename CT>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_plus_backward(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, const uint32_t *__restrict__ nzmask,
                const int64_t *__restrict__ cand_off, const int32_t *__restrict__ rule_local, int H,
                const float *__restrict__ dA, const float *__restrict__ dB, float *__restrict__ gA,
                float *__restrict__ gB)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.y;
    const int N = g.num_entities;
    const int q = s.slot_head[slot];
    const uint32_t *ms = nzmask + (size_t)slot * N;
    const int64_t *co = cand_off + (size_t)slot * N;
    auto contribute = [&](float cf, int rule, uint32_t bits, long long base) {   // cf = this lane's count (0 if none)
        const int lr = rule_local[rule];
        const uint32_t nzl = __ballot_sync(FULL, cf != 0.f);
        for (int h0 = 0; h0 < H; h0 += 32) {
            float a = 0.f, b = 0.f;
            uint32_t todo = nzl;
            while (todo) {
                const int bq = __ffs(todo) - 1;
                todo &= todo - 1;
                const float cb = __shfl_sync(FULL, cf, bq);
                const long long idx = base + __popc(bits & ((1u << bq) - 1u));
                if (h0 + lane < H) {
                    a += cb * dA[idx * H + h0 + lane];
                    if (dB) b += cb * dB[idx * H + h0 + lane];
                }
            }
            if (h0 + lane < H) {
                if (a != 0.f) atomicAdd(gA + (size_t)lr * H + h0 + lane, a);
                if (dB && b != 0.f) atomicAdd(gB + (size_t)lr * H + h0 + lane, b);
            }
        }
    };
    if (blockIdx.x == 0 && warp == 0 && r.zr_ptr[q + 1] > r.zr_ptr[q]) {         // empty-body rules: count = one_hot(h)
        const int hq = s.lane_h[slot * RL_LANES + lane];
        for (int bq = 0; bq < 32; ++bq) {
            const int e = __shfl_sync(FULL, hq, bq);
            if (e < 0) continue;
            const uint32_t bits = ms[e];
            const long long base = co[e];
            for (int t = r.zr_ptr[q]; t < r.zr_ptr[q + 1]; ++t) contribute(lane == bq ? 1.f : 0.f, r.zr_rule[t], bits, base);
        }
    }
    const int n = fr.item_cnt[slot];
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    const int4 *it = reinterpret_cast<const int4 *>(fr.items) + fr.item_off[slot];
    for (int i = blockIdx.x * WARPS_PER_BLOCK + warp; i < n; i += PLUS_ITEM_BLOCKS * WARPS_PER_BLOCK) {
        const int4 rec = __ldg(it + i);                            // {row, first rule end, entity, rule ends}
        const float cf = (float)arena[(size_t)rec.x * RL_LANES + lane];
        const uint32_t bits = ms[rec.z];
        const long long base = co[rec.z];
        for (int t = rec.y; t < rec.y + rec.w; ++t) contribute(cf, r.node_term_rule[t], bits, base);
    }
}

// ------------------------------------------------------------------------------------------
// E-step statistics (Predictor.compute_H, src/predictors.py:82-119): per rule end and query,
// the count at the query's answer entity and the sum of the counts over all entities.
// Indexed by t - node_term_ptr[first node of the head] (the head's rules in node order).
// ------------------------------------------------------------------------------------------
template <typename CT>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_rule_stats(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, int max_terms, double *__restrict__ sum_cnt,
             double *__restrict__ pos_cnt)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.y;
    const int q = s.slot_head[slot];
    const int t_first = r.node_term_ptr[r.head_node_ptr[q]];
    const int ans = s.lane_t[slot * RL_LANES + lane];
    double *sums = sum_cnt + (size_t)slot * max_terms * RL_LANES;
    double *poss = pos_cnt + (size_t)slot * max_terms * RL_LANES;
    const int n = fr.item_cnt[slot];
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    const int4 *it = reinterpret_cast<const int4 *>(fr.items) + fr.item_off[slot];
    for (int i = blockIdx.x * WARPS_PER_BLOCK + warp; i < n; i += PLUS_ITEM_BLOCKS * WARPS_PER_BLOCK) {
        const int4 rec = __ldg(it + i);
        const CT c = arena[(size_t)rec.x * RL_LANES + lane];
        if (c == 0) continue;
        for (int t = rec.y; t < rec.y + rec.w; ++t) {
            atomicAdd(sums + (size_t)(t - t_first) * RL_LANES + lane, (double)c);
            if (rec.z == ans) poss[(size_t)(t - t_first) * RL_LANES + lane] = (double)c;
        }
    }
}


// ==========================================================================================
// PredictorPlus on candidate cells (rl_cells): aggregates per cell, backward into the rule embeddings.
// Cells are numbered by rl_cells_build before any count row is read again (the candidate words come from the
// items' lane masks), so one pass over the count rows produces the aggregates at their final place.
// ==========================================================================================
#define CH 16                                                     // hidden_dim of the cell kernels

// ---- PredictorPlus on the item list as k_numeric appended it: one thread per (item, quarter of the hidden vector) ----
#define PN_BLOCKS 16
// F[cell][16] += fp32(count) * emb[rule][16] (layers.py:68-72) with 16-byte vector atomics
template <typename CT>
__global__ void __launch_bounds__(256)
k_plus_item_features(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, rl_cells c, const float *__restrict__ emb,
                     float *__restrict__ F)
{
    const int slot = blockIdx.y;
    const int n = fr.item_cnt[slot];
    const long long ib = fr.item_off[slot];
    const int4 *items = reinterpret_cast<const int4 *>(fr.items) + ib;
    const uint32_t *masks = fr.item_mask + ib;
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    const size_t srow = (size_t)slot * g.num_entities;
    const int part = threadIdx.x & 3;
    for (int i = (blockIdx.x * 256 + threadIdx.x) >> 2; i < n; i += PN_BLOCKS * 64) {
        uint32_t m = __ldg(masks + i);
        if (!m) continue;
        const int4 it = __ldg(items + i);                         // {row, first rule end, entity, rule ends}
        float4 e4 = __ldg(reinterpret_cast<const float4 *>(emb + (size_t)__ldg(r.node_term_rule + it.y) * CH) + part);
        for (int t = it.y + 1; t < it.y + it.w; ++t) {            // duplicate rules: their embeddings add up
            const float4 x = __ldg(reinterpret_cast<const float4 *>(emb + (size_t)__ldg(r.node_term_rule + t) * CH) + part);
            e4.x += x.x; e4.y += x.y; e4.z += x.z; e4.w += x.w;
        }
        const uint32_t bits = c.nzmask[srow + it.z];
        const int off = c.cand_off[srow + it.z];
        const CT *row = arena + (size_t)it.x * RL_LANES;
        for (; m; m &= m - 1) {
            const int b = __ffs(m) - 1;
            const int cell = off + __popc(bits & ((1u << b) - 1u));
            if (cell >= c.cap) continue;
            const float v = (float)row[b];
            atomicAdd(reinterpret_cast<float4 *>(F + (size_t)cell * CH) + part, make_float4(v * e4.x, v * e4.y, v * e4.z, v * e4.w));
        }
    }
}

// empty-body rules: count = one_hot(h) -> the cell (h_b, b) gets the sum of their embeddings
__global__ void __launch_bounds__(128)
k_plus_zr_features(rl_graph g, rl_rules r, rl_slots s, rl_cells c, const float *__restrict__ emb, float *__restrict__ F)
{
    const int slot = blockIdx.x, b = threadIdx.x >> 2, part = threadIdx.x & 3;
    const int q = s.slot_head[slot];
    const int z0 = r.zr_ptr[q], z1 = r.zr_ptr[q + 1];
    if (z1 <= z0) return;
    const int h = s.lane_h[slot * RL_LANES + b];
    if (h < 0) return;
    const size_t srow = (size_t)slot * g.num_entities;
    const uint32_t bits = c.nzmask[srow + h];
    const int cell = c.cand_off[srow + h] + __popc(bits & ((1u << b) - 1u));
    if (cell >= c.cap) return;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int t = z0; t < z1; ++t) {
        const float4 e4 = __ldg(reinterpret_cast<const float4 *>(emb + (size_t)r.zr_rule[t] * CH) + part);
        a.x += e4.x; a.y += e4.y; a.z += e4.z; a.w += e4.w;
    }
    atomicAdd(reinterpret_cast<float4 *>(F + (size_t)cell * CH) + part, a);
}

// gEmb[rule][16] += sum over the item's non-zero queries of fp32(count) * dF[cell][16]: one vector atomic per
// (item, rule, quarter)
template <typename CT>
__global__ void __launch_bounds__(256)
k_plus_item_bwd(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, rl_cells c, const float *__restrict__ dF,
                float *__restrict__ gEmb)
{
    const int slot = blockIdx.y;
    const int n = fr.item_cnt[slot];
    const long long ib = fr.item_off[slot];
    const int4 *items = reinterpret_cast<const int4 *>(fr.items) + ib;
    const uint32_t *masks = fr.item_mask + ib;
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    const size_t srow = (size_t)slot * g.num_entities;
    const int part = threadIdx.x & 3;
    for (int i = (blockIdx.x * 256 + threadIdx.x) >> 2; i < n; i += PN_BLOCKS * 64) {
        uint32_t m = __ldg(masks + i);
        if (!m) continue;
        const int4 it = __ldg(items + i);
        const uint32_t bits = c.nzmask[srow + it.z];
        const int off = c.cand_off[srow + it.z];
        const CT *row = arena + (size_t)it.x * RL_LANES;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        for (; m; m &= m - 1) {
            const int b = __ffs(m) - 1;
            const int cell = off + __popc(bits & ((1u << b) - 1u));
            if (cell >= c.cap) continue;
            const float v = (float)row[b];
            const float4 d4 = __ldg(reinterpret_cast<const float4 *>(dF + (size_t)cell * CH) + part);
            a.x = fmaf(v, d4.x, a.x); a.y = fmaf(v, d4.y, a.y); a.z = fmaf(v, d4.z, a.z); a.w = fmaf(v, d4.w, a.w);
        }
        for (int t = it.y; t < it.y + it.w; ++t)
            atomicAdd(reinterpret_cast<float4 *>(gEmb + (size_t)__ldg(r.node_term_rule + t) * CH) + part, a);
    }
}

__global__ void __launch_bounds__(128)
k_plus_zr_bwd(rl_graph g, rl_rules r, rl_slots s, rl_cells c, const float *__restrict__ dF, float *__restrict__ gEmb)
{
    const int slot = blockIdx.x, b = threadIdx.x >> 2, part = threadIdx.x & 3;
    const int q = s.slot_head[slot];
    const int z0 = r.zr_ptr[q], z1 = r.zr_ptr[q + 1];
    if (z1 <= z0) return;
    const int h = s.lane_h[slot * RL_LANES + b];
    if (h < 0) return;
    const size_t srow = (size_t)slot * g.num_entities;
    const uint32_t bits = c.nzmask[srow + h];
    const int cell = c.cand_off[srow + h] + __popc(bits & ((1u << b) - 1u));
    if (cell >= c.cap) return;
    const float4 d4 = __ldg(reinterpret_cast<const float4 *>(dF + (size_t)cell * CH) + part);
    for (int t = z0; t < z1; ++t) atomicAdd(reinterpret_cast<float4 *>(gEmb + (size_t)r.zr_rule[t] * CH) + part, d4);
}

// ------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------
static int bad_frontier(const rl_frontier *fr)
{
    return !fr || !fr->arena || !fr->row_mask || !fr->node_cnt || !fr->items || !fr->items_sorted || !fr->item_cnt ||
           !fr->bucket_cnt || !fr->bucket_off || (fr->count_bits != 32 && fr->count_bits != 64);
}

static int no_item_arg(const rl_frontier *fr)
{
    return !fr || !fr->arena || !fr->items || !fr->item_off || !fr->item_cnt || !fr->item_mask ||
           (fr->count_bits != 32 && fr->count_bits != 64);
}

extern "C" {

int rl_plus_mask(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr, uint32_t *nzmask,
                 int32_t *cand_cnt, void *stream)
{
    if (!g || !r || !s || !nzmask || !cand_cnt || bad_frontier(fr)) return rl_fail(RL_ERR_ARG, "rl_plus_mask: bad argument");
    if (s->num_slots <= 0) return RL_OK;
    dim3 grid((g->rank_words + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, s->num_slots);
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = rl_sort_items(g, s, fr, stream);              // bucket the item list by entity word first
    if (rc != RL_OK) return rc;
    if (fr->count_bits == 32) k_plus_mask<uint32_t><<<grid, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, *fr, nzmask, cand_cnt);
    else k_plus_mask<unsigned long long><<<grid, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, *fr, nzmask, cand_cnt);
    CHECK_LAUNCH("k_plus_mask");
    return RL_OK;
}

int rl_plus_features(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                     const uint32_t *nzmask, const int64_t *cand_off, const int32_t *q_off, const int32_t *rule_local,
                     const float *emb, int32_t H, int32_t pna, float *out_sum, float *out_sq, float *out_min,
                     float *out_max, int32_t *arg_min, int32_t *arg_max, float *degree, int64_t *cand_query,
                     void *stream)
{
    if (!g || !r || !s || !nzmask || !cand_off || !q_off || !rule_local || !emb || !out_sum || !cand_query || bad_frontier(fr) || H <= 0)
        return rl_fail(RL_ERR_ARG, "rl_plus_features: bad argument");
    if (pna && (!out_sq || !out_min || !out_max || !arg_min || !arg_max || !degree))
        return rl_fail(RL_ERR_ARG, "rl_plus_features: PNA outputs missing");
    if (s->num_slots <= 0) return RL_OK;
    dim3 grid((g->rank_words + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, s->num_slots);
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH_FEAT(CT, P) k_plus_features<CT, P><<<grid, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, *fr, nzmask, cand_off, q_off, rule_local, emb, H, out_sum, out_sq, out_min, out_max, arg_min, arg_max, degree, cand_query)
    if (fr->count_bits == 32) { if (pna) LAUNCH_FEAT(uint32_t, true); else LAUNCH_FEAT(uint32_t, false); }
    else { if (pna) LAUNCH_FEAT(unsigned long long, true); else LAUNCH_FEAT(unsigned long long, false); }
#undef LAUNCH_FEAT
    CHECK_LAUNCH("k_plus_features");
    return RL_OK;
}

int rl_rule_stats(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr, int32_t max_terms,
                  double *sum_cnt, double *pos_cnt, void *stream)
{
    if (!g || !r || !s || !sum_cnt || !pos_cnt || no_item_arg(fr) || max_terms <= 0) return rl_fail(RL_ERR_ARG, "rl_rule_stats: bad argument");
    if (s->num_slots <= 0) return RL_OK;
    dim3 grid(PLUS_ITEM_BLOCKS, s->num_slots);
    cudaStream_t st = (cudaStream_t)stream;
    if (fr->count_bits == 32) k_rule_stats<uint32_t><<<grid, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, *fr, max_terms, sum_cnt, pos_cnt);
    else k_rule_stats<unsigned long long><<<grid, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, *fr, max_terms, sum_cnt, pos_cnt);
    CHECK_LAUNCH("k_rule_stats");
    return RL_OK;
}

int rl_plus_scatter(const rl_graph *g, const rl_slots *s, const uint32_t *nzmask, const int64_t *cand_off,
                    const float *zc, const float *bias, const float *extra, int32_t fill_neg_inf, float *Z, void *stream)
{
    if (!g || !s || !nzmask || !cand_off || !zc || !Z) return rl_fail(RL_ERR_ARG, "rl_plus_scatter: null argument");
    if (s->num_slots <= 0) return RL_OK;
    const size_t n = (size_t)g->num_entities * RL_LANES;
    k_plus_scatter<<<dim3((unsigned)((n + 255) / 256), s->num_slots), 256, 0, (cudaStream_t)stream>>>(
        g->num_entities, nzmask, cand_off, zc, bias, extra, fill_neg_inf, Z);
    CHECK_LAUNCH("k_plus_scatter");
    return RL_OK;
}

int rl_plus_gather(const rl_graph *g, const rl_slots *s, const uint32_t *nzmask, const int64_t *cand_off,
                   const float *G, float *dz, void *stream)
{
    if (!g || !s || !nzmask || !cand_off || !G || !dz) return rl_fail(RL_ERR_ARG, "rl_plus_gather: null argument");
    if (s->num_slots <= 0) return RL_OK;
    const size_t n = (size_t)g->num_entities * RL_LANES;
    k_plus_gather<<<dim3((unsigned)((n + 255) / 256), s->num_slots), 256, 0, (cudaStream_t)stream>>>(
        g->num_entities, nzmask, cand_off, G, dz);
    CHECK_LAUNCH("k_plus_gather");
    return RL_OK;
}

static int bad_cells_arg(const rl_cells *c)
{
    return !c || !c->counters || !c->nzmask || !c->cand_off || !c->cell_key || c->cap <= 0;
}

/* F must hold cap*16 floats; it is cleared here */
int rl_plus_item_features(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                         const rl_cells *c, const float *emb, int32_t H, float *F, void *stream)
{
    if (!g || !r || !s || !emb || !F || bad_cells_arg(c) || no_item_arg(fr)) return rl_fail(RL_ERR_ARG, "rl_plus_item_features: bad argument");
    if (H != CH) return rl_fail(RL_ERR_ARG, "rl_plus_item_features: built for hidden_dim 16");
    if (s->num_slots <= 0) return RL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(F, 0, (size_t)c->cap * CH * sizeof(float), st);
    if (e != cudaSuccess) return rl_fail(RL_ERR_CUDA, "rl_plus_item_features: memset", e);
    if (fr->count_bits == 32) k_plus_item_features<uint32_t><<<dim3(PN_BLOCKS, s->num_slots), 256, 0, st>>>(*g, *r, *s, *fr, *c, emb, F);
    else k_plus_item_features<unsigned long long><<<dim3(PN_BLOCKS, s->num_slots), 256, 0, st>>>(*g, *r, *s, *fr, *c, emb, F);
    CHECK_LAUNCH("k_plus_item_features");
    if (r->num_zero_rules > 0) {
        k_plus_zr_features<<<s->num_slots, 128, 0, st>>>(*g, *r, *s, *c, emb, F);
        CHECK_LAUNCH("k_plus_zr_features");
    }
    return RL_OK;
}

int rl_plus_item_backward(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                         const rl_cells *c, int32_t H, const float *dF, float *grad_emb, void *stream)
{
    if (!g || !r || !s || !dF || !grad_emb || bad_cells_arg(c) || no_item_arg(fr)) return rl_fail(RL_ERR_ARG, "rl_plus_item_backward: bad argument");
    if (H != CH) return rl_fail(RL_ERR_ARG, "rl_plus_item_backward: built for hidden_dim 16");
    if (s->num_slots <= 0) return RL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (fr->count_bits == 32) k_plus_item_bwd<uint32_t><<<dim3(PN_BLOCKS, s->num_slots), 256, 0, st>>>(*g, *r, *s, *fr, *c, dF, grad_emb);
    else k_plus_item_bwd<unsigned long long><<<dim3(PN_BLOCKS, s->num_slots), 256, 0, st>>>(*g, *r, *s, *fr, *c, dF, grad_emb);
    CHECK_LAUNCH("k_plus_item_bwd");
    if (r->num_zero_rules > 0) {
        k_plus_zr_bwd<<<s->num_slots, 128, 0, st>>>(*g, *r, *s, *c, dF, grad_emb);
        CHECK_LAUNCH("k_plus_zr_bwd");
    }
    return RL_OK;
}

int rl_plus_backward(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                     const uint32_t *nzmask, const int64_t *cand_off, const int32_t *rule_local, int32_t H,
                     const float *dA, const float *dB, int32_t max_terms, float *gA, float *gB, void *stream)
{
    if (!g || !r || !s || !nzmask || !cand_off || !rule_local || !dA || !gA || bad_frontier(fr) || H <= 0 || (dB && !gB))
        return rl_fail(RL_ERR_ARG, "rl_plus_backward: bad argument");
    if (s->num_slots <= 0) return RL_OK;
    (void)max_terms;
    dim3 grid(PLUS_ITEM_BLOCKS, s->num_slots);
    cudaStream_t st = (cudaStream_t)stream;
    if (fr->count_bits == 32) k_plus_backward<uint32_t><<<grid, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, *fr, nzmask, cand_off, rule_local, H, dA, dB, gA, gB);
    else k_plus_backward<unsigned long long><<<grid, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, *fr, nzmask, cand_off, rule_local, H, dA, dB, gA, gB);
    CHECK_LAUNCH("k_plus_backward");
    return RL_OK;
}

}  // extern "C"
