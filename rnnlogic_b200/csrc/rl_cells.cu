// rnnlogic_b200 -- the scoring half of the hot path on CANDIDATE CELLS instead of dense [N][32] matrices.
//
// A cell is a (query, entity) pair whose total path count is non-zero (src/predictors.py:224-225,239).
// With an entity bias every other logit of a query is just bias[e] (predictors.py:257-262: zeros scattered
// with the candidate scores, plus bias), so the all-entity softmax cross-entropy (src/trainer.py:88-89)
// splits exactly into one per-step scalar pair over all entities
//        Mg = max_e bias[e],   Sg = sum_e exp(bias[e] - Mg)
// plus corrections over a query's cells,
//        S_b = Sg * exp(Mg - M_b) + sum_cells [exp(bias[e] + z - M_b) - exp(bias[e] - M_b)],
// and the dense part of the bias gradient is rank one: exp(bias[e] - Mg) * K.  Without an entity feature
// (predictors.py:267-269: -inf outside the mask) the softmax runs over the cells alone.  Nothing of size
// [S][N][32] is written or read: per slot there are two int32 tables of N entries (candidate word + first
// cell) and per cell a score, a gradient, a key and an entity.  On the FB15k-237-shape workload 3.3 % of the
// (query, entity) pairs are cells.
//
// The counts arrive as the ITEM LIST of the frontier: k_numeric (rl_kernels.cu) appends one item per non-zero row of
// a rule-end node together with the row's lane mask (which queries are non-zero) and ORs that mask into the
// entity's candidate word.  Every kernel below is then one thread per item or one thread per cell with a few
// atomics -- no sort, no per-warp walks of ragged lists, and of a count row only the sectors of its non-zero
// lanes are read.
//
// Pipeline of a train step (all launches on one stream, no host sync):
//   rl_expand_level (items + lane masks + candidate words) -> rl_cells_build (number the cells) ->
//   scores per cell (rl_predictor_item_scores, or the PredictorPlus aggregate + MLP kernels) ->
//   rl_cells_softmax_ce (loss + gradient per cell + bias gradient) -> backward (rl_predictor_item_backward /
//   PredictorPlus kernels).
#include "rl_device.cuh"

#define ITEM_GRID 8            // blocks per slot of the thread-per-item kernels

// order-preserving float <-> unsigned key (atomicMax on floats of either sign)
__device__ __forceinline__ unsigned fkey(float v)
{
    const unsigned b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(unsigned k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

static int grid_for(long long n, int per_block, int max_blocks)
{
    long long b = (n + per_block - 1) / per_block;
    if (b < 1) b = 1;
    return (int)(b < max_blocks ? b : max_blocks);
}

// ------------------------------------------------------------------------------------------
// cell numbering: one block per slot.  Cells are numbered slot by slot (base from ONE atomicAdd per
// slot -- the order between slots is arbitrary and internal), entity-major, lane-minor.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512)
k_cell_scan(rl_graph g, rl_rules r, rl_slots s, rl_cells c)
{
    __shared__ int wsum[16];
    __shared__ int s_base;
    const int slot = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = g.num_entities;
    uint32_t *nz = c.nzmask + (size_t)slot * N;
    int32_t *off = c.cand_off + (size_t)slot * N;
    const int q = s.slot_head[slot];
    if (tid < 32) {
        if (r.zr_ptr[q + 1] > r.zr_ptr[q]) {                    // empty-body rules: count = one_hot(h) -> (h_b, b) is a cell
            const int h = s.lane_h[slot * RL_LANES + tid];
            if (h >= 0) atomicOr(nz + h, 1u << tid);
        }
        if (c.qmax) {                                           // per-query softmax statistics of rl_cells_softmax_ce
            c.qmax[slot * RL_LANES + tid] = fkey(-INFINITY);
            c.qsum[slot * RL_LANES + tid] = 0.f;
        }
    }
    __syncthreads();
    int tot = 0;
    for (int e = tid; e < N; e += 512) tot += __popc(__ldcg(nz + e));
    tot = warp_sumi(tot);
    if (lane == 0) wsum[warp] = tot;
    __syncthreads();
    if (tid == 0) {
        int t = 0;
        for (int k = 0; k < 16; ++k) t += wsum[k];
        s_base = atomicAdd(c.counters, t);
        c.slot_ncell[slot] = t;
        if ((long long)s_base + t > (long long)c.cap) c.counters[1] = 1;     // the step must be redone with larger arrays
    }
    __syncthreads();
    int carry = s_base;
    for (int e0 = 0; e0 < N; e0 += 512) {
        const int e = e0 + tid;
        uint32_t bits = e < N ? __ldcg(nz + e) : 0u;
        const int v = __popc(bits);
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        int wbase = 0, total = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const int t = wsum[k];
            if (k < warp) wbase += t;
            total += t;
        }
        int idx = carry + wbase + incl - v;
        if (e < N) off[e] = idx;
        while (bits) {                                          // cell -> (slot, lane) key and entity for the per-cell kernels
            const int b = __ffs(bits) - 1;
            bits &= bits - 1;
            if (idx < c.cap) {
                c.cell_key[idx] = slot * RL_LANES + b;
                c.cell_ent[idx] = e;
            }
            ++idx;
        }
        carry += total;
        __syncthreads();
    }
}

// Mg = max bias, Sg = sum exp(bias - Mg)
__global__ void __launch_bounds__(1024)
k_bias_stats(int N, const float *__restrict__ bias, double *__restrict__ acc)
{
    __shared__ float red_m[32];
    __shared__ double red_s[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float m = -INFINITY;
    for (int e = tid; e < N; e += 1024) m = fmaxf(m, bias[e]);
    m = warp_maxf(m);
    if (lane == 0) red_m[warp] = m;
    __syncthreads();
    m = red_m[0];
    for (int k = 1; k < 32; ++k) m = fmaxf(m, red_m[k]);
    double sum = 0.0;
    for (int e = tid; e < N; e += 1024) sum += (double)expf(bias[e] - m);
    sum = warp_sum(sum);
    if (lane == 0) red_s[warp] = sum;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int k = 0; k < 32; ++k) t += red_s[k];
        acc[0] = (double)m;
        acc[1] = t;
        acc[2] = 0.0;
    }
}

// ------------------------------------------------------------------------------------------
// Predictor (predictors.py:58-65): zc[cell] += w_rule * fp32(count).  One THREAD per item (= non-zero row of a
// rule-end node, in the order k_numeric appended them): it reads the counts of the queries in its lane mask
// (one 32-byte sector for the typical one or two) and adds to their cells.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int cell_of(const rl_cells &c, size_t srow, int e, int b)
{
    const uint32_t bits = c.nzmask[srow + e];
    return c.cand_off[srow + e] + __popc(bits & ((1u << b) - 1u));
}

template <typename CT>
__global__ void __launch_bounds__(256)
k_pred_item_fwd(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, rl_cells c, const float *__restrict__ w,
                float *__restrict__ zc)
{
    const int slot = blockIdx.y;
    const int n = fr.item_cnt[slot];
    const long long ib = fr.item_off[slot];
    const int4 *items = reinterpret_cast<const int4 *>(fr.items) + ib;
    const uint32_t *masks = fr.item_mask + ib;
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    const size_t srow = (size_t)slot * g.num_entities;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += ITEM_GRID * 256) {
        uint32_t m = __ldg(masks + i);
        if (!m) continue;
        const int4 it = __ldg(items + i);                         // {row, first rule end, entity, rule ends}
        float ws = __ldg(w + __ldg(r.node_term_rule + it.y));
        for (int t = it.y + 1; t < it.y + it.w; ++t) ws += __ldg(w + __ldg(r.node_term_rule + t));   // duplicate rules
        const uint32_t bits = c.nzmask[srow + it.z];
        const int off = c.cand_off[srow + it.z];
        const CT *row = arena + (size_t)it.x * RL_LANES;
        for (; m; m &= m - 1) {
            const int b = __ffs(m) - 1;
            const int cell = off + __popc(bits & ((1u << b) - 1u));
            if (cell < c.cap) atomicAdd(zc + cell, ws * (float)row[b]);       // x.float() * w (predictors.py:64)
        }
    }
}

// empty-body rules: count = one_hot(h) -> the cell (h_b, b) gets the sum of their weights
__global__ void __launch_bounds__(32)
k_pred_zr_fwd(rl_graph g, rl_rules r, rl_slots s, rl_cells c, const float *__restrict__ w, float *__restrict__ zc)
{
    const int lane = threadIdx.x, slot = blockIdx.x;
    const int q = s.slot_head[slot];
    const int z0 = r.zr_ptr[q], z1 = r.zr_ptr[q + 1];
    if (z1 <= z0) return;
    const int h = s.lane_h[slot * RL_LANES + lane];
    if (h < 0) return;
    double zsum = 0.0;
    for (int t = z0; t < z1; ++t) zsum += (double)__ldg(w + r.zr_rule[t]);
    const int cell = cell_of(c, (size_t)slot * g.num_entities, h, lane);
    if (cell < c.cap) atomicAdd(zc + cell, (float)zsum);
}

template <typename CT>
__global__ void __launch_bounds__(256)
k_pred_item_bwd(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, rl_cells c, const float *__restrict__ Gc,
                float *__restrict__ grad_w)
{
    const int slot = blockIdx.y;
    const int n = fr.item_cnt[slot];
    const long long ib = fr.item_off[slot];
    const int4 *items = reinterpret_cast<const int4 *>(fr.items) + ib;
    const uint32_t *masks = fr.item_mask + ib;
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    const size_t srow = (size_t)slot * g.num_entities;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += ITEM_GRID * 256) {
        uint32_t m = __ldg(masks + i);
        if (!m) continue;
        const int4 it = __ldg(items + i);
        const uint32_t bits = c.nzmask[srow + it.z];
        const int off = c.cand_off[srow + it.z];
        const CT *row = arena + (size_t)it.x * RL_LANES;
        float v = 0.f;
        for (; m; m &= m - 1) {
            const int b = __ffs(m) - 1;
            const int cell = off + __popc(bits & ((1u << b) - 1u));
            if (cell < c.cap) v = fmaf((float)row[b], Gc[cell], v);
        }
        if (v != 0.f)
            for (int t = it.y; t < it.y + it.w; ++t) atomicAdd(grad_w + __ldg(r.node_term_rule + t), v);
    }
}

__global__ void __launch_bounds__(32)
k_pred_zr_bwd(rl_graph g, rl_rules r, rl_slots s, rl_cells c, const float *__restrict__ Gc, float *__restrict__ grad_w)
{
    const int lane = threadIdx.x, slot = blockIdx.x;
    const int q = s.slot_head[slot];
    const int z0 = r.zr_ptr[q], z1 = r.zr_ptr[q + 1];
    if (z1 <= z0) return;
    const int h = s.lane_h[slot * RL_LANES + lane];
    double v = 0.0;
    if (h >= 0) {
        const int cell = cell_of(c, (size_t)slot * g.num_entities, h, lane);
        if (cell < c.cap) v = (double)Gc[cell];
    }
    v = warp_sum(v);
    if (lane == 0 && v != 0.0)
        for (int t = z0; t < z1; ++t) atomicAdd(grad_w + r.zr_rule[t], (float)v);
}

// ------------------------------------------------------------------------------------------
// log(softmax + 1e-8) CE on the cells (trainer.py:84,88-89)
// ------------------------------------------------------------------------------------------
// one thread per cell: per-query max of the cell logits, then per-query sum of exp(l - M) - exp(bias - M).
// The cells of a slot are contiguous (slots in the order their blocks numbered them), so the 256 consecutive cells of a
// block iteration belong to one or two slots -- the first cell's and the last cell's: their per-query partials are combined
// in shared memory first (2 x 32 entries) and reach the global per-query words with one atomic per touched query instead of
// one per cell; a cell of any other slot (tiny slots in between) goes to the global word directly.
__global__ void __launch_bounds__(256)
k_cell_max(rl_cells c, const float *__restrict__ bias, const float *__restrict__ zc)
{
    __shared__ uint32_t sm[64];
    const int n = min(c.counters[0], c.cap);
    for (int base = blockIdx.x * 256; base < n; base += gridDim.x * 256) {
        if (threadIdx.x < 64) sm[threadIdx.x] = 0u;                // fkey(x) > 0 for every float
        __syncthreads();
        const int ka = c.cell_key[base] & ~31, kb = c.cell_key[min(base + 255, n - 1)] & ~31;   // query words of the two slots
        const int i = base + threadIdx.x;
        if (i < n) {
            const float l = (bias ? bias[c.cell_ent[i]] : 0.f) + zc[i];
            const int key = c.cell_key[i], ks = key & ~31;
            if (ks == ka) atomicMax(sm + (key & 31), fkey(l));
            else if (ks == kb) atomicMax(sm + 32 + (key & 31), fkey(l));
            else atomicMax(c.qmax + key, fkey(l));
        }
        __syncthreads();
        if (threadIdx.x < 64 && sm[threadIdx.x]) atomicMax(c.qmax + (threadIdx.x < 32 ? ka : kb) + (threadIdx.x & 31), sm[threadIdx.x]);
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
k_cell_sum(rl_cells c, const float *__restrict__ bias, const double *__restrict__ acc, const float *__restrict__ zc)
{
    __shared__ float sm[64];
    const int n = min(c.counters[0], c.cap);
    const float Mg = bias ? (float)acc[0] : 0.f;
    for (int base = blockIdx.x * 256; base < n; base += gridDim.x * 256) {
        if (threadIdx.x < 64) sm[threadIdx.x] = 0.f;
        __syncthreads();
        const int ka = c.cell_key[base] & ~31, kb = c.cell_key[min(base + 255, n - 1)] & ~31;
        const int i = base + threadIdx.x;
        if (i < n) {
            const int key = c.cell_key[i], ks = key & ~31;
            const float bl = bias ? bias[c.cell_ent[i]] : 0.f;
            const float Mc = fkey_inv(c.qmax[key]);
            const float M = bias ? fmaxf(Mg, Mc) : Mc;
            const float v = expf(bl + zc[i] - M) - (bias ? expf(bl - M) : 0.f);
            if (v != 0.f) {
                if (ks == ka) atomicAdd(sm + (key & 31), v);
                else if (ks == kb) atomicAdd(sm + 32 + (key & 31), v);
                else atomicAdd(c.qsum + key, v);
            }
        }
        __syncthreads();
        if (threadIdx.x < 64 && sm[threadIdx.x] != 0.f) atomicAdd(c.qsum + (threadIdx.x < 32 ? ka : kb) + (threadIdx.x & 31), sm[threadIdx.x]);
        __syncthreads();
    }
}

// logit of (query b of the slot, entity e): bias[e] + cell score, or "no logit" (mask mode, not a cell)
__device__ __forceinline__ bool cell_logit(const rl_cells &c, const float *__restrict__ bias, const float *__restrict__ zc,
                                           size_t srow, int e, int b, float &l, int &idx)
{
    const uint32_t bits = c.nzmask[srow + e];
    idx = -1;
    l = bias ? bias[e] : 0.f;
    if ((bits >> b) & 1u) {
        idx = c.cand_off[srow + e] + __popc(bits & ((1u << b) - 1u));
        if (idx < c.cap) l += zc[idx]; else idx = -1;
        return true;
    }
    return bias != nullptr;
}

// one block per slot, one warp per query lane: (M_b, S_b) from the per-query statistics, then the sparse smoothed
// target of the query (data.py:207-212, trainer.py:84) -> loss sums.  stats[slot][lane] = (M, S, S_b, valid)
__global__ void __launch_bounds__(CE_WARPS * 32)
k_ce_targets(rl_graph g, rl_slots s, rl_cells c, rl_answers ans, float smoothing, const float *__restrict__ bias,
             const double *__restrict__ acc, const float *__restrict__ zc, float *__restrict__ stats,
             float *__restrict__ slot_lsum, float *__restrict__ slot_tsum)
{
    __shared__ double red_l[CE_WARPS], red_t[CE_WARPS];
    const int lane = threadIdx.x & 31, b = threadIdx.x >> 5;
    const int slot = blockIdx.x;
    const int N = g.num_entities;
    const int q = s.slot_head[slot];
    const size_t srow = (size_t)slot * N;
    const float Mc = fkey_inv(c.qmax[slot * RL_LANES + b]);
    float M, S;
    if (bias) {
        const float Mg = (float)acc[0];
        M = fmaxf(Mg, Mc);
        S = (float)(acc[1] * (double)expf(Mg - M) + (double)c.qsum[slot * RL_LANES + b]);
    } else {
        M = Mc;
        S = c.qsum[slot * RL_LANES + b];
    }
    const int h = s.lane_h[slot * RL_LANES + b];
    const int t = s.lane_t[slot * RL_LANES + b];
    float lsum = 0.f, tacc = 0.f, sb = 0.f;
    bool saw_t = false;
    const bool valid = h >= 0 && M != -INFINITY;
    if (valid) {
        auto term = [&](int e, float tg) {
            float l;
            int idx;
            if (!cell_logit(c, bias, zc, srow, e, b, l, idx)) return;       // outside the mask (trainer.py:89)
            const float p = expf(l - M) / S;
            lsum += logf(p + 1e-8f) * tg;
            tacc += tg;
            sb += tg / (p + 1e-8f) * p;
        };
        const int ki = find_key(ans, (long long)q * N + h);
        const int a0 = ki >= 0 ? ans.ptr[ki] : 0, a1 = ki >= 0 ? ans.ptr[ki + 1] : 0;
        for (int a = a0 + lane; a < a1; a += 32) {
            const int e = ans.ent[a];
            float tg = smoothing;
            if (e == t) { tg += 1.f - smoothing; saw_t = true; }
            term(e, tg);
        }
        saw_t = __any_sync(FULL, saw_t);
        if (!saw_t && t >= 0 && lane == 0) term(t, 1.f - smoothing);
    }
    lsum = warp_sumf(lsum);
    tacc = warp_sumf(tacc);
    sb = warp_sumf(sb);
    if (lane == 0) {
        float *st = stats + ((size_t)slot * 32 + b) * 4;
        st[0] = M; st[1] = S; st[2] = sb; st[3] = valid ? 1.f : 0.f;
        red_l[b] = (double)lsum;
        red_t[b] = (double)tacc;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double L = 0.0, T = 0.0;
        for (int k = 0; k < CE_WARPS; ++k) { L += red_l[k]; T += red_t[k]; }
        slot_tsum[slot] = (float)T;
        slot_lsum[slot] = (float)(-L);
    }
}

// Gc[cell] = scale * softmax * S_b / T'  (dense part of dloss/dlogit at the cells), and the bias gradient's
// correction at the cells: what the cell's logit contributes beyond the rank-one term exp(bias - M_b) * coef.
// After k_group_reduce: stats[.][3] = S_b / sum-exp / T'.  One thread per cell.
__global__ void __launch_bounds__(256)
k_grad_cells(rl_cells c, const float *__restrict__ bias, const float *__restrict__ zc, const float *__restrict__ stats,
             float scale, float *__restrict__ Gc, float *__restrict__ grad_bias)
{
    const int n = min(c.counters[0], c.cap);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        const float4 st = __ldg(reinterpret_cast<const float4 *>(stats) + c.cell_key[i]);
        const float coef = st.w * scale;
        float gq = 0.f;
        if (coef != 0.f) {
            const int e = c.cell_ent[i];
            const float bl = bias ? bias[e] : 0.f;
            gq = expf(bl + zc[i] - st.x) * coef;
            if (bias) {
                const float corr = gq - expf(bl - st.x) * coef;
                if (corr != 0.f) atomicAdd(grad_bias + e, corr);
            }
        }
        Gc[i] = gq;
    }
}

// target terms: dlogit -= scale * p * tgt / (p + eps) / T' at the target entries (one warp per query lane); also
// K = sum over queries of coef * exp(Mg - M_b), the factor of the rank-one bias gradient
__global__ void __launch_bounds__(CE_WARPS * 32)
k_grad_targets(rl_graph g, rl_slots s, rl_cells c, rl_answers ans, float smoothing, const float *__restrict__ bias,
               double *__restrict__ acc, const float *__restrict__ zc, const float *__restrict__ stats,
               const float *__restrict__ slot_invT, float scale, float *__restrict__ Gc, float *__restrict__ grad_bias)
{
    const int lane = threadIdx.x & 31, b = threadIdx.x >> 5;
    const int slot = blockIdx.x;
    const int N = g.num_entities;
    const int q = s.slot_head[slot];
    const float *st = stats + ((size_t)slot * 32 + b) * 4;
    if (st[3] == 0.f) return;
    const float M = st[0], S = st[1];
    if (bias && lane == 0) atomicAdd(acc + 2, (double)(st[3] * scale) * (double)expf((float)acc[0] - M));
    const float iT = slot_invT[slot] * scale;
    const int h = s.lane_h[slot * RL_LANES + b];
    const int t = s.lane_t[slot * RL_LANES + b];
    const size_t srow = (size_t)slot * N;
    auto apply = [&](int e, float tg) {
        float l;
        int idx;
        if (!cell_logit(c, bias, zc, srow, e, b, l, idx)) return;
        const float p = expf(l - M) / S;
        const float term = p * (tg / (p + 1e-8f)) * iT;
        if (idx >= 0) atomicAdd(Gc + idx, -term);
        if (grad_bias) atomicAdd(grad_bias + e, -term);
    };
    const int ki = find_key(ans, (long long)q * N + h);
    const int a0 = ki >= 0 ? ans.ptr[ki] : 0, a1 = ki >= 0 ? ans.ptr[ki + 1] : 0;
    bool saw_t = false;
    for (int a = a0 + lane; a < a1; a += 32) {
        const int e = ans.ent[a];
        float tg = smoothing;
        if (e == t) { tg += 1.f - smoothing; saw_t = true; }
        apply(e, tg);
    }
    saw_t = __any_sync(FULL, saw_t);
    if (!saw_t && t >= 0 && lane == 0) apply(t, 1.f - smoothing);
}

// the rank-one part of the bias gradient: every (query, entity) pair contributes exp(bias[e] - M_b) * coef_b
__global__ void __launch_bounds__(256)
k_bias_finish(int N, const float *__restrict__ bias, const double *__restrict__ acc, float *__restrict__ grad_bias)
{
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= N) return;
    grad_bias[e] += (float)(acc[2] * (double)expf(bias[e] - (float)acc[0]));
}

// ------------------------------------------------------------------------------------------
// filtered rank on the cells (trainer.py:189-201).  With a bias: #{e : logit > val} = #{e : bias[e] > val}
// (binary search in the sorted bias table) + corrections over the query's cells - the known answers.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
k_rank_vals(rl_graph g, rl_slots s, rl_cells c, const float *__restrict__ bias, const float *__restrict__ zc,
            float *__restrict__ vals)
{
    const int lane = threadIdx.x, slot = blockIdx.x;
    const int t = s.lane_t[slot * RL_LANES + lane];
    float val = INFINITY;
    if (t >= 0) {
        int idx;
        if (!cell_logit(c, bias, zc, (size_t)slot * g.num_entities, t, lane, val, idx)) val = INFINITY;
    }
    vals[slot * RL_LANES + lane] = val;
}

__global__ void __launch_bounds__(256)
k_rank_cells(rl_cells c, const float *__restrict__ bias, const float *__restrict__ zc, const float *__restrict__ vals,
             int32_t *__restrict__ counters)
{
    const int n = min(c.counters[0], c.cap);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        const int key = c.cell_key[i];
        const float val = vals[key];
        const float bl = bias ? bias[c.cell_ent[i]] : 0.f;
        const float l = bl + zc[i];
        const int gt = (l > val) - (bias ? (bl > val) : 0);
        const int ge = (l >= val) - (bias ? (bl >= val) : 0);
        if (gt) atomicAdd(counters + (size_t)key * 2, gt);
        if (ge) atomicAdd(counters + (size_t)key * 2 + 1, ge);
    }
}

__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_rank_cells_finalize(rl_graph g, rl_slots s, rl_cells c, rl_answers known, const float *__restrict__ bias,
                      const float *__restrict__ sorted_bias, const float *__restrict__ zc,
                      const int32_t *__restrict__ counters, int64_t *__restrict__ LH)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x;
    const int N = g.num_entities;
    const int q = s.slot_head[slot];
    const size_t srow = (size_t)slot * N;
    for (int b = warp; b < 32; b += WARPS_PER_BLOCK) {
        const int h = s.lane_h[slot * RL_LANES + b];
        const int t = s.lane_t[slot * RL_LANES + b];
        long long L = 0, H = 0;
        if (h >= 0 && t >= 0) {
            float val;
            int idx;
            if (!cell_logit(c, bias, zc, srow, t, b, val, idx)) { L = 1; H = (long long)N + 1; }   // mask[k,t] False (trainer.py:198-200)
            else {
                int gt = counters[((size_t)slot * 32 + b) * 2], ge = counters[((size_t)slot * 32 + b) * 2 + 1];
                if (bias) {                                     // entities whose logit is the bare bias: sorted table
                    int lo = 0, hi = N;                         // first index with sorted_bias > val
                    while (lo < hi) { const int mid = (lo + hi) >> 1; if (sorted_bias[mid] > val) hi = mid; else lo = mid + 1; }
                    gt += N - lo;
                    lo = 0; hi = N;                             // first index with sorted_bias >= val
                    while (lo < hi) { const int mid = (lo + hi) >> 1; if (sorted_bias[mid] >= val) hi = mid; else lo = mid + 1; }
                    ge += N - lo;
                }
                const int ki = find_key(known, (long long)q * N + h);
                const int a0 = ki >= 0 ? known.ptr[ki] : 0, a1 = ki >= 0 ? known.ptr[ki + 1] : 0;
                int fgt = 0, fge = 0;
                for (int a = a0 + lane; a < a1; a += 32) {      // flag False at the known answers (data.py:250-254)
                    float l;
                    int ix;
                    if (cell_logit(c, bias, zc, srow, known.ent[a], b, l, ix)) { fgt += l > val; fge += l >= val; }
                }
                fgt = warp_sumi(fgt);
                fge = warp_sumi(fge);
                L = (long long)(gt - fgt) + 1;
                H = (long long)(ge - fge) + 2;
            }
        }
        if (lane == 0) {
            LH[((size_t)slot * 32 + b) * 2] = L;
            LH[((size_t)slot * 32 + b) * 2 + 1] = H;
        }
    }
}

// ------------------------------------------------------------------------------------------
// cells <-> dense entity-major matrices (the RotatE entity feature is dense by nature; the [B,N] scores of forward())
// ------------------------------------------------------------------------------------------
// mode 0: Z[cell position] += zc     mode 1: Gc = G[cell position]
__global__ void __launch_bounds__(256)
k_cells_dense(int N, rl_cells c, float *__restrict__ cellv, float *__restrict__ dense, int mode)
{
    const int n = min(c.counters[0], c.cap);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        const int key = c.cell_key[i];
        float *d = dense + ((size_t)(key >> 5) * N + c.cell_ent[i]) * RL_LANES + (key & 31);
        if (mode == 0) *d += cellv[i]; else cellv[i] = *d;
    }
}

// ------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------
static int bad_cells(const rl_cells *c)
{
    return !c || !c->counters || !c->nzmask || !c->cand_off || !c->cell_key || !c->cell_ent || !c->slot_ncell || c->cap <= 0;
}
static int bad_item_frontier(const rl_frontier *fr)
{
    return !fr || !fr->arena || !fr->items || !fr->item_cnt || !fr->item_off || !fr->nzmask ||
           (fr->count_bits != 32 && fr->count_bits != 64);
}
extern "C" {

int rl_cells_build(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                   const rl_cells *c, void *stream)
{
    if (!g || !r || !s || bad_cells(c) || bad_item_frontier(fr)) return rl_fail(RL_ERR_ARG, "rl_cells_build: bad argument");
    if (c->nzmask != fr->nzmask) return rl_fail(RL_ERR_ARG, "rl_cells_build: cells and frontier must share nzmask");
    if ((c->qmax == nullptr) != (c->qsum == nullptr)) return rl_fail(RL_ERR_ARG, "rl_cells_build: qmax and qsum go together");
    if (s->num_slots <= 0) return RL_OK;
    if (!fr->item_mask) return rl_fail(RL_ERR_ARG, "rl_cells_build: the frontier was expanded without lane masks");
    if (fr->bucket_cnt)                                           // the sort, not k_numeric, fills nzmask of such a frontier
        return rl_fail(RL_ERR_ARG, "rl_cells_build: the frontier has sort buffers; expand it without bucket tables");
    k_cell_scan<<<s->num_slots, 512, 0, (cudaStream_t)stream>>>(*g, *r, *s, *c);
    CHECK_LAUNCH("k_cell_scan");
    return RL_OK;
}

int rl_bias_stats(int32_t N, const float *bias, double *acc, void *stream)
{
    if (!bias || !acc || N <= 0) return rl_fail(RL_ERR_ARG, "rl_bias_stats: bad argument");
    k_bias_stats<<<1, 1024, 0, (cudaStream_t)stream>>>(N, bias, acc);
    CHECK_LAUNCH("k_bias_stats");
    return RL_OK;
}

int rl_predictor_item_scores(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                             const rl_cells *c, const float *w, float *zc, void *stream)
{
    if (!g || !r || !s || !w || !zc || bad_cells(c) || bad_item_frontier(fr) || !fr->item_mask)
        return rl_fail(RL_ERR_ARG, "rl_predictor_item_scores: bad argument");
    if (s->num_slots <= 0) return RL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(zc, 0, (size_t)c->cap * sizeof(float), st);
    if (e != cudaSuccess) return rl_fail(RL_ERR_CUDA, "rl_predictor_item_scores: memset", e);
    const dim3 grid(ITEM_GRID, s->num_slots);
    if (fr->count_bits == 32) k_pred_item_fwd<uint32_t><<<grid, 256, 0, st>>>(*g, *r, *s, *fr, *c, w, zc);
    else k_pred_item_fwd<unsigned long long><<<grid, 256, 0, st>>>(*g, *r, *s, *fr, *c, w, zc);
    CHECK_LAUNCH("k_pred_item_fwd");
    if (r->num_zero_rules > 0) {
        k_pred_zr_fwd<<<s->num_slots, 32, 0, st>>>(*g, *r, *s, *c, w, zc);
        CHECK_LAUNCH("k_pred_zr_fwd");
    }
    return RL_OK;
}

int rl_predictor_item_backward(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                               const rl_cells *c, const float *Gc, float *grad_w, void *stream)
{
    if (!g || !r || !s || !Gc || !grad_w || bad_cells(c) || bad_item_frontier(fr) || !fr->item_mask)
        return rl_fail(RL_ERR_ARG, "rl_predictor_item_backward: bad argument");
    if (s->num_slots <= 0) return RL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 grid(ITEM_GRID, s->num_slots);
    if (fr->count_bits == 32) k_pred_item_bwd<uint32_t><<<grid, 256, 0, st>>>(*g, *r, *s, *fr, *c, Gc, grad_w);
    else k_pred_item_bwd<unsigned long long><<<grid, 256, 0, st>>>(*g, *r, *s, *fr, *c, Gc, grad_w);
    CHECK_LAUNCH("k_pred_item_bwd");
    if (r->num_zero_rules > 0) {
        k_pred_zr_bwd<<<s->num_slots, 32, 0, st>>>(*g, *r, *s, *c, Gc, grad_w);
        CHECK_LAUNCH("k_pred_zr_bwd");
    }
    return RL_OK;
}

int rl_cells_softmax_ce(const rl_graph *g, const rl_slots *s, const rl_cells *c, const rl_answers *ans, float smoothing,
                        const float *bias, double *acc, const float *zc, int32_t n_groups, const int32_t *group_ptr,
                        float grad_scale, float *stats, float *slot_sums, float *group_loss, float *group_tsum,
                        float *Gc, float *grad_bias, void *stream)
{
    if (!g || !s || !ans || !zc || !stats || !slot_sums || !group_loss || !group_tsum || bad_cells(c) || !c->qmax || !c->qsum)
        return rl_fail(RL_ERR_ARG, "rl_cells_softmax_ce: null argument");
    if (bias && !acc) return rl_fail(RL_ERR_ARG, "rl_cells_softmax_ce: bias needs the rl_bias_stats accumulator");
    if (Gc && bias && !grad_bias) return rl_fail(RL_ERR_ARG, "rl_cells_softmax_ce: bias needs grad_bias");
    const int S = s->num_slots, N = g->num_entities;
    if (S <= 0) return RL_OK;
    if (n_groups <= 0 || n_groups > S || (!group_ptr && n_groups != S)) return rl_fail(RL_ERR_ARG, "rl_cells_softmax_ce: bad group table");
    cudaStream_t st = (cudaStream_t)stream;
    float *slot_lsum = slot_sums, *slot_tsum = slot_sums + S, *slot_invT = slot_sums + 2 * (size_t)S;
    const int cgrid = grid_for(c->cap, 256 * 4, 148 * 8);
    k_cell_max<<<cgrid, 256, 0, st>>>(*c, bias, zc);
    CHECK_LAUNCH("k_cell_max");
    k_cell_sum<<<cgrid, 256, 0, st>>>(*c, bias, acc, zc);
    CHECK_LAUNCH("k_cell_sum");
    k_ce_targets<<<S, CE_WARPS * 32, 0, st>>>(*g, *s, *c, *ans, smoothing, bias, acc, zc, stats, slot_lsum, slot_tsum);
    CHECK_LAUNCH("k_ce_targets");
    k_group_reduce<<<n_groups, 32, 0, st>>>(n_groups, group_ptr, slot_lsum, slot_tsum, group_loss, group_tsum, slot_invT, stats);
    CHECK_LAUNCH("k_group_reduce");
    if (!Gc) return RL_OK;
    if (bias) {                                                  // K of the rank-one bias gradient, accumulated by k_grad_targets
        cudaError_t e = cudaMemsetAsync(acc + 2, 0, sizeof(double), st);
        if (e != cudaSuccess) return rl_fail(RL_ERR_CUDA, "rl_cells_softmax_ce: memset", e);
    }
    k_grad_cells<<<cgrid, 256, 0, st>>>(*c, bias, zc, stats, grad_scale, Gc, bias ? grad_bias : nullptr);
    CHECK_LAUNCH("k_grad_cells");
    k_grad_targets<<<S, CE_WARPS * 32, 0, st>>>(*g, *s, *c, *ans, smoothing, bias, acc, zc, stats, slot_invT, grad_scale, Gc,
                                                 bias ? grad_bias : nullptr);
    CHECK_LAUNCH("k_grad_targets");
    if (bias) {
        k_bias_finish<<<(N + 255) / 256, 256, 0, st>>>(N, bias, acc, grad_bias);
        CHECK_LAUNCH("k_bias_finish");
    }
    return RL_OK;
}

int rl_cells_rank(const rl_graph *g, const rl_slots *s, const rl_cells *c, const rl_answers *known, const float *bias,
                  const float *sorted_bias, const float *zc, int32_t *counters, int64_t *LH, void *stream)
{
    if (!g || !s || !known || !zc || !counters || !LH || bad_cells(c) || !c->qsum) return rl_fail(RL_ERR_ARG, "rl_cells_rank: null argument");
    if (bias && !sorted_bias) return rl_fail(RL_ERR_ARG, "rl_cells_rank: bias needs its ascending-sorted copy");
    const int S = s->num_slots;
    if (S <= 0) return RL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(counters, 0, (size_t)S * 64 * sizeof(int32_t), st);
    if (e != cudaSuccess) return rl_fail(RL_ERR_CUDA, "rl_cells_rank: memset", e);
    k_rank_vals<<<S, 32, 0, st>>>(*g, *s, *c, bias, zc, c->qsum);             // qsum doubles as the per-query target logit
    CHECK_LAUNCH("k_rank_vals");
    k_rank_cells<<<grid_for(c->cap, 256 * 4, 148 * 8), 256, 0, st>>>(*c, bias, zc, c->qsum, counters);
    CHECK_LAUNCH("k_rank_cells");
    k_rank_cells_finalize<<<S, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *s, *c, *known, bias, sorted_bias, zc, counters, LH);
    CHECK_LAUNCH("k_rank_cells_finalize");
    return RL_OK;
}

int rl_cells_add_to_dense(const rl_graph *g, const rl_slots *s, const rl_cells *c, const float *zc, float *Z, void *stream)
{
    if (!g || !s || !zc || !Z || bad_cells(c)) return rl_fail(RL_ERR_ARG, "rl_cells_add_to_dense: null argument");
    if (s->num_slots <= 0) return RL_OK;
    k_cells_dense<<<grid_for(c->cap, 256 * 4, 148 * 8), 256, 0, (cudaStream_t)stream>>>(g->num_entities, *c, const_cast<float *>(zc), Z, 0);
    CHECK_LAUNCH("k_cells_dense");
    return RL_OK;
}

int rl_cells_gather_dense(const rl_graph *g, const rl_slots *s, const rl_cells *c, const float *G, float *Gc, void *stream)
{
    if (!g || !s || !G || !Gc || bad_cells(c)) return rl_fail(RL_ERR_ARG, "rl_cells_gather_dense: null argument");
    if (s->num_slots <= 0) return RL_OK;
    k_cells_dense<<<grid_for(c->cap, 256 * 4, 148 * 8), 256, 0, (cudaStream_t)stream>>>(g->num_entities, *c, Gc, const_cast<float *>(G), 1);
    CHECK_LAUNCH("k_cells_dense");
    return RL_OK;
}

}  // extern "C"
