// rnnlogic_b200 -- hand-written sm_100a kernels + C-ABI (include/rnnlogic_b200.h).
//
// Hot path of RNNLogic's reasoning predictor (reference: src/data.py:136-173 grounding,
// src/predictors.py:53-80 aggregation, src/trainer.py:84-89 loss, :189-238 rank/metrics).
// All per-slot matrices are entity-major [row][32 lanes]: a warp owns rows, lane b owns query b,
// so every frontier / logit access is one coalesced 128-byte line.  This is HBM/L2-bound
// integer work: no tensor cores, the levers are coalescing, loads in flight and grid sizing.
#include "rl_device.cuh"
#include <limits.h>
#include <stdlib.h>

static thread_local char g_err[512] = "";
static long long g_launches = 0;   // kernels enqueued through this library (bench.py: gpu_launches)

int rl_fail(int code, const char *what, cudaError_t e)
{
    if (e != cudaSuccess) snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    else snprintf(g_err, sizeof(g_err), "%s", what);
    return code;
}
void rl_count_launch() { ++g_launches; }
static int fail(int code, const char *what, cudaError_t e = cudaSuccess) { return rl_fail(code, what, e); }

// ------------------------------------------------------------------------------------------
// slot preparation (trainer.py:69-82 batch tensors -> lane arrays)
// ------------------------------------------------------------------------------------------
__global__ void k_prepare_slots(rl_graph g, int S, const int32_t *__restrict__ slot_head,
                                const int32_t *__restrict__ q_off, const int64_t *__restrict__ all_h,
                                const int64_t *__restrict__ all_t, const int64_t *__restrict__ etr, int remove_query_edges,
                                int32_t *lane_h, int32_t *lane_t, int32_t *lane_eh, int32_t *lane_et)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S * RL_LANES) return;
    int s = i >> 5, lane = i & 31;
    int qi = q_off[s] + lane;
    bool valid = qi < q_off[s + 1];
    int64_t hv = valid ? all_h[qi] : -1, tv = (valid && all_t) ? all_t[qi] : -1;
    if (hv < 0 || hv >= g.num_entities) hv = -1;            // out-of-range ids become padding lanes
    if (tv < 0 || tv >= g.num_entities) tv = -1;
    lane_h[i] = (int32_t)hv;
    lane_t[i] = (int32_t)tv;
    int eh = -1, et = -1;
    const int rel = slot_head[s];
    if (valid && etr) {
        int64_t k = etr[qi];
        int64_t n = g.ord_ptr[rel + 1] - g.ord_ptr[rel];
        if (k >= 0 && k < n) {
            eh = g.ord_h[g.ord_ptr[rel] + k];
            et = g.ord_t[g.ord_ptr[rel] + k];
        }
    } else if (valid && remove_query_edges && hv >= 0 && tv >= 0) {
        // the query's own triple (h, head, t), when it is a train edge (data.py:214-216 looks its index up)
        const int row = rank_row(g, rel, (int)tv);
        if (row >= 0) {
            const long long grow = g.dst_ptr[rel] + row;
            for (long long k = g.row_start[grow]; k < g.row_start[grow + 1]; ++k)
                if (g.edge_src[k] == (int)hv) { eh = (int)hv; et = (int)tv; break; }
        }
    }
    lane_eh[i] = eh;
    lane_et[i] = et;
}

// ------------------------------------------------------------------------------------------
// kernel (1): frontier expansion, two launches per trie depth.
//
//  k_symbolic  one warp per (slot, trie node): decides WHICH destination rows of the node can be
//              non-zero.  It walks the valid rows of the parent frontier (bitmap), looks each
//              entity up in the relation's forward DCSR and ORs the reached destination rows into
//              the node's row bitmap (one 32-bit word per 32-row chunk).  A parent with more than
//              dense_num/dense_den of its rows valid switches the node to "all rows" (plain SpMM).
//  k_numeric   one warp per run of chunks: the valid rows of a trie node are expanded 32 at a time.
//              Depth > 1: warp-scan compaction of the rows' pair-table entries (the in-edges whose
//              source is a tail of the parent relation, already resolved to parent rows), coalesced
//              fetch, one parent-bitmap word per entry, then the live parent rows are pulled (128 B
//              each, lane = query, 8 loads in flight) and reduced per destination row.
//              Depth 1: each lane finds the tile's rows in the sorted forward list of its own query entity
//              (one binary search per tile and lane, then a merge).
//              Rows outside the bitmap are never written or read.  The query's own edge is cut with
//              an exact integer fix-up.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int srank_row(const rl_graph &g, int rel, int e)
{
    const uint2 w = __ldg(reinterpret_cast<const uint2 *>(g.srank_tab) + (size_t)rel * g.rank_words + (e >> 5));
    const uint32_t bit = 1u << (e & 31);
    return (w.x & bit) ? (int)(w.y + __popc(w.x & (bit - 1))) : -1;
}

__device__ __forceinline__ void mark_out_edges(const rl_graph &g, int rho, int ent, uint32_t *cm)
{
    const int sr = srank_row(g, rho, ent);
    if (sr < 0) return;
    const int fb = g.fsrc_ptr[rho] + sr;
    const int k1 = g.frow_start[fb + 1];
    for (int k = g.frow_start[fb]; k < k1; ++k) {
        const int dr = __ldg(g.fedge_dstrow + k);
        atomicOr(cm + (dr >> 5), 1u << (dr & 31));
    }
}

// Work item = (trie node, block of 32 parent bitmap words): hub relations with thousands of valid
// parent rows are spread over many warps instead of serialising in one.
template <bool ROOT>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_symbolic(rl_graph g, rl_rules r, rl_slots s, int depth, rl_frontier fr, int dense_num, int dense_den, int force_dense)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.y;
    const int q = s.slot_head[slot];
    const int32_t *ip = r.lvl_sym_ptr + (size_t)q * (r.max_len + 1);
    const int item = ip[depth - 1] + blockIdx.x * WARPS_PER_BLOCK + warp;
    if (item >= ip[depth]) return;
    const int v = r.sym_node[item], w0 = r.sym_w0[item];
    const int4 ra = __ldg(reinterpret_cast<const int4 *>(r.node_rec) + 2 * (size_t)v);
    const int4 rb4 = __ldg(reinterpret_cast<const int4 *>(r.node_rec) + 2 * (size_t)v + 1);
    const int rho = ra.x;
    const int D = rb4.x;
    const int nw = (D + 31) >> 5;
    if (nw == 0) return;
    const int hc0 = r.lvl_ptr[(size_t)q * (r.max_len + 1)];
    uint32_t *mbase = fr.row_mask + (size_t)s.mask_off[slot];
    uint32_t *cm = mbase + (rb4.y - hc0);
    const int nzb = s.nz_off[slot] - r.head_node_ptr[q];
    bool dense = force_dense != 0;
    const uint32_t *pm = nullptr;
    int rho_p = -1, Dp = 0;
    if (!ROOT) {
        const int p = ra.y;
        const int cntp = fr.node_cnt[nzb + p];
        if (!dense && cntp == 0) return;                       // empty parent => empty node
        rho_p = ra.z;
        Dp = g.dst_ptr[rho_p + 1] - g.dst_ptr[rho_p];
        if ((long long)cntp * dense_den > (long long)Dp * dense_num) dense = true;
        pm = mbase + (rb4.z - hc0);
    }
    if (dense) {
        if (w0 == 0)                                            // the node's first item fills the whole bitmap
            for (int w = lane; w < nw; w += 32)
                cm[w] = (w == nw - 1 && (D & 31)) ? ((1u << (D & 31)) - 1u) : 0xffffffffu;
        return;
    }
    if (ROOT) {
        const int h = s.lane_h[slot * RL_LANES + lane];
        if (h >= 0) mark_out_edges(g, rho, h, cm);
    } else {
        const int nwp = (Dp + 31) >> 5;
        const int pb = g.dst_ptr[rho_p];
        const int wi = w0 + lane;
        uint32_t word = wi < nwp ? pm[wi] : 0u;
        // spread the valid parent rows of these 32 words evenly over the lanes
        const int mine = __popc(word);
        int P = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, P, o);
            if (lane >= o) P += t;
        }
        const int T = __shfl_sync(FULL, P, 31);
        const int first = P - mine;
        for (int base = 0; base < T; base += 32) {
            const int k = min(base + lane, T - 1);
            int src_lane = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1)
                if (__shfl_sync(FULL, P, src_lane + step - 1) <= k) src_lane += step;
            const uint32_t wsel = __shfl_sync(FULL, word, src_lane);
            const int nth = k - __shfl_sync(FULL, first, src_lane);
            if (base + lane < T) {
                const int bit = __fns(wsel, 0, nth + 1);
                mark_out_edges(g, rho, __ldg(g.row_dst + pb + (w0 + src_lane) * 32 + bit), cm);
            }
        }
    }
}

#define EDGE_GROUP 8
#ifndef NUM_WARPS
#define NUM_WARPS 4             // warps per k_numeric block (2, 4, 8 measured within 1.5 % of each other)
#endif
// Up to 32 valid destination rows of node v, one per lane (myrow = row index inside the node, -1 =
// none).  Returns the lanes whose row ended up NON-ZERO (exact frontier support).
template <typename CT, bool ROOT, bool PRUNE>
__device__ __forceinline__ uint32_t numeric_rows(const rl_graph &g, const rl_rules &r, const rl_slots &s, const rl_frontier &fr,
                                                 int slot, int q, int hc0, const uint32_t *mbase, int v, int myrow,
                                                 int h, int lane_eh, int lane_et, bool &ovf)
{
    const int lane = threadIdx.x & 31;
    // one 32-byte node record instead of a chain of dependent look-ups
    const int4 ra = __ldg(reinterpret_cast<const int4 *>(r.node_rec) + 2 * (size_t)v);
    const int4 rb4 = __ldg(reinterpret_cast<const int4 *>(r.node_rec) + 2 * (size_t)v + 1);
    const int rho = ra.x, prel = ra.z, nterm = rb4.w;
    const size_t abase = (size_t)s.arena_off[slot];
    CT *arena = reinterpret_cast<CT *>(fr.arena);
    const CT *__restrict__ X = nullptr;
    const uint32_t *__restrict__ pm = nullptr;
    if (!ROOT) {
        X = arena + (abase + (size_t)r.node_prow_off[v]) * RL_LANES;
        pm = mbase + (rb4.z - hc0);
    }
    CT *__restrict__ Y = arena + (abase + (size_t)r.node_row_off[v]) * RL_LANES;
    const bool active = myrow >= 0;
    const int grow = ra.w + max(myrow, 0);                   // global row (dst_ptr[rel] + row)
    // depth 1: the row's in-edges; deeper: the row's entries of the (parent relation, relation) pair table --
    // only the in-edges whose source is a tail of the parent relation, already resolved to parent rows
    const int my_dst = active ? g.row_dst[grow] : -1;
    const bool masked = (rho == q);
    const int eh = masked ? lane_eh : -1;
    const int et = masked ? lane_et : -1;

    int cur = -1;
    unsigned long long acc = 0;
    uint32_t nzrows = 0;
    uint32_t my_lanes = 0;                                   // lane j: which queries of row j are non-zero
    auto flush = [&](int j) {
        if (masked) {                                        // warp-uniform: only hops over the head relation cut an edge
            const int d = __shfl_sync(FULL, my_dst, j);
            if (eh >= 0 && et == d) {                        // data.py:164-170: drop the query's own edge
                unsigned long long sub;
                if (ROOT) sub = (eh == h) ? 1ull : 0ull;
                else {
                    int pr = rank_row(g, prel, eh);
                    if (pr >= 0 && !((pm[pr >> 5] >> (pr & 31)) & 1u)) pr = -1;
                    sub = pr >= 0 ? (unsigned long long)X[(size_t)pr * RL_LANES + lane] : 0ull;
                }
                acc -= sub;
            }
        }
        if (sizeof(CT) == 4 && (acc >> 32)) ovf = true;
        const uint32_t nzl = __ballot_sync(FULL, acc != 0);
        if (!PRUNE || nzl) {                                 // all-zero rows are dropped from the bitmap
            Y[(size_t)__shfl_sync(FULL, myrow, j) * RL_LANES + lane] = (CT)acc;
            nzrows |= 1u << j;
            if (lane == j) my_lanes = nzl;
        }
        acc = 0;
    };

    constexpr bool SEARCH = ROOT && PRUNE;                    // dense mode (every row of a node) keeps the streaming in-edge scan
    if (SEARCH) {
        // Depth 1: the count of row d for query b is the multiplicity of the edge (h_b -> d), found in the SORTED
        // forward list of h_b under this relation (forward DCSR).  The tile's rows ascend with the lane (the active
        // lanes are a prefix), so each lane finds the part of its list inside [first row, last row] of the tile with
        // ONE binary search and matches those few entries to the tile's rows by a search over the lanes -- instead of
        // one search per (row, lane): most rows are non-zero for one or two queries only.
        auto own_edges = [&](int &fs, int &fe) {             // h's forward list under this relation
            fs = fe = 0;
            const int sr = h >= 0 ? srank_row(g, rho, h) : -1;
            if (sr >= 0) {
                const int fb = g.fsrc_ptr[rho] + sr;
                fs = g.frow_start[fb];
                fe = g.frow_start[fb + 1];
            }
        };
        int lo, fe;
        own_edges(lo, fe);
        const uint32_t act = __ballot_sync(FULL, active);
        const int key = active ? myrow : INT_MAX;
        const int r_lo = __shfl_sync(FULL, myrow, 0), r_hi = __shfl_sync(FULL, myrow, __popc(act) - 1);
        for (int hi = fe; lo < hi;) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(g.fedge_dstrow + mid) < r_lo) lo = mid + 1; else hi = mid;
        }
        uint32_t hit = 0;                                    // bit j: the edge (h -> row of lane j) exists
        bool multi = false;                                  // ... more than once (parallel edges)
        int d = lo < fe ? __ldg(g.fedge_dstrow + lo) : INT_MAX;
        while (__any_sync(FULL, d <= r_hi)) {
            int j = 0;                                       // #lanes whose row is < d
#pragma unroll
            for (int step = 16; step > 0; step >>= 1)
                if (__shfl_sync(FULL, key, j + step - 1) < d) j += step;
            const bool match = __shfl_sync(FULL, key, j & 31) == d && j < 32 && d <= r_hi;
            if (match) {
                multi |= (hit >> j) & 1u;
                hit |= 1u << j;
            }
            if (d <= r_hi) d = ++lo < fe ? __ldg(g.fedge_dstrow + lo) : INT_MAX;
        }
        for (uint32_t todo = act; todo; todo &= todo - 1) {
            const int j = __ffs(todo) - 1;
            const int rj = __shfl_sync(FULL, myrow, j);
            acc = (hit >> j) & 1u;
            if (multi && acc) {                              // a repeated triple (KnowledgeGraph rejects them): count it
                int a, b;
                own_edges(a, b);
                const int end = b;
                while (a < b) {
                    const int mid = (a + b) >> 1;
                    if (__ldg(g.fedge_dstrow + mid) < rj) a = mid + 1; else b = mid;
                }
                int cnt = 0;
                while (a + cnt < end && __ldg(g.fedge_dstrow + a + cnt) == rj) ++cnt;
                acc = (unsigned long long)cnt;
            }
            flush(j);
        }
    } else {
    const int32_t *__restrict__ rs = ROOT ? g.row_start + grow : r.pair_ptr + (r.node_pair_off[v] + max(myrow, 0));
    const int my_rs = active ? rs[0] : 0;
    const int my_re = active ? rs[1] : 0;
    const int deg = my_re - my_rs;
    int P = deg;                                            // inclusive scan of deg over lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL, P, o);
        if (lane >= o) P += t;
    }
    const int T = __shfl_sync(FULL, P, 31);
    const int my_first = P - deg;                            // position of my row's first entry in the list
    for (int base = 0; base < T; base += 32) {
        const int n = min(32, T - base);
        const int k = min(base + lane, T - 1);
        int row = 0;                                         // #lanes with P <= k  (binary search over lanes)
#pragma unroll
        for (int step = 16; step > 0; step >>= 1)
            if (__shfl_sync(FULL, P, row + step - 1) <= k) row += step;
        const int e = __shfl_sync(FULL, my_rs, row) + (k - __shfl_sync(FULL, my_first, row));
        const int src = lane < n ? __ldg((ROOT ? g.edge_src : r.pair_ent) + e) : -1;     // ROOT: source entity; else: parent row
        int pr = -1;
        if (!ROOT && src >= 0 && ((pm[src >> 5] >> (src & 31)) & 1u)) pr = src;
        // only entries whose parent row is non-zero are pulled (ROOT: every in-edge, the value is a compare)
        uint32_t todo = ROOT ? (n == 32 ? FULL : ((1u << n) - 1u)) : __ballot_sync(FULL, pr >= 0);
        while (todo) {
            CT vals[EDGE_GROUP];
            int rws[EDGE_GROUP];
#pragma unroll
            for (int u = 0; u < EDGE_GROUP; ++u) {           // EDGE_GROUP row loads in flight
                const int kk = todo ? __ffs(todo) - 1 : -1;
                todo &= todo - 1;
                rws[u] = kk >= 0 ? __shfl_sync(FULL, row, kk) : -1;
                if (ROOT) {
                    const int sv = __shfl_sync(FULL, src, kk & 31);
                    vals[u] = (CT)((kk >= 0) && (sv == h));
                } else {
                    const int p = __shfl_sync(FULL, pr, kk & 31);
                    vals[u] = kk >= 0 ? X[(size_t)p * RL_LANES + lane] : (CT)0;
                }
            }
#pragma unroll
            for (int u = 0; u < EDGE_GROUP; ++u) {
                if (rws[u] >= 0) {
                    if (rws[u] != cur) {
                        if (cur >= 0) flush(cur);
                        cur = rws[u];
                    }
                    acc += (unsigned long long)vals[u];
                }
            }
        }
    }
    if (cur >= 0) flush(cur);
    }
    if (nterm > 0 && nzrows) {
        const bool mine = (nzrows >> lane) & 1u;
        if (fr.items) {                                      // {row, first rule end, entity, rule ends} items for the aggregation / backward
            const int term0 = __ldg(r.node_term_ptr + v);
            int base = 0;
            if (lane == 0) base = atomicAdd(fr.item_cnt + slot, __popc(nzrows));
            base = __shfl_sync(FULL, base, 0);
            if (mine) {
                const long long pos = fr.item_off[slot] + base + __popc(nzrows & ((1u << lane) - 1u));
                reinterpret_cast<int4 *>(fr.items)[pos] = make_int4((int)(r.node_row_off[v] + myrow), term0, my_dst, nterm);
                if (fr.item_mask) fr.item_mask[pos] = my_lanes;
                if (fr.bucket_cnt) atomicAdd(fr.bucket_cnt + (size_t)slot * RL_BUCKET_STRIDE(g.rank_words) + my_dst, 1);
                else if (fr.nzmask && my_lanes) atomicOr(fr.nzmask + (size_t)slot * g.num_entities + my_dst, my_lanes);
            }
        }
    }
    return nzrows;
}

// One warp = cpw consecutive chunks of one slot at this depth: their valid-row words are read with
// one coalesced load, then the valid rows of all chunks of the same trie node are merged and expanded
// 32 at a time (full tiles even when each chunk holds only a few valid rows).
template <typename CT, bool ROOT, bool PRUNE>
__global__ void __launch_bounds__(NUM_WARPS * 32, 48 / NUM_WARPS)    // <= 40 registers, 48 warps per SM -- latency-bound; small blocks so a slow warp strands few slots
k_numeric(rl_graph g, rl_rules r, rl_slots s, int depth, rl_frontier fr, int cpw)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.y;
    const int q = s.slot_head[slot];
    const int32_t *lp = r.lvl_ptr + (size_t)q * (r.max_len + 1);
    const int c_end = lp[depth];
    const int c0 = lp[depth - 1] + (blockIdx.x * NUM_WARPS + warp) * cpw;   // cpw (<= 32) chunks per warp
    if (c0 >= c_end) return;
    const int hc0 = lp[0];
    uint32_t *mbase = fr.row_mask + (size_t)s.mask_off[slot];
    const int nzb = s.nz_off[slot] - r.head_node_ptr[q];
    const int my_chunk = c0 + lane;
    const bool mine = lane < cpw && my_chunk < c_end;
    const uint32_t my_m = mine ? mbase[my_chunk - hc0] : 0u;
    uint32_t todo = __ballot_sync(FULL, my_m != 0u);
    if (todo == 0u) return;
    const int my_node = my_m ? r.chunk_node[my_chunk] : -1;
    const int my_row0 = my_m ? r.chunk_row0[my_chunk] : 0;
    const int h = s.lane_h[slot * RL_LANES + lane];
    const int leh = s.lane_eh[slot * RL_LANES + lane];
    const int let_ = s.lane_et[slot * RL_LANES + lane];
    bool ovf = false;
    int rows_done = 0;                                           // non-zero rows this warp produced (level statistic)
    while (todo) {
        const int v = __shfl_sync(FULL, my_node, __ffs(todo) - 1);
        const uint32_t seg = __ballot_sync(FULL, my_m != 0u && my_node == v);       // this node's chunks in my range
        todo &= ~seg;
        const int cnt = ((seg >> lane) & 1u) ? __popc(my_m) : 0;
        int P = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, P, o);
            if (lane >= o) P += t;
        }
        const int V = __shfl_sync(FULL, P, 31);
        const int first = P - cnt;
        for (int g0 = 0; g0 < V; g0 += 32) {
            const bool have = g0 + lane < V;
            const int k = min(g0 + lane, V - 1);
            int sl = 0;                                                             // lane holding the k-th valid row's chunk
#pragma unroll
            for (int step = 16; step > 0; step >>= 1)
                if (__shfl_sync(FULL, P, sl + step - 1) <= k) sl += step;
            const uint32_t wsel = __shfl_sync(FULL, my_m, sl);
            const int nth = k - __shfl_sync(FULL, first, sl);
            const int r0 = __shfl_sync(FULL, my_row0, sl);
            const int bit = __fns(wsel, 0, nth + 1);
            const int myrow = have ? r0 + bit : -1;
            const uint32_t nz = numeric_rows<CT, ROOT, PRUNE>(g, r, s, fr, slot, q, hc0, mbase, v, myrow, h, leh, let_, ovf);
            if (have && !((nz >> lane) & 1u)) atomicAnd(mbase + (c0 + sl - hc0), ~(1u << bit));   // bitmap = exact support
            if (lane == 0 && nz) atomicAdd(fr.node_cnt + nzb + v, __popc(nz));
            rows_done += __popc(nz);
        }
    }
    // overflow[1 + depth]: non-zero rows of this depth over the whole call -- the host sizes the next call's launch with it
    if (lane == 0 && rows_done && depth < 8) atomicAdd(fr.overflow + 1 + depth, rows_done);
    if (__any_sync(FULL, ovf) && lane == 0) fr.overflow[0] = 1;
}

// Pair tables (built once per rule set): for every (parent relation rp, relation rr) that occurs as a hop of some trie and
// every destination row d of rr, the in-edges of d whose SOURCE is a tail of rp, stored as the source's row index under
// rp.  That map depends only on the relation pair, not on the query, so k_numeric neither looks sources up in the rank
// table nor touches the in-edges that can never carry a count.  One block per pair; FILL = false counts
// (out[base + d]; out[base + D] = 0 closes the pair), FILL = true writes the entries at ptr[base + d].
template <bool FILL>
__global__ void __launch_bounds__(128)
k_pair_table(rl_graph g, const int32_t *__restrict__ pair_prel, const int32_t *__restrict__ pair_rel,
             const int64_t *__restrict__ pair_base, const int32_t *__restrict__ ptr, int32_t *__restrict__ out)
{
    const int p = blockIdx.x;
    const int rp = pair_prel[p], rr = pair_rel[p];
    const long long base = pair_base[p];
    const int row0 = g.dst_ptr[rr], D = g.dst_ptr[rr + 1] - row0;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        int n = 0;
        const int pos = FILL ? ptr[base + d] : 0;
        const int k1 = g.row_start[row0 + d + 1];
        for (int k = g.row_start[row0 + d]; k < k1; ++k) {
            const int pr = rank_row(g, rp, __ldg(g.edge_src + k));
            if (pr >= 0) {
                if (FILL) out[pos + n] = pr;
                ++n;
            }
        }
        if (!FILL) out[base + d] = n;
    }
    if (!FILL && threadIdx.x == 0) out[base + D] = 0;
}

// One hop from an ARBITRARY dense frontier (KnowledgeGraph.propagate, src/data.py:149-173):
// out[t][b] = sum over the relation's edges (s -> t) of x[s][b], minus x[h_k][b] at t_k for the edge
// k = edges_to_remove[b] of query b (data.py:164-170 zeroes message[k][b]).  x / out are the reference's
// int64 [N][B] (entity-major already); one warp per entity, lanes stride over the B queries.
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_propagate_dense(rl_graph g, int rel, int B, const int64_t *__restrict__ x, const int64_t *__restrict__ etr,
                  int64_t *__restrict__ out)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int e = blockIdx.x * WARPS_PER_BLOCK + warp;
    if (e >= g.num_entities) return;
    const int row = rank_row(g, rel, e);
    const long long o0 = g.ord_ptr[rel], n_ord = g.ord_ptr[rel + 1] - o0;
    for (int b = lane; b < B; b += 32) {
        unsigned long long acc = 0;                          // wraps exactly like the reference's int64
        if (row >= 0) {
            const long long grow = g.dst_ptr[rel] + row;
            for (int k = g.row_start[grow]; k < g.row_start[grow + 1]; ++k)
                acc += (unsigned long long)x[(size_t)g.edge_src[k] * B + b];
            if (etr) {
                const long long k = etr[b];
                if (k >= 0 && k < n_ord && g.ord_t[o0 + k] == e) acc -= (unsigned long long)x[(size_t)g.ord_h[o0 + k] * B + b];
            }
        }
        out[(size_t)e * B + b] = (int64_t)acc;
    }
}

// dense int64 [32][N] view of one node (debug / KnowledgeGraph.grounding return value)
template <typename CT>
__global__ void k_node_dense(rl_graph g, rl_rules r, rl_slots s, int slot, int node, rl_frontier fr,
                             int64_t *__restrict__ out)
{
    __shared__ long long tile[32][33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;     // 32 warps
    const int N = g.num_entities;
    const int e = blockIdx.x * 32 + w;
    long long c = 0;
    if (e < N) {
        if (node < 0) c = (s.lane_h[slot * RL_LANES + lane] == e);
        else {
            const int q = s.slot_head[slot];
            const int hc0 = r.lvl_ptr[(size_t)q * (r.max_len + 1)];
            const uint32_t *mbase = fr.row_mask + (size_t)s.mask_off[slot];
            const int row = rank_row(g, r.node_rel[node], e);
            if (row >= 0 && row_valid(r.node_chunk0, mbase, hc0, node, row))
                c = (long long)reinterpret_cast<const CT *>(fr.arena)[((size_t)s.arena_off[slot] + r.node_row_off[node] + row) * RL_LANES + lane];
        }
    }
    tile[w][lane] = c;                                            // [entity][lane]
    __syncthreads();
    const int eo = blockIdx.x * 32 + lane;
    if (eo < N) out[(size_t)w * N + eo] = tile[lane][w];          // lane-major row w
}

// ------------------------------------------------------------------------------------------
// kernel (2a): rule-weight aggregation from the item list.  k_numeric appended one item
// {row, first rule end, entity, rule ends} per NON-ZERO row of every rule-end node (exactly the rows that
// contribute; the rules ending at the node are node_term_rule[first .. first + n)).
// k_items_sort buckets the items of a slot by entity word (counting sort); k_predictor_scores then
// gives one warp the 32 entities of a word: default rows (bias / -inf, empty-body rules) for entities
// without items, and for the others an fp64 accumulation of fp32(count) * w over their items.
// No table walk: work is proportional to the non-zero terminal rows.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512)
k_items_scan(int W, rl_frontier fr)
{
    // exclusive scan of the slot's per-entity item counts; one thread owns the 32 entities of a word (8 x int4)
    __shared__ int wsum[16];
    const int slot = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int4 *cnt4 = reinterpret_cast<int4 *>(fr.bucket_cnt + (size_t)slot * RL_BUCKET_STRIDE(W));
    int4 *off4 = reinterpret_cast<int4 *>(fr.bucket_off + (size_t)slot * RL_BUCKET_STRIDE(W));
    int carry = 0;
    for (int w0 = 0; w0 < W; w0 += 512) {
        const int w = w0 + tid;
        int4 c[8];
        int sum = 0;
        if (w < W) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                c[k] = cnt4[(size_t)w * 8 + k];
                sum += (c[k].x + c[k].y) + (c[k].z + c[k].w);
            }
        }
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        int wbase = 0, total = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const int v = wsum[k];
            if (k < warp) wbase += v;
            total += v;
        }
        int run = carry + wbase + incl - sum;
        if (w < W) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                int4 o;
                o.x = run; run += c[k].x;
                o.y = run; run += c[k].y;
                o.z = run; run += c[k].z;
                o.w = run; run += c[k].w;
                off4[(size_t)w * 8 + k] = o;
                cnt4[(size_t)w * 8 + k] = make_int4(0, 0, 0, 0);      // becomes the scatter cursor
            }
        }
        carry += total;
        __syncthreads();
    }
    if (tid == 0) fr.bucket_off[(size_t)slot * RL_BUCKET_STRIDE(W) + (size_t)W * 32] = carry;
}

#define SCATTER_BLOCKS 16
__global__ void __launch_bounds__(256)
k_items_scatter(int N, int W, rl_frontier fr)
{
    const int slot = blockIdx.y;
    int *cnt = fr.bucket_cnt + (size_t)slot * RL_BUCKET_STRIDE(W);
    const int *off = fr.bucket_off + (size_t)slot * RL_BUCKET_STRIDE(W);
    const int n = fr.item_cnt[slot];
    const int4 *in = reinterpret_cast<const int4 *>(fr.items) + fr.item_off[slot];
    int4 *out = reinterpret_cast<int4 *>(fr.items_sorted) + fr.item_off[slot];
    const uint32_t *min_ = fr.item_mask ? fr.item_mask + fr.item_off[slot] : nullptr;
    uint32_t *mout = fr.item_mask_sorted ? fr.item_mask_sorted + fr.item_off[slot] : nullptr;
    uint32_t *nz = fr.nzmask ? fr.nzmask + (size_t)slot * N : nullptr;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += SCATTER_BLOCKS * 256) {
        const int4 it = in[i];
        const int pos = off[it.z] + atomicAdd(cnt + it.z, 1);     // cnt ends as the per-entity item counts again
        out[pos] = it;
        if (min_ && mout) {
            const uint32_t m = min_[i];
            mout[pos] = m;
            if (nz && m) atomicOr(nz + it.z, m);                  // candidate word of the entity
        }
    }
}

static int launch_items_sort(const rl_graph *g, const rl_slots *s, const rl_frontier *fr, cudaStream_t st)
{
    k_items_scan<<<s->num_slots, 512, 0, st>>>(g->rank_words, *fr);
    CHECK_LAUNCH("k_items_scan");
    k_items_scatter<<<dim3(SCATTER_BLOCKS, s->num_slots), 256, 0, st>>>(g->num_entities, g->rank_words, *fr);
    CHECK_LAUNCH("k_items_scatter");
    return RL_OK;
}

template <typename CT>
__global__ void __launch_bounds__(SCORE_WARPS_MAX * 32, SCORE_MIN_BLOCKS)       
k_predictor_scores(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, const float *__restrict__ w,
                   const float *__restrict__ bias, int fill_neg_inf, float *__restrict__ Z,
                   uint32_t *__restrict__ nzmask, float *__restrict__ partial)
{
    __shared__ float sm_m[SCORE_WARPS_MAX][32];
    __shared__ float sm_s[SCORE_WARPS_MAX][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int slot = blockIdx.y;
    const int ew = blockIdx.x * nwarps + warp;                    // entity word
    const int N = g.num_entities, W = g.rank_words;
    float run_m = -INFINITY;                                      // online softmax of the lane's query over the warp's rows
    float run_s = 0.f;
    if (ew < W) {
    const int q = s.slot_head[slot];
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    const int h = s.lane_h[slot * RL_LANES + lane];
    const int z0 = r.zr_ptr[q], z1 = r.zr_ptr[q + 1];
    double zsum = 0.0;
    if (z1 > z0) for (int t = z0; t < z1; ++t) zsum += (double)__ldg(w + r.zr_rule[t]);
    float *Zs = Z + (size_t)slot * N * RL_LANES;
    uint32_t *ms = nzmask + (size_t)slot * N;
    const int e1 = min(32, N - ew * 32);
    const float bias_l = (bias && lane < e1) ? bias[ew * 32 + lane] : 0.f;      // lane i: bias of entity i of the word
    uint32_t my_bits = 0u;                                                       // lane i: nzmask word of entity i
    auto finish = [&](int i, double acc, bool any) {              // one logit row (all lanes) + its nzmask word
        const int e = ew * 32 + i;
        if (z1 > z0 && h == e) { acc += zsum; any = true; }       // empty-body rules: count = one_hot(h)
        float z = (float)acc + __shfl_sync(FULL, bias_l, i);
        if (fill_neg_inf && !any) z = -INFINITY;
        Zs[(size_t)e * RL_LANES + lane] = z;
        const uint32_t bits = __ballot_sync(FULL, any);
        if (lane == i) my_bits = bits;
        if (partial && z != -INFINITY) {
            const float mn = fmaxf(run_m, z);                     // branch-free online softmax (<= 32 rows per warp, fp32)
            run_s = run_s * expf(run_m - mn) + expf(z - mn);
            run_m = mn;
        }
    };
    WordItems wi = load_word_items(fr, s, W, slot, ew);
    // Entities without items have the same logit for every query (bias[e], or -inf): their rows are plain
    // broadcast stores and their softmax share is one warp reduction -- unless a query's head sits there
    // and the head relation has empty-body rules, then the entity takes the general path.
    uint32_t slow = wi.present;
    if (z1 > z0) slow |= __reduce_or_sync(FULL, (h >= 0 && (h >> 5) == ew) ? 1u << (h & 31) : 0u);
    const uint32_t fast = ~slow & (e1 == 32 ? FULL : (1u << e1) - 1u);
    const float zdef = fill_neg_inf ? -INFINITY : bias_l;
    for (uint32_t todo = fast; todo; todo &= todo - 1) {
        const int i = __ffs(todo) - 1;
        Zs[(size_t)(ew * 32 + i) * RL_LANES + lane] = __shfl_sync(FULL, zdef, i);
    }
    if (partial && !fill_neg_inf && fast) {
        const bool mine = (fast >> lane) & 1u;
        run_m = warp_maxf(mine ? bias_l : -INFINITY);
        run_s = warp_sumf(mine ? expf(bias_l - run_m) : 0.f);
    }
    // The word's items are one contiguous, entity-grouped range: stream it SCORE_ROWS rows at a time (the
    // count rows and rule weights of a group are all in flight together, whatever entities they belong
    // to) and close a logit row whenever the entity changes.
    {
        int cur = -1;
        double acc = 0.0;
        bool any = false;
        const int B0 = __shfl_sync(FULL, wi.b0, 0), B1 = wi.wend;
        for (int c0 = B0; c0 < B1; c0 += 32) {
            if (c0 != wi.wbase) word_items_window(wi, c0);
            const int cnt = min(32, B1 - c0);
            for (int j0 = 0; j0 < cnt; j0 += SCORE_ROWS) {
                CT cv[SCORE_ROWS];
                float wv[SCORE_ROWS];
#pragma unroll
                for (int u = 0; u < SCORE_ROWS; ++u) {
                    const int src = (j0 + u) & 31;
                    const int a = __shfl_sync(FULL, wi.win.x, src);
                    const int t0 = __shfl_sync(FULL, wi.win.y, src);
                    const bool ok = j0 + u < cnt;
                    cv[u] = ok ? arena[(size_t)a * RL_LANES + lane] : (CT)0;
                    wv[u] = ok ? __ldg(w + __ldg(r.node_term_rule + t0)) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < SCORE_ROWS; ++u) {
                    if (j0 + u >= cnt) break;
                    const int src = (j0 + u) & 31;
                    const int i = __shfl_sync(FULL, wi.win.z, src) & 31;
                    const int nt = __shfl_sync(FULL, wi.win.w, src);
                    if (i != cur) {
                        if (cur >= 0) finish(cur, acc, any);
                        cur = i;
                        acc = 0.0;
                        any = false;
                    }
                    const double cf = (double)(float)cv[u];                               // x.float() * w (predictors.py:64)
                    acc += cf * (double)wv[u];
                    if (nt > 1) {                                                         // duplicate rules ending at the same node
                        const int t0 = __shfl_sync(FULL, wi.win.y, src);
                        for (int t = t0 + 1; t < t0 + nt; ++t) acc += cf * (double)__ldg(w + r.node_term_rule[t]);
                    }
                    any |= cv[u] != 0;
                }
            }
        }
        if (cur >= 0) finish(cur, acc, any);
    }
    for (uint32_t todo = slow & ~wi.present; todo; todo &= todo - 1) finish(__ffs(todo) - 1, 0.0, false);   // heads with empty-body rules only
    if (lane < e1) ms[ew * 32 + lane] = my_bits;
    }
    if (!partial) return;
    // one (max, sum-exp) pair per query and block, in k_softmax_partial's layout: one sweep over Z saved
    sm_m[warp][lane] = run_m;
    sm_s[warp][lane] = run_s;
    __syncthreads();
    if (warp == 0) {
        float M = -INFINITY;
        for (int k = 0; k < nwarps; ++k) M = fmaxf(M, sm_m[k][lane]);
        double S = 0.0;
        for (int k = 0; k < nwarps; ++k)
            if (sm_m[k][lane] != -INFINITY) S += sm_s[k][lane] * (double)expf(sm_m[k][lane] - M);
        float *p = partial + ((size_t)slot * gridDim.x + blockIdx.x) * 64;
        p[lane] = M;
        p[32 + lane] = (float)S;
    }
}

// ------------------------------------------------------------------------------------------
// kernel (2b): log(softmax + 1e-8) CE + backward (trainer.py:84,88-89)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_softmax_partial(int N, const float *__restrict__ Z, float *__restrict__ partial, int nblk)
{
    __shared__ float sm_m[WARPS_PER_BLOCK][32], sm_s[WARPS_PER_BLOCK][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.y;
    const float *Zs = Z + (size_t)slot * N * RL_LANES;
    const int e0 = blockIdx.x * SM_ROWS_PER_BLOCK;
    const int e1 = min(N, e0 + SM_ROWS_PER_BLOCK);
    // two passes over the warp's rows (the second one hits L1): max first, then one expf per logit with
    // four independent accumulators -- no serial max/sum dependency chain, half the MUFU work
    float m = -INFINITY;
    for (int e = e0 + warp; e < e1; e += WARPS_PER_BLOCK) m = fmaxf(m, Zs[(size_t)e * RL_LANES + lane]);
    float s4[4] = {0.f, 0.f, 0.f, 0.f};
    if (m != -INFINITY) {
        int e = e0 + warp;
        for (; e + 3 * WARPS_PER_BLOCK < e1; e += 4 * WARPS_PER_BLOCK) {
#pragma unroll
            for (int u = 0; u < 4; ++u) s4[u] += expf(Zs[(size_t)(e + u * WARPS_PER_BLOCK) * RL_LANES + lane] - m);
        }
        for (; e < e1; e += WARPS_PER_BLOCK) s4[0] += expf(Zs[(size_t)e * RL_LANES + lane] - m);
    }
    const float sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
    sm_m[warp][lane] = m;
    sm_s[warp][lane] = sum;
    __syncthreads();
    if (warp == 0) {
        float M = -INFINITY;
        for (int k = 0; k < WARPS_PER_BLOCK; ++k) M = fmaxf(M, sm_m[k][lane]);
        float S = 0.f;
        for (int k = 0; k < WARPS_PER_BLOCK; ++k)
            if (sm_m[k][lane] != -INFINITY) S += sm_s[k][lane] * expf(sm_m[k][lane] - M);
        float *p = partial + ((size_t)slot * nblk + blockIdx.x) * 64;
        p[lane] = M;
        p[32 + lane] = S;
    }
}

// one block per slot, one warp per query lane: combine the lane's partials, then walk its sparse targets
// stats[slot][lane][4] = (max, sumexp, S_b, valid)
__global__ void __launch_bounds__(CE_WARPS * 32)
k_ce_finalize(rl_graph g, rl_slots s, rl_answers ans, float smoothing, int use_mask,
              const float *__restrict__ Z, const uint32_t *__restrict__ nzmask,
              const float *__restrict__ partial, int nblk, float *__restrict__ stats,
              float *__restrict__ slot_lsum, float *__restrict__ slot_tsum)
{
    __shared__ double red_l[CE_WARPS], red_t[CE_WARPS];
    const int lane = threadIdx.x & 31, b = threadIdx.x >> 5;
    const int slot = blockIdx.x;
    const int N = g.num_entities;
    const int q = s.slot_head[slot];
    const float *pp = partial + (size_t)slot * nblk * 64;
    float M = -INFINITY;
    for (int k = lane; k < nblk; k += 32) M = fmaxf(M, pp[k * 64 + b]);
    M = warp_maxf(M);
    float S = 0.f;
    for (int k = lane; k < nblk; k += 32) {
        const float mk = pp[k * 64 + b];
        if (mk != -INFINITY) S += pp[k * 64 + 32 + b] * expf(mk - M);
    }
    S = warp_sumf(S);
    const float *Zs = Z + (size_t)slot * N * RL_LANES;
    const uint32_t *ms = nzmask + (size_t)slot * N;
    const int h = s.lane_h[slot * RL_LANES + b];
    const int t = s.lane_t[slot * RL_LANES + b];
    float lsum = 0.f, tacc = 0.f, sb = 0.f;
    bool saw_t = false;
    if (h >= 0 && M != -INFINITY) {
        const int ki = find_key(ans, (long long)q * N + h);
        const int a0 = ki >= 0 ? ans.ptr[ki] : 0, a1 = ki >= 0 ? ans.ptr[ki + 1] : 0;
        for (int a = a0 + lane; a < a1; a += 32) {
            const int e = ans.ent[a];
            float tg = smoothing;
            if (e == t) { tg += 1.f - smoothing; saw_t = true; }
            if (use_mask && !((ms[e] >> b) & 1u)) continue;
            const float p = expf(Zs[(size_t)e * RL_LANES + b] - M) / S;
            lsum += logf(p + 1e-8f) * tg;
            tacc += tg;
            sb += tg / (p + 1e-8f) * p;
        }
        saw_t = __any_sync(FULL, saw_t);
        if (!saw_t && t >= 0 && lane == 0 && !(use_mask && !((ms[t] >> b) & 1u))) {
            const float tg = 1.f - smoothing;
            const float p = expf(Zs[(size_t)t * RL_LANES + b] - M) / S;
            lsum += logf(p + 1e-8f) * tg;
            tacc += tg;
            sb += tg / (p + 1e-8f) * p;
        }
    }
    lsum = warp_sumf(lsum);
    tacc = warp_sumf(tacc);
    sb = warp_sumf(sb);
    if (lane == 0) {
        float *st = stats + ((size_t)slot * 32 + b) * 4;
        st[0] = M; st[1] = S; st[2] = sb; st[3] = (h >= 0 && M != -INFINITY) ? 1.f : 0.f;
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

// G[e][b] = softmax * S_b / T'   (dense part of dloss/dZ)
__global__ void __launch_bounds__(256)
k_grad_dense(int N, const float *__restrict__ Z, const float *__restrict__ stats,
             const float *__restrict__ slot_invT, float *__restrict__ G)
{
    const int slot = blockIdx.y;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)N * RL_LANES) return;
    const int b = (int)(i & 31);
    const float *st = stats + ((size_t)slot * 32 + b) * 4;
    float gval = 0.f;
    if (st[3] != 0.f) {                                      // st[3] = S_b / sum-exp / T'
        const float z = Z[(size_t)slot * N * RL_LANES + i];
        if (z != -INFINITY) gval = expf(z - st[0]) * st[3];
    }
    G[(size_t)slot * N * RL_LANES + i] = gval;
}

// sparse part: G[e][b] -= p * tgt / (p + eps) / T' at the target entries (one warp per query lane); with
// grad_bias != NULL the same terms also go into the bias gradient (the dense part comes from k_grad_dense_bias)
__global__ void __launch_bounds__(CE_WARPS * 32)
k_grad_sparse(rl_graph g, rl_slots s, rl_answers ans, float smoothing, int use_mask,
              const float *__restrict__ Z, const uint32_t *__restrict__ nzmask,
              const float *__restrict__ stats, const float *__restrict__ slot_invT, float *__restrict__ G,
              const float *__restrict__ slot_scale, float *__restrict__ grad_bias)
{
    const int lane = threadIdx.x & 31, b = threadIdx.x >> 5;
    const int slot = blockIdx.x;
    const int N = g.num_entities;
    const int q = s.slot_head[slot];
    const float *Zs = Z + (size_t)slot * N * RL_LANES;
    float *Gs = G + (size_t)slot * N * RL_LANES;
    const uint32_t *ms = nzmask + (size_t)slot * N;
    const float iT = slot_invT[slot];
    const float *st = stats + ((size_t)slot * 32 + b) * 4;
    if (st[3] == 0.f) return;
    const int h = s.lane_h[slot * RL_LANES + b];
    const int t = s.lane_t[slot * RL_LANES + b];
    const float M = st[0], S = st[1];
    const float scale = slot_scale ? slot_scale[slot] : 1.f;
    auto apply = [&](int e, float tg) {
        const float p = expf(Zs[(size_t)e * RL_LANES + b] - M) / S;
        const float term = p * (tg / (p + 1e-8f)) * iT;
        Gs[(size_t)e * RL_LANES + b] -= term;
        if (grad_bias) atomicAdd(grad_bias + e, -term * scale);
    };
    const int ki = find_key(ans, (long long)q * N + h);
    const int a0 = ki >= 0 ? ans.ptr[ki] : 0, a1 = ki >= 0 ? ans.ptr[ki + 1] : 0;
    bool saw_t = false;
    for (int a = a0 + lane; a < a1; a += 32) {
        const int e = ans.ent[a];
        float tg = smoothing;
        if (e == t) { tg += 1.f - smoothing; saw_t = true; }
        if (use_mask && !((ms[e] >> b) & 1u)) continue;
        apply(e, tg);
    }
    saw_t = __any_sync(FULL, saw_t);
    if (!saw_t && t >= 0 && lane == 0 && !(use_mask && !((ms[t] >> b) & 1u))) apply(t, 1.f - smoothing);
}

// ------------------------------------------------------------------------------------------
// kernel (2c): backward into rule weights / bias
// ------------------------------------------------------------------------------------------
// Backward over the entity-grouped item list (after rl_sort_items): one warp per 32 entities streams
// the word's items four at a time (count row + G row of each in flight together; items of one entity hit
// the same G row), fp32 products as the reference's x.float() * grad, one warp reduction per item.
template <typename CT>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_predictor_bwd_stream(rl_graph g, rl_rules r, rl_slots s, rl_frontier fr, const float *__restrict__ G,
                       const float *__restrict__ slot_scale, float *__restrict__ grad_w)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.y;
    const int ew = blockIdx.x * WARPS_PER_BLOCK + warp;
    const int N = g.num_entities, W = g.rank_words;
    const int q = s.slot_head[slot];
    const float scale = slot_scale ? slot_scale[slot] : 1.f;
    const float *Gs = G + (size_t)slot * N * RL_LANES;
    const int z0 = r.zr_ptr[q], z1 = r.zr_ptr[q + 1];
    if (blockIdx.x == 0 && warp == 0 && z1 > z0) {                 // empty-body rules: count = one_hot(h)
        const int h = s.lane_h[slot * RL_LANES + lane];
        double v = h >= 0 ? (double)Gs[(size_t)h * RL_LANES + lane] : 0.0;
        v = warp_sum(v);
        if (lane == 0)
            for (int t = z0; t < z1; ++t) atomicAdd(grad_w + r.zr_rule[t], (float)v * scale);
    }
    if (ew >= W) return;
    const CT *arena = reinterpret_cast<const CT *>(fr.arena) + (size_t)s.arena_off[slot] * RL_LANES;
    WordItems wi = load_word_items(fr, s, W, slot, ew);
    const int B0 = __shfl_sync(FULL, wi.b0, 0), B1 = wi.wend;
    for (int c0 = B0; c0 < B1; c0 += 32) {
        if (c0 != wi.wbase) word_items_window(wi, c0);
        const int cnt = min(32, B1 - c0);
        for (int j0 = 0; j0 < cnt; j0 += BWD_ROWS) {
            float pv[BWD_ROWS];
#pragma unroll
            for (int u = 0; u < BWD_ROWS; ++u) {
                const int src = (j0 + u) & 31;
                const int a = __shfl_sync(FULL, wi.win.x, src);
                const int e = __shfl_sync(FULL, wi.win.z, src);
                const bool ok = j0 + u < cnt;
                const CT c = ok ? arena[(size_t)a * RL_LANES + lane] : (CT)0;
                const float gq = ok ? Gs[(size_t)e * RL_LANES + lane] : 0.f;
                pv[u] = c != 0 ? (float)c * gq : 0.f;             // skips NaN*0 of masked cells
            }
#pragma unroll
            for (int u = 0; u < BWD_ROWS; ++u) {
                if (j0 + u >= cnt) break;
                const float v = warp_sumf(pv[u]);
                const int src = (j0 + u) & 31;
                const int t0 = __shfl_sync(FULL, wi.win.y, src), nt = __shfl_sync(FULL, wi.win.w, src);
                if (lane == 0 && v != 0.f)
                    for (int t = t0; t < t0 + nt; ++t) atomicAdd(grad_w + r.node_term_rule[t], v * scale);
            }
        }
    }
}

// k_grad_dense and the dense part of the bias gradient in one sweep over Z: a warp owns BIAS_ROWS consecutive
// entities (1 KB of contiguous logits per slot) and loops over slots, so the per-query (max, coefficient)
// pair is loaded once per slot and warp instead of once per row; G[sl][e][b] = coef_b * exp(z - max_b) is
// written and summed into grad_bias[e] on the way.
#define BIAS_SLOT_SPLIT 16
#define BIAS_ROWS 8
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_grad_dense_bias(int N, int S, const float *__restrict__ Z, const float *__restrict__ stats,
                  const float *__restrict__ slot_scale, float *__restrict__ G, float *__restrict__ grad_bias)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int e0 = (blockIdx.x * WARPS_PER_BLOCK + warp) * BIAS_ROWS;
    if (e0 >= N) return;
    const int ne = min(BIAS_ROWS, N - e0);
    double acc[BIAS_ROWS];
#pragma unroll
    for (int u = 0; u < BIAS_ROWS; ++u) acc[u] = 0.0;
    for (int sl = blockIdx.y; sl < S; sl += BIAS_SLOT_SPLIT) {
        const float4 st = __ldg(reinterpret_cast<const float4 *>(stats) + (size_t)sl * 32 + lane);
        const float sc = slot_scale ? slot_scale[sl] : 1.f;
        const size_t at = ((size_t)sl * N + e0) * RL_LANES + lane;
        float z[BIAS_ROWS];
#pragma unroll
        for (int u = 0; u < BIAS_ROWS; ++u) z[u] = u < ne ? Z[at + (size_t)u * RL_LANES] : -INFINITY;
#pragma unroll
        for (int u = 0; u < BIAS_ROWS; ++u) {
            const float gval = (st.w != 0.f && z[u] != -INFINITY) ? expf(z[u] - st.x) * st.w : 0.f;
            if (u < ne) G[at + (size_t)u * RL_LANES] = gval;
            acc[u] += (double)(gval * sc);
        }
    }
#pragma unroll
    for (int u = 0; u < BIAS_ROWS; ++u) {
        const double v = warp_sum(acc[u]);
        if (lane == 0 && u < ne) atomicAdd(grad_bias + e0 + u, (float)v);
    }
}

// ------------------------------------------------------------------------------------------
// kernel (3): filtered rank (trainer.py:189-201) + metrics (trainer.py:211-232)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_rank_count(int N, rl_slots s, const float *__restrict__ Z, int32_t *__restrict__ counters)
{
    __shared__ int sm_gt[WARPS_PER_BLOCK][32], sm_ge[WARPS_PER_BLOCK][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.y;
    const float *Zs = Z + (size_t)slot * N * RL_LANES;
    const int t = s.lane_t[slot * RL_LANES + lane];
    const float val = t >= 0 ? Zs[(size_t)t * RL_LANES + lane] : INFINITY;
    const int e0 = blockIdx.x * SM_ROWS_PER_BLOCK, e1 = min(N, e0 + SM_ROWS_PER_BLOCK);
    int gt = 0, ge = 0;
    for (int e = e0 + warp; e < e1; e += WARPS_PER_BLOCK) {
        const float z = Zs[(size_t)e * RL_LANES + lane];
        gt += z > val;
        ge += z >= val;
    }
    sm_gt[warp][lane] = gt;
    sm_ge[warp][lane] = ge;
    __syncthreads();
    if (warp == 0) {
        int a = 0, b = 0;
        for (int k = 0; k < WARPS_PER_BLOCK; ++k) { a += sm_gt[k][lane]; b += sm_ge[k][lane]; }
        atomicAdd(counters + ((size_t)slot * 32 + lane) * 2, a);
        atomicAdd(counters + ((size_t)slot * 32 + lane) * 2 + 1, b);
    }
}

__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
k_rank_finalize(rl_graph g, rl_slots s, rl_answers known, int use_mask, const float *__restrict__ Z,
                const uint32_t *__restrict__ nzmask, const int32_t *__restrict__ counters,
                int64_t *__restrict__ LH)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x;
    const int N = g.num_entities;
    const int q = s.slot_head[slot];
    const float *Zs = Z + (size_t)slot * N * RL_LANES;
    for (int b = warp; b < 32; b += WARPS_PER_BLOCK) {
        const int h = s.lane_h[slot * RL_LANES + b];
        const int t = s.lane_t[slot * RL_LANES + b];
        long long L = 0, H = 0;
        if (h >= 0 && t >= 0) {
            if (use_mask && !((nzmask[(size_t)slot * N + t] >> b) & 1u)) { L = 1; H = (long long)N + 1; }
            else {
                const float val = Zs[(size_t)t * RL_LANES + b];
                const int ki = find_key(known, (long long)q * N + h);
                const int a0 = ki >= 0 ? known.ptr[ki] : 0, a1 = ki >= 0 ? known.ptr[ki + 1] : 0;
                int gt = 0, ge = 0;
                for (int a = a0 + lane; a < a1; a += 32) {
                    const float z = Zs[(size_t)known.ent[a] * RL_LANES + b];
                    gt += z > val;
                    ge += z >= val;
                }
                gt = warp_sumi(gt);
                ge = warp_sumi(ge);
                L = (long long)(counters[((size_t)slot * 32 + b) * 2] - gt) + 1;
                H = (long long)(counters[((size_t)slot * 32 + b) * 2 + 1] - ge) + 2;
            }
        }
        if (lane == 0) {
            LH[((size_t)slot * 32 + b) * 2] = L;
            LH[((size_t)slot * 32 + b) * 2 + 1] = H;
        }
    }
}

__global__ void __launch_bounds__(256)
k_rank_dense(long long N, const float *__restrict__ logits, const uint8_t *__restrict__ flag,
             const uint8_t *__restrict__ mask, const int64_t *__restrict__ t, int64_t *__restrict__ LH)
{
    __shared__ int red[2][8];
    const long long k = blockIdx.x;
    const float *row = logits + k * N;
    const uint8_t *fl = flag + k * N;
    const long long tk = t[k];
    if (!mask[k * N + tk]) {
        if (threadIdx.x == 0) { LH[2 * k] = 1; LH[2 * k + 1] = N + 1; }
        return;
    }
    const float val = row[tk];
    int gt = 0, ge = 0;
    for (long long e = threadIdx.x; e < N; e += blockDim.x) {
        if (fl[e]) { gt += row[e] > val; ge += row[e] >= val; }
    }
    gt = warp_sumi(gt);
    ge = warp_sumi(ge);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = gt; red[1][threadIdx.x >> 5] = ge; }
    __syncthreads();
    if (threadIdx.x == 0) {
        int a = 0, b = 0;
        for (int i = 0; i < 8; ++i) { a += red[0][i]; b += red[1][i]; }
        LH[2 * k] = a + 1;
        LH[2 * k + 1] = b + 2;
    }
}

__global__ void __launch_bounds__(256)
k_rank_metrics(long long Q, const int64_t *__restrict__ LH, const double *__restrict__ weight, int expectation,
               const double *__restrict__ harmonic, double *__restrict__ sums)
{
    __shared__ double red[5][8];
    double v[5] = {0, 0, 0, 0, 0};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < Q; i += (long long)gridDim.x * blockDim.x) {
        const double wgt = weight ? weight[i] : 1.0;
        const long long L = LH[2 * i], H = LH[2 * i + 1];
        if (wgt == 0.0 || H <= L) continue;
        if (expectation) {
            const double n = (double)(H - L);
            const long long hi = H - 1;
            v[0] += wgt * (double)max(0ll, min(hi, 1ll) - L + 1) / n;
            v[1] += wgt * (double)max(0ll, min(hi, 3ll) - L + 1) / n;
            v[2] += wgt * (double)max(0ll, min(hi, 10ll) - L + 1) / n;
            v[3] += wgt * 0.5 * (double)(L + hi);
            v[4] += wgt * (harmonic[hi] - harmonic[L - 1]) / n;
        } else {
            const long long rank = H - 1;
            v[0] += wgt * (rank <= 1);
            v[1] += wgt * (rank <= 3);
            v[2] += wgt * (rank <= 10);
            v[3] += wgt * (double)rank;
            v[4] += wgt / (double)rank;
        }
    }
    for (int m = 0; m < 5; ++m) {
        const double x = warp_sum(v[m]);
        if ((threadIdx.x & 31) == 0) red[m][threadIdx.x >> 5] = x;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        double x = 0;
        for (int i = 0; i < 8; ++i) x += red[threadIdx.x][i];
        atomicAdd(sums + threadIdx.x, x);
    }
}

// Adam (torch.optim.Adam semantics: L2 weight decay folded into the gradient, bias-corrected moments,
// eps added after the square root).  torch's fused multi-tensor Adam puts 65 k elements in one block,
// which makes the 146 k-parameter Predictor step take ~90 us; one element per thread takes ~3 us.
__global__ void __launch_bounds__(256)
k_adam(long long n, float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m, float *__restrict__ v,
       float lr, float b1, float b2, float eps, float wd, float bc1, float bc2_sqrt)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float grad = g[i];
    const float w = p[i];
    if (wd != 0.f) grad = fmaf(wd, w, grad);
    const float mi = fmaf(b1, m[i], (1.f - b1) * grad);            // m = b1*m + (1-b1)*g   (lerp, as torch)
    const float vi = fmaf(b2, v[i], (1.f - b2) * grad * grad);
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = w - (lr / bc1) * (mi / denom);
}

// entity-major slot -> reference layout
__global__ void k_slot_to_dense(int N, int nq, const float *__restrict__ Zs, float *__restrict__ out, long long stride)
{
    __shared__ float tile[32][33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int e = blockIdx.x * 32 + w;
    tile[w][lane] = e < N ? Zs[(size_t)e * RL_LANES + lane] : 0.f;
    __syncthreads();
    const int eo = blockIdx.x * 32 + lane;
    if (eo < N && w < nq) out[(size_t)w * stride + eo] = tile[lane][w];
}

__global__ void k_mask_to_dense(int N, int nq, const uint32_t *__restrict__ ms, uint8_t *__restrict__ out, long long stride)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    const uint32_t bits = ms[e];
    for (int b = 0; b < nq; ++b) out[(size_t)b * stride + e] = (bits >> b) & 1u;
}

// ------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------
extern "C" {

int rl_abi_version(void) { return RL_ABI_VERSION; }
const char *rl_last_error(void) { return g_err; }
long long rl_launch_count(void) { return g_launches; }

int rl_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(RL_ERR_NO_DEVICE, "no CUDA device visible (rnnlogic_b200 has no CPU fallback)");
    }
    return n;
}

int rl_prepare_slots(const rl_graph *g, int32_t S, const int32_t *slot_head, const int32_t *q_off,
                     const int64_t *all_h, const int64_t *all_t, const int64_t *etr, int32_t remove_query_edges,
                     int32_t *lane_h, int32_t *lane_t, int32_t *lane_eh, int32_t *lane_et, void *stream)
{
    if (!g || !slot_head || !q_off || !all_h || !lane_h || !lane_t || !lane_eh || !lane_et || S <= 0)
        return fail(RL_ERR_ARG, "rl_prepare_slots: bad argument");
    const int n = S * RL_LANES;
    if (remove_query_edges && !all_t) return fail(RL_ERR_ARG, "rl_prepare_slots: remove_query_edges needs all_t");
    k_prepare_slots<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(*g, S, slot_head, q_off, all_h, all_t, etr,
                                                                        remove_query_edges, lane_h, lane_t, lane_eh, lane_et);
    CHECK_LAUNCH("k_prepare_slots");
    return RL_OK;
}

static int check_frontier(const rl_frontier *fr, const char *who)
{
    if (!fr || !fr->arena || !fr->row_mask || !fr->node_cnt || !fr->overflow) return fail(RL_ERR_ARG, who);
    if (fr->count_bits != 32 && fr->count_bits != 64) return fail(RL_ERR_ARG, "count_bits must be 32 or 64");
    return RL_OK;
}

int rl_pair_table(const rl_graph *g, int32_t n_pairs, const int32_t *pair_prel, const int32_t *pair_rel,
                  const int64_t *pair_base, const int32_t *ptr, int32_t *out, void *stream)
{
    if (!g || !pair_prel || !pair_rel || !pair_base || !out) return fail(RL_ERR_ARG, "rl_pair_table: null argument");
    if (n_pairs <= 0) return RL_OK;
    if (ptr) k_pair_table<true><<<n_pairs, 128, 0, (cudaStream_t)stream>>>(*g, pair_prel, pair_rel, pair_base, ptr, out);
    else k_pair_table<false><<<n_pairs, 128, 0, (cudaStream_t)stream>>>(*g, pair_prel, pair_rel, pair_base, ptr, out);
    CHECK_LAUNCH("k_pair_table");
    return RL_OK;
}

int rl_expand_level(const rl_graph *g, const rl_rules *r, const rl_slots *s, int32_t depth, int32_t grid_nodes,
                    int32_t grid_chunks, const rl_frontier *fr, int32_t dense_num, int32_t dense_den,
                    int32_t force_dense, int32_t chunks_per_warp, void *stream)
{
    if (!g || !r || !s) return fail(RL_ERR_ARG, "rl_expand_level: null argument");
    if (check_frontier(fr, "rl_expand_level: incomplete rl_frontier") != RL_OK) return RL_ERR_ARG;
    if (depth < 1 || depth > r->max_len) return fail(RL_ERR_ARG, "rl_expand_level: depth out of range");
    if (dense_den <= 0 || dense_num < 0) return fail(RL_ERR_ARG, "rl_expand_level: bad dense threshold");
    if (grid_chunks <= 0 || grid_nodes <= 0 || s->num_slots <= 0) return RL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 gs((grid_nodes + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, s->num_slots);   // grid_nodes = symbolic work items
    if (depth == 1) k_symbolic<true><<<gs, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, depth, *fr, dense_num, dense_den, force_dense);
    else k_symbolic<false><<<gs, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, depth, *fr, dense_num, dense_den, force_dense);
    CHECK_LAUNCH("k_symbolic");
    // chunks per warp: many when most chunks are empty (one coalesced read of their bitmap words),
    // few when every chunk is expanded (more warps in flight to hide the look-up latency)
    static const int cpw_env = []() { const char *e = getenv("RL_CPW"); const int v = e ? atoi(e) : 0; return (v >= 1 && v <= 32) ? v : 0; }();
    const int cpw = cpw_env ? cpw_env : (chunks_per_warp >= 1 && chunks_per_warp <= 32 ? chunks_per_warp : (force_dense ? 4 : 16));
    dim3 grid((grid_chunks + NUM_WARPS * cpw - 1) / (NUM_WARPS * cpw), s->num_slots);
    // force_dense: plain dense SpMM -- every row of every node is written (zeros included) and read
#define LAUNCH_NUM(CT, ROOT, PRUNE) k_numeric<CT, ROOT, PRUNE><<<grid, NUM_WARPS * 32, 0, st>>>(*g, *r, *s, depth, *fr, cpw)
    if (fr->count_bits == 32) {
        if (depth == 1) { if (force_dense) LAUNCH_NUM(uint32_t, true, false); else LAUNCH_NUM(uint32_t, true, true); }
        else { if (force_dense) LAUNCH_NUM(uint32_t, false, false); else LAUNCH_NUM(uint32_t, false, true); }
    } else {
        if (depth == 1) { if (force_dense) LAUNCH_NUM(unsigned long long, true, false); else LAUNCH_NUM(unsigned long long, true, true); }
        else { if (force_dense) LAUNCH_NUM(unsigned long long, false, false); else LAUNCH_NUM(unsigned long long, false, true); }
    }
#undef LAUNCH_NUM
    CHECK_LAUNCH("k_numeric");
    return RL_OK;
}

int rl_node_counts_dense(const rl_graph *g, const rl_rules *r, const rl_slots *s, int32_t slot, int32_t node,
                         const rl_frontier *fr, int64_t *out, void *stream)
{
    if (!g || !r || !s || !out) return fail(RL_ERR_ARG, "rl_node_counts_dense: null argument");
    if (check_frontier(fr, "rl_node_counts_dense: incomplete rl_frontier") != RL_OK) return RL_ERR_ARG;
    if (slot < 0 || slot >= s->num_slots || node >= r->num_nodes) return fail(RL_ERR_ARG, "rl_node_counts_dense: index out of range");
    const int grid = (g->num_entities + 31) / 32;
    if (fr->count_bits == 32) k_node_dense<uint32_t><<<grid, 1024, 0, (cudaStream_t)stream>>>(*g, *r, *s, slot, node, *fr, out);
    else k_node_dense<unsigned long long><<<grid, 1024, 0, (cudaStream_t)stream>>>(*g, *r, *s, slot, node, *fr, out);
    CHECK_LAUNCH("k_node_dense");
    return RL_OK;
}

int rl_propagate_dense(const rl_graph *g, int32_t relation, int32_t B, const int64_t *x, const int64_t *etr,
                       int64_t *out, void *stream)
{
    if (!g || !x || !out) return fail(RL_ERR_ARG, "rl_propagate_dense: null argument");
    if (relation < 0 || relation >= g->num_relations) return fail(RL_ERR_ARG, "rl_propagate_dense: relation out of range");
    if (B <= 0 || g->num_entities <= 0) return RL_OK;
    k_propagate_dense<<<(g->num_entities + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, WARPS_PER_BLOCK * 32, 0, (cudaStream_t)stream>>>(
        *g, relation, B, x, etr, out);
    CHECK_LAUNCH("k_propagate_dense");
    return RL_OK;
}

static int check_items(const rl_frontier *fr, const char *who)
{
    if (!fr->items || !fr->items_sorted || !fr->item_off || !fr->item_cnt || !fr->bucket_cnt || !fr->bucket_off) return fail(RL_ERR_ARG, who);
    return RL_OK;
}

int rl_sort_items(const rl_graph *g, const rl_slots *s, const rl_frontier *fr, void *stream)
{
    if (!g || !s) return fail(RL_ERR_ARG, "rl_sort_items: null argument");
    if (check_frontier(fr, "rl_sort_items: incomplete rl_frontier") != RL_OK) return RL_ERR_ARG;
    if (check_items(fr, "rl_sort_items: the frontier was expanded without an item list") != RL_OK) return RL_ERR_ARG;
    if (s->num_slots <= 0) return RL_OK;
    return launch_items_sort(g, s, fr, (cudaStream_t)stream);
}

// warps per k_predictor_scores block (tail-bound kernel: hub words make long warps; swept on the B200)
static int score_warps()
{
    static int v = 0;
    if (!v) {
        const char *e = getenv("RL_SCORE_WARPS");
        v = e ? atoi(e) : 4;                                   // 4 beat 8 by 2 % (shorter block tails)
        if (v < 1 || v > SCORE_WARPS_MAX) v = 4;
    }
    return v;
}

int rl_predictor_scores(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                        const float *w, const float *bias, int32_t fill_neg_inf, float *Z, uint32_t *nzmask,
                        float *partial, void *stream)
{
    if (!g || !r || !s || !w || !Z || !nzmask) return fail(RL_ERR_ARG, "rl_predictor_scores: null argument");
    if (check_frontier(fr, "rl_predictor_scores: incomplete rl_frontier") != RL_OK) return RL_ERR_ARG;
    if (check_items(fr, "rl_predictor_scores: the frontier was expanded without an item list") != RL_OK) return RL_ERR_ARG;
    if (s->num_slots <= 0) return RL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (launch_items_sort(g, s, fr, st) != RL_OK) return RL_ERR_CUDA;
    const int sw = score_warps();
    dim3 grid((g->rank_words + sw - 1) / sw, s->num_slots);           // one block = one softmax partial
    if (fr->count_bits == 32) k_predictor_scores<uint32_t><<<grid, sw * 32, 0, st>>>(*g, *r, *s, *fr, w, bias, fill_neg_inf, Z, nzmask, partial);
    else k_predictor_scores<unsigned long long><<<grid, sw * 32, 0, st>>>(*g, *r, *s, *fr, w, bias, fill_neg_inf, Z, nzmask, partial);
    CHECK_LAUNCH("k_predictor_scores");
    return RL_OK;
}

static int sweep_blocks(int N) { return (N + SM_ROWS_PER_BLOCK - 1) / SM_ROWS_PER_BLOCK; }
static int score_blocks(int N) { const int W = (N + 31) / 32, sw = score_warps(); return (W + sw - 1) / sw; }
// scratch sizing: partials come either from k_softmax_partial or from k_predictor_scores
int rl_softmax_blocks(int32_t N) { return sweep_blocks(N) > score_blocks(N) ? sweep_blocks(N) : score_blocks(N); }

// loss half shared by rl_softmax_ce and rl_predictor_ce_backward
static int ce_forward(const rl_graph *g, const rl_slots *s, const rl_answers *ans, float smoothing, int32_t use_mask,
                      const float *Z, const uint32_t *nzmask, int32_t n_groups, const int32_t *group_ptr, float *partial,
                      int partial_ready, float *stats, float *slot_sums, float *group_loss, float *group_tsum, cudaStream_t st)
{
    const int S = s->num_slots, N = g->num_entities;
    const int nblk = partial_ready ? score_blocks(N) : sweep_blocks(N);
    float *slot_lsum = slot_sums, *slot_tsum = slot_sums + S, *slot_invT = slot_sums + 2 * (size_t)S;
    if (!partial_ready) {
        k_softmax_partial<<<dim3(nblk, S), WARPS_PER_BLOCK * 32, 0, st>>>(N, Z, partial, nblk);
        CHECK_LAUNCH("k_softmax_partial");
    }
    k_ce_finalize<<<S, CE_WARPS * 32, 0, st>>>(*g, *s, *ans, smoothing, use_mask, Z, nzmask, partial, nblk, stats, slot_lsum, slot_tsum);
    CHECK_LAUNCH("k_ce_finalize");
    k_group_reduce<<<n_groups, 32, 0, st>>>(n_groups, group_ptr, slot_lsum, slot_tsum, group_loss, group_tsum, slot_invT, stats);
    CHECK_LAUNCH("k_group_reduce");
    return RL_OK;
}

int rl_softmax_ce(const rl_graph *g, const rl_slots *s, const rl_answers *ans, float smoothing, int32_t use_mask,
                  const float *Z, const uint32_t *nzmask, int32_t n_groups, const int32_t *group_ptr,
                  float *partial, float *stats, float *slot_sums, float *group_loss, float *group_tsum,
                  float *G, void *stream)
{
    if (!g || !s || !ans || !Z || !nzmask || !partial || !stats || !slot_sums || !group_loss || !group_tsum)
        return fail(RL_ERR_ARG, "rl_softmax_ce: null argument");
    const int S = s->num_slots, N = g->num_entities;
    if (S <= 0) return RL_OK;
    if (n_groups <= 0 || n_groups > S || (!group_ptr && n_groups != S)) return fail(RL_ERR_ARG, "rl_softmax_ce: bad group table");
    cudaStream_t st = (cudaStream_t)stream;
    float *slot_invT = slot_sums + 2 * (size_t)S;
    const int rc = ce_forward(g, s, ans, smoothing, use_mask, Z, nzmask, n_groups, group_ptr, partial, 0, stats, slot_sums,
                              group_loss, group_tsum, st);
    if (rc != RL_OK) return rc;
    if (G) {
        const size_t n = (size_t)N * RL_LANES;
        k_grad_dense<<<dim3((unsigned)((n + 255) / 256), S), 256, 0, st>>>(N, Z, stats, slot_invT, G);
        CHECK_LAUNCH("k_grad_dense");
        k_grad_sparse<<<S, CE_WARPS * 32, 0, st>>>(*g, *s, *ans, smoothing, use_mask, Z, nzmask, stats, slot_invT, G, nullptr, nullptr);
        CHECK_LAUNCH("k_grad_sparse");
    }
    return RL_OK;
}

int rl_predictor_ce_backward(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                             const rl_answers *ans, float smoothing, int32_t use_mask, const float *Z,
                             const uint32_t *nzmask, int32_t n_groups, const int32_t *group_ptr, float *partial,
                             int32_t partial_ready, float *stats, float *slot_sums, float *group_loss, float *group_tsum,
                             float *G, const float *slot_scale, float *grad_w, float *grad_bias, void *stream)
{
    if (!g || !r || !s || !ans || !Z || !nzmask || !partial || !stats || !slot_sums || !group_loss || !group_tsum || !G || !grad_w)
        return fail(RL_ERR_ARG, "rl_predictor_ce_backward: null argument");
    if (check_frontier(fr, "rl_predictor_ce_backward: incomplete rl_frontier") != RL_OK) return RL_ERR_ARG;
    if (check_items(fr, "rl_predictor_ce_backward: the frontier was expanded without an item list") != RL_OK) return RL_ERR_ARG;
    const int S = s->num_slots, N = g->num_entities;
    if (S <= 0) return RL_OK;
    if (n_groups <= 0 || n_groups > S || (!group_ptr && n_groups != S)) return fail(RL_ERR_ARG, "rl_predictor_ce_backward: bad group table");
    cudaStream_t st = (cudaStream_t)stream;
    float *slot_invT = slot_sums + 2 * (size_t)S;
    int rc = ce_forward(g, s, ans, smoothing, use_mask, Z, nzmask, n_groups, group_ptr, partial, partial_ready, stats,
                        slot_sums, group_loss, group_tsum, st);
    if (rc != RL_OK) return rc;
    if (grad_bias) {
        const int rows_per_block = WARPS_PER_BLOCK * BIAS_ROWS;
        k_grad_dense_bias<<<dim3((N + rows_per_block - 1) / rows_per_block, BIAS_SLOT_SPLIT), WARPS_PER_BLOCK * 32, 0, st>>>(
            N, S, Z, stats, slot_scale, G, grad_bias);
        CHECK_LAUNCH("k_grad_dense_bias");
    } else {
        const size_t n = (size_t)N * RL_LANES;
        k_grad_dense<<<dim3((unsigned)((n + 255) / 256), S), 256, 0, st>>>(N, Z, stats, slot_invT, G);
        CHECK_LAUNCH("k_grad_dense");
    }
    k_grad_sparse<<<S, CE_WARPS * 32, 0, st>>>(*g, *s, *ans, smoothing, use_mask, Z, nzmask, stats, slot_invT, G, slot_scale, grad_bias);
    CHECK_LAUNCH("k_grad_sparse");
    const dim3 grid((g->rank_words + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, S);
    if (fr->count_bits == 32) k_predictor_bwd_stream<uint32_t><<<grid, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, *fr, G, slot_scale, grad_w);
    else k_predictor_bwd_stream<unsigned long long><<<grid, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *r, *s, *fr, G, slot_scale, grad_w);
    CHECK_LAUNCH("k_predictor_bwd_stream");
    return RL_OK;
}

int rl_filtered_rank(const rl_graph *g, const rl_slots *s, const rl_answers *known, int32_t use_mask,
                     const float *Z, const uint32_t *nzmask, int32_t *counters, int64_t *LH, void *stream)
{
    if (!g || !s || !known || !Z || !nzmask || !counters || !LH) return fail(RL_ERR_ARG, "rl_filtered_rank: null argument");
    const int S = s->num_slots, N = g->num_entities;
    if (S <= 0) return RL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(counters, 0, (size_t)S * 64 * sizeof(int32_t), st);
    if (e != cudaSuccess) return fail(RL_ERR_CUDA, "rl_filtered_rank: memset", e);
    k_rank_count<<<dim3(sweep_blocks(N), S), WARPS_PER_BLOCK * 32, 0, st>>>(N, *s, Z, counters);
    CHECK_LAUNCH("k_rank_count");
    k_rank_finalize<<<S, WARPS_PER_BLOCK * 32, 0, st>>>(*g, *s, *known, use_mask, Z, nzmask, counters, LH);
    CHECK_LAUNCH("k_rank_finalize");
    return RL_OK;
}

int rl_filtered_rank_dense(int64_t Q, int64_t N, const float *logits, const uint8_t *flag, const uint8_t *mask,
                           const int64_t *t, int64_t *LH, void *stream)
{
    if (!logits || !flag || !mask || !t || !LH) return fail(RL_ERR_ARG, "rl_filtered_rank_dense: null argument");
    if (Q <= 0) return RL_OK;
    k_rank_dense<<<(unsigned)Q, 256, 0, (cudaStream_t)stream>>>(N, logits, flag, mask, t, LH);
    CHECK_LAUNCH("k_rank_dense");
    return RL_OK;
}

int rl_rank_metrics(int64_t Q, const int64_t *LH, const double *weight, int32_t expectation,
                    const double *harmonic, double *sums, void *stream)
{
    if (!LH || !sums || (expectation && !harmonic)) return fail(RL_ERR_ARG, "rl_rank_metrics: null argument");
    if (Q <= 0) return RL_OK;
    int grid = (int)((Q + 255) / 256);
    if (grid > 592) grid = 592;
    k_rank_metrics<<<grid, 256, 0, (cudaStream_t)stream>>>(Q, LH, weight, expectation, harmonic, sums);
    CHECK_LAUNCH("k_rank_metrics");
    return RL_OK;
}

int rl_adam_step(int64_t n, float *param, const float *grad, float *exp_avg, float *exp_avg_sq, float lr, float beta1,
                 float beta2, float eps, float weight_decay, int64_t step, void *stream)
{
    if (!param || !grad || !exp_avg || !exp_avg_sq || step < 1) return fail(RL_ERR_ARG, "rl_adam_step: bad argument");
    if (n <= 0) return RL_OK;
    const double bc1 = 1.0 - pow((double)beta1, (double)step);
    const double bc2 = 1.0 - pow((double)beta2, (double)step);
    k_adam<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, param, grad, exp_avg, exp_avg_sq, lr, beta1, beta2, eps,
                                                                        weight_decay, (float)bc1, (float)sqrt(bc2));
    CHECK_LAUNCH("k_adam");
    return RL_OK;
}

int rl_slot_to_dense(int32_t N, int32_t nq, const float *Zs, float *out, int64_t stride, void *stream)
{
    if (!Zs || !out || nq < 0 || nq > RL_LANES) return fail(RL_ERR_ARG, "rl_slot_to_dense: bad argument");
    k_slot_to_dense<<<(N + 31) / 32, 1024, 0, (cudaStream_t)stream>>>(N, nq, Zs, out, stride);
    CHECK_LAUNCH("k_slot_to_dense");
    return RL_OK;
}

int rl_mask_to_dense(int32_t N, int32_t nq, const uint32_t *ms, uint8_t *out, int64_t stride, void *stream)
{
    if (!ms || !out || nq < 0 || nq > RL_LANES) return fail(RL_ERR_ARG, "rl_mask_to_dense: bad argument");
    k_mask_to_dense<<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(N, nq, ms, out, stride);
    CHECK_LAUNCH("k_mask_to_dense");
    return RL_OK;
}

}  // extern "C"
