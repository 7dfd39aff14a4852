/*
 * rnnlogic_b200 -- C-ABI of the B200-native (sm_100a) reasoning-predictor hot path.
 *
 * Drop-in boundary.  The reference (DeepGraphLearning/RNNLogic) has no FFI: its boundary for
 * this path is Python (src/data.py, src/predictors.py, src/trainer.py).  Each entry point
 * below names the reference interface it replaces (file:line relative to /root/reference);
 * the Python classes of the same names in rnnlogic_b200/ (re-exported by compat/) bind these
 * symbols with ctypes (rnnlogic_b200/_lib.py).  INTEGRATION.md shows the binding a reference
 * maintainer would add.
 *
 * Conventions
 *  - plain C: pointers + sizes only, no torch types.  All `const T*` inside the structs are
 *    DEVICE pointers (cudaMalloc / torch caching allocator); the structs themselves are host
 *    memory and are passed by pointer.  `stream` is a cudaStream_t cast to void*.
 *  - every function returns 0 on success, a negative rl_status otherwise; the message of the
 *    last failure on the calling thread is rl_last_error().  Nothing here synchronises the
 *    device or allocates device memory; kernels are enqueued on `stream`.
 *  - queries are processed in SLOTS of RL_LANES = 32 queries that share one head relation
 *    (the reference's single-relation batch, predictors.py:55,212).  All per-slot matrices
 *    are ENTITY-MAJOR: X[row][lane], one 128-byte line per row for 32-bit counts.
 */
#ifndef RNNLOGIC_B200_H
#define RNNLOGIC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RL_LANES 32
#define RL_ABI_VERSION 5

enum rl_status {
    RL_OK = 0,
    RL_ERR_ARG = -1,      /* bad argument (null pointer, size, level out of range) */
    RL_ERR_CUDA = -2,     /* a CUDA runtime call / launch failed */
    RL_ERR_NO_DEVICE = -3 /* no CUDA device visible: there is NO CPU fallback */
};

/* Knowledge graph, replaces KnowledgeGraph.relation2adjacency / relation2ht2index
 * (src/data.py:39-40,63-69,101-104).  Relation-sorted DCSR *by destination*: for relation rho
 * the distinct tails are rows [dst_ptr[rho], dst_ptr[rho+1]); row k has tail row_dst[k] and
 * in-edges edge_src[row_start[k] .. row_start[k+1]).  rank_tab answers "which row of relation
 * rho is entity e" with one 8-byte load: word w = e>>5 holds {bits, rows before this word}.
 * ord_* keep the reference's per-relation edge order (train.txt order) so that an
 * `edges_to_remove` index (data.py:164-170) maps to its (head, tail).  fsrc_ptr/frow_start/
 * fedge_dstrow/srank_tab are the same edges sorted by (relation, head, tail). */
typedef struct rl_graph {
    int32_t num_entities, num_relations, rank_words, total_rows, num_edges;
    const int32_t *dst_ptr;    /* [R+1]            */
    const int32_t *row_dst;    /* [total_rows]     */
    const int32_t *row_start;  /* [total_rows+1]   */
    const int32_t *edge_src;   /* [E]              */
    const uint32_t *rank_tab;  /* [R*rank_words*2] */
    const int32_t *ord_ptr;    /* [R+1]            */
    const int32_t *ord_h;      /* [E] head of the k-th train edge of the relation */
    const int32_t *ord_t;      /* [E] tail ...                                    */
    /* forward DCSR (by source), used to find which destination rows a frontier can reach */
    const int32_t *fsrc_ptr;     /* [R+1] distinct heads per relation */
    const int32_t *frow_start;   /* [total_srcs+1] out-edge offsets */
    const int32_t *fedge_dstrow; /* [E] destination row (local to the relation) of each out-edge */
    const uint32_t *srank_tab;   /* [R*rank_words*2] rank table over heads */
} rl_graph;

/* Compiled rule set, replaces Predictor.relation2rules (src/predictors.py:46-49, 186-189).
 * Per head relation the rule bodies form a prefix trie (one node per distinct non-empty body
 * prefix); nodes of one head are contiguous and ordered by depth.  A node's frontier is a
 * [rows(node_rel) x 32] block at row offset node_row_off inside the slot's arena.  Work is cut
 * into chunks of <= 32 consecutive rows of one node; lvl_ptr[q*(max_len+1)+d] .. [..+d+1] is
 * the chunk range of depth d+1 of head q.  node_term_* lists the rules ending at each node; zr_* the
 * rules with an empty body. */
typedef struct rl_rules {
    int32_t num_nodes, num_rules, max_len, num_chunks, num_terms, num_zero_rules;
    const int32_t *node_rel;      /* [num_nodes] */
    const int64_t *node_row_off;  /* [num_nodes] */
    const int32_t *head_node_ptr; /* [R+1] */
    const int32_t *lvl_ptr;       /* [R*(max_len+1)] */
    const int32_t *chunk_node;    /* [num_chunks] */
    const int32_t *chunk_row0;    /* [num_chunks] first row, local to the node */
    const int32_t *zr_ptr;        /* [R+1] */
    const int32_t *zr_rule;       /* [#empty-body rules] */
    const int32_t *node_chunk0;   /* [num_nodes] global id of the node's first chunk */
    /* packed per-node record, 32-byte aligned: {rel, parent, parent rel, dst_ptr[rel],
     *  rows(rel), chunk0, parent chunk0, nterm} -- one load instead of a look-up chain */
    const int32_t *node_rec;      /* [num_nodes*8] */
    const int64_t *node_prow_off; /* [num_nodes] node_row_off of the parent (0 for depth 1) */
    /* symbolic-phase work items: (node, first parent bitmap word); one item per 32 parent words
     * (one item per node at depth 1); lvl_sym_ptr is indexed like lvl_ptr */
    const int32_t *lvl_sym_ptr;   /* [R*(max_len+1)] */
    const int32_t *sym_node;      /* [#items] */
    const int32_t *sym_w0;        /* [#items] */
    /* rules ending at a node: node_term_rule[node_term_ptr[v] .. node_term_ptr[v+1]) */
    const int32_t *node_term_ptr;  /* [num_nodes+1] */
    const int32_t *node_term_rule; /* [num_terms] */
    /* pair tables (rl_pair_table): for a node v of depth > 1 and its destination row d, the parent rows that have an
     * edge into d are pair_ent[pair_ptr[node_pair_off[v] + d] .. pair_ptr[node_pair_off[v] + d + 1]) */
    const int64_t *node_pair_off;  /* [num_nodes] first pair_ptr entry of the node's (parent relation, relation) pair */
    const int32_t *pair_ptr;       /* [sum over pairs of rows(rel) + 1] */
    const int32_t *pair_ent;       /* parent row indices */
} rl_rules;

/* One call's queries, cut into slots (<= 32 queries of one head relation each). */
typedef struct rl_slots {
    int32_t num_slots;
    const int32_t *slot_head;  /* [S] head relation */
    const int32_t *lane_h;     /* [S*32] query entity, -1 = padding lane */
    const int32_t *lane_t;     /* [S*32] answer entity (train / eval), -1 = none */
    const int32_t *lane_eh;    /* [S*32] head of the removed edge, -1 = no removal */
    const int32_t *lane_et;    /* [S*32] tail of the removed edge */
    const int64_t *arena_off;  /* [S] first arena row of the slot */
    const int32_t *nz_off;     /* [S] first node_cnt entry of the slot */
    const int64_t *mask_off;   /* [S] first row_mask word of the slot (one word per chunk) */
} rl_slots;

/* Per-call frontier state (all DEVICE memory owned by the caller; row_mask, node_cnt
 * and overflow must be zero before depth 1).  A row of a node is meaningful iff its row_mask bit
 * is set; rows outside the bitmap are never written nor read (exact: they are all-zero). */
typedef struct rl_frontier {
    int32_t count_bits;    /* 32: uint32 counts + overflow flag, 64: wraps like the reference's int64 */
    void *arena;           /* [rows][32] counts */
    uint32_t *row_mask;    /* one word per 32-row chunk */
    int32_t *node_cnt;     /* valid rows per (slot, node) */
    int32_t *overflow;     /* int32[9], zeroed by the caller: [0] set to 1 when a 32-bit count overflowed; [1 + d] non-zero
                            * rows produced at depth d (d < 8) over all slots -- feedback for the next call's chunks_per_warp */
    /* Item list (may be all NULL when only rl_expand_level / rl_node_counts_dense are used): one
     * int32x4 record {row (slot-relative), t0, entity, n} per NON-ZERO row of every rule-end node
     * (the rules ending at that node are node_term_rule[t0 .. t0+n)),
     * appended by k_numeric; slot s owns [item_off[s], item_off[s+1]) (capacity = rows of its head's
     * rule-end nodes, so it cannot overflow).  item_cnt[S] and bucket_cnt[S*B] (per-entity item counts,
     * B = rank_words*32 + 32 ints per slot, 16-byte aligned) zeroed by the caller; items_sorted /
     * bucket_off[S*B] are filled by rl_sort_items: the items of entity e of a slot are
     * items_sorted[item_off + bucket_off[e] .. bucket_off[e+1]). */
    int32_t *items;        /* as int32x4, 16-byte aligned */
    int32_t *items_sorted;
    const int64_t *item_off;
    int32_t *item_cnt;
    int32_t *bucket_cnt;
    int32_t *bucket_off;
    /* Lane mask of every item (bit b: the count of query b in that row is non-zero), written by k_numeric
     * next to the item and carried through the sort.  The OR of an entity's item masks is its candidate
     * word nzmask[slot][entity] (predictors.py:224-225,239: a cell is a candidate iff its total count is
     * non-zero).  nzmask ([S][N], zeroed by the caller) is accumulated by k_numeric itself when the frontier has
     * no sort buffers (bucket_cnt == NULL: the cell kernels walk the items in the order they were appended),
     * else by rl_sort_items. */
    uint32_t *item_mask;
    uint32_t *item_mask_sorted;
    uint32_t *nzmask;
} rl_frontier;

/* Known-answer lists, replaces KnowledgeGraph.hr2o / hr2oo / hr2ooo (src/data.py:36-38,49-61,
 * 79-99): sorted keys r*N+h, CSR of de-duplicated tails.  Used for the smoothed multi-hot
 * target (data.py:207-212) and the eval filter (data.py:250-254, 287-291). */
typedef struct rl_answers {
    int64_t num_keys;
    const int64_t *keys;  /* [num_keys] ascending */
    const int32_t *ptr;   /* [num_keys+1] */
    const int32_t *ent;   /* [ptr[num_keys]] */
} rl_answers;

/* Candidate cells of a call (rl_cells.cu).  A cell is a (query, entity) pair with a non-zero total path
 * count (src/predictors.py:224-225,239: mask != 0 -> candidate_set).  Cells are numbered slot by slot,
 * entity-major, lane-minor; the cells of entity e of slot s are cand_off[s*N+e] .. + popc(nzmask[s*N+e]).
 * All DEVICE memory owned by the caller; counters must be zero before rl_cells_build.  When the call has
 * more cells than `cap`, counters[1] is set, cells beyond cap are skipped by every kernel, and the caller
 * redoes the call with larger per-cell arrays. */
typedef struct rl_cells {
    int32_t cap;          /* capacity of the per-cell arrays */
    int32_t *counters;    /* [8]: [0] number of cells, [1] != 0: cap exceeded */
    uint32_t *nzmask;     /* [S][N] candidate word per entity (= rl_frontier.nzmask) */
    int32_t *cand_off;    /* [S][N] first cell of the entity */
    int32_t *cell_key;    /* [cap] slot*32 + lane of the cell */
    int32_t *cell_ent;    /* [cap] entity of the cell */
    int32_t *slot_ncell;  /* [S] cells per slot (= mask.sum() of the batch without an entity feature, trainer.py:96) */
    uint32_t *qmax;       /* [S*32] scratch: per-query max of the cell logits (order-preserving key) */
    float *qsum;          /* [S*32] scratch: per-query sum of the softmax corrections */
} rl_cells;

int rl_abi_version(void);
const char *rl_last_error(void);
/* Kernels enqueued by this library since it was loaded (per process). */
long long rl_launch_count(void);
/* Number of visible CUDA devices (>= 1) or RL_ERR_NO_DEVICE. */
int rl_device_count(void);

/* Fill lane_h / lane_t / lane_eh / lane_et from the reference's batch tensors
 * (all_h, all_t, edges_to_remove int64[Q] on the device; trainer.py:69-82).  Query i of slot s
 * is q_off[s] + lane (q_off is a DEVICE int32[S+1]).  all_t / edges_to_remove may be NULL.
 * remove_query_edges != 0 with edges_to_remove == NULL: the removed edge of a query is its own
 * triple (h, head, t) when that is a train edge -- what TrainDataset builds by looking the
 * triple's index up (src/data.py:214-216) -- found on the device, no host look-up. */
int rl_prepare_slots(const rl_graph *g, int32_t num_slots, const int32_t *slot_head,
                     const int32_t *q_off, const int64_t *all_h, const int64_t *all_t,
                     const int64_t *edges_to_remove, int32_t remove_query_edges, int32_t *lane_h,
                     int32_t *lane_t, int32_t *lane_eh, int32_t *lane_et, void *stream);

/* Pair tables of a rule set (rl_rules.pair_ptr / pair_ent): pair p = (pair_prel[p], pair_rel[p]) owns the entries
 * [pair_base[p], pair_base[p] + rows(pair_rel[p]) + 1) of the pointer array.  Call once with ptr == NULL: out = per-row
 * entry counts (int32, same indexing, a zero closes each pair); the caller turns them into exclusive prefix sums; call
 * again with ptr = the sums: out = pair_ent. */
int rl_pair_table(const rl_graph *g, int32_t n_pairs, const int32_t *pair_prel, const int32_t *pair_rel,
                  const int64_t *pair_base, const int32_t *ptr, int32_t *out, void *stream);

/* Kernel (1): frontier expansion of one trie depth for every slot, replaces
 * KnowledgeGraph.propagate (src/data.py:149-173) for all rules of the head at once.  Two
 * launches: k_symbolic (which destination rows can be non-zero -> row_mask) and k_numeric (the
 * segmented pull SpMM over those rows, query edge removed on hops of the head relation).
 * grid_nodes / grid_chunks = max over the call's slots of the number of symbolic work items
 * (lvl_sym_ptr) / chunks at this depth.  A node whose parent has more than dense_num/dense_den of its rows valid takes all
 * its rows; force_dense != 0 does that for every node (plain dense SpMM: every algorithmic byte
 * of SURVEY.md 8d is moved -- the mode the roofline figure is quoted on).  chunks_per_warp: consecutive 32-row chunks one k_numeric warp owns (1..32; 0 = default 16, 4 in dense mode): many when
 * most chunks are empty (one coalesced read of their bitmap words), few when the frontier is dense (finer, balanced work). */
int rl_expand_level(const rl_graph *g, const rl_rules *r, const rl_slots *s, int32_t depth,
                    int32_t grid_nodes, int32_t grid_chunks, const rl_frontier *fr,
                    int32_t dense_num, int32_t dense_den, int32_t force_dense, int32_t chunks_per_warp, void *stream);

/* Bucket the frontier's item list by entity word (counting sort, idempotent).  Called by
 * rl_predictor_scores and rl_plus_mask themselves; exported for callers that drive the kernels. */
int rl_sort_items(const rl_graph *g, const rl_slots *s, const rl_frontier *fr, void *stream);

/* Debug / API parity: dense int64[32][N] (lane-major, like the reference's [B,N]) counts of
 * one trie node of one slot; node < 0 selects the one-hot root (empty body).  Replaces the
 * return value of KnowledgeGraph.grounding (src/data.py:147). */
int rl_node_counts_dense(const rl_graph *g, const rl_rules *r, const rl_slots *s, int32_t slot,
                         int32_t node, const rl_frontier *fr, int64_t *out, void *stream);

/* One hop from an arbitrary dense frontier: KnowledgeGraph.propagate (src/data.py:149-173).  x / out are
 * the reference's int64 [N][B] (its [N,B,1] tensor); etr (may be NULL) holds one index per query into the
 * relation's train-order edge list whose message is dropped for that query (data.py:164-170).  int64
 * arithmetic, wraps like the reference. */
int rl_propagate_dense(const rl_graph *g, int32_t relation, int32_t B, const int64_t *x, const int64_t *etr,
                       int64_t *out, void *stream);

/* Kernel (2a): rule-weight aggregation, replaces the loop of Predictor.forward
 * (src/predictors.py:58-65,73-78).  Z[S][N][32] fp32 = sum_rule w_rule * fp32(count) (+ bias[e]
 * when bias != NULL).  nzmask[S][N]: bit b set <=> sum_rule count[e][b] != 0.  With
 * fill_neg_inf != 0 cells with a clear bit get -inf (entity_feature != 'bias').
 * softmax_partial (may be NULL): S * rl_softmax_blocks(N) * 64 floats; when given, the kernel also
 * leaves the per-block (max, sum-exp) of every query there, which rl_predictor_ce_backward accepts
 * (partial_ready != 0) instead of sweeping Z once more. */
int rl_predictor_scores(const rl_graph *g, const rl_rules *r, const rl_slots *s,
                        const rl_frontier *fr, const float *rule_weights, const float *bias,
                        int32_t fill_neg_inf, float *Z, uint32_t *nzmask, float *softmax_partial,
                        void *stream);

/* Kernel (2b): log(softmax + 1e-8) cross-entropy against the smoothed target, replaces
 * src/trainer.py:84,88-89, fused with its backward.  target = smoothing * multi_hot(train
 * answers of (h, head)) + (1 - smoothing) * one_hot(t).  A GROUP is one reference batch: slots
 * [group_ptr[i], group_ptr[i+1]) (DEVICE int32[n_groups+1]; NULL <=> every slot is its own
 * group).  Outputs: group_loss[n_groups] = -sum lp*target / max(sum target, 1), group_tsum
 * [n_groups] = sum target, and (when G != NULL) G[S][N][32] = d group_loss / dZ.
 * use_mask != 0 <=> entity_feature != 'bias' (only cells with their nzmask bit take part).
 * Scratch: partial = S * rl_softmax_blocks(N) * 64 floats, stats = S*32*4 floats
 * (max, sum-exp, S_b, valid per lane), slot_sums = 3*S floats. */
int rl_softmax_blocks(int32_t num_entities);
int rl_softmax_ce(const rl_graph *g, const rl_slots *s, const rl_answers *train_answers,
                  float smoothing, int32_t use_mask, const float *Z, const uint32_t *nzmask,
                  int32_t n_groups, const int32_t *group_ptr, float *partial, float *stats,
                  float *slot_sums, float *group_loss, float *group_tsum, float *G, void *stream);

/* Kernel (2b) fused with the backward into rule weights and bias for Predictor's dense train step (src/trainer.py:84,88-90 + autograd
 * through src/predictors.py:64,74): same loss outputs and scratch as rl_softmax_ce, then the
 * backward with the passes fused (softmax gradient + bias gradient in one sweep over Z, target
 * terms pushed into G and grad_bias together, item walk over the entity-grouped list).
 * partial_ready != 0: `partial` was filled by rl_predictor_scores.  G[S][N][32] is scratch.
 * grad_w[num_rules], grad_bias[N] (may be NULL) are ACCUMULATED into:
 * += sum_groups slot_scale * d group_loss / d param. */
int rl_predictor_ce_backward(const rl_graph *g, const rl_rules *r, const rl_slots *s,
                             const rl_frontier *fr, const rl_answers *train_answers, float smoothing,
                             int32_t use_mask, const float *Z, const uint32_t *nzmask, int32_t n_groups,
                             const int32_t *group_ptr, float *partial, int32_t partial_ready,
                             float *stats, float *slot_sums, float *group_loss, float *group_tsum,
                             float *G, const float *slot_scale, float *grad_w, float *grad_bias,
                             void *stream);

/* Kernel (3): filtered rank bounds, replaces src/trainer.py:189-201.  LH[S*32][2] int64:
 * L = #{e not known: z_e > z_t} + 1, H = #{e not known: z_e >= z_t} + 2; (1, N+1) when the
 * answer's nzmask bit is clear and use_mask != 0.  `known` = hr2oo (valid) / hr2ooo (test).
 * counters is scratch int32[S*64], zeroed by the call. */
int rl_filtered_rank(const rl_graph *g, const rl_slots *s, const rl_answers *known,
                     int32_t use_mask, const float *Z, const uint32_t *nzmask,
                     int32_t *counters, int64_t *LH, void *stream);

/* Same bounds from the reference's dense tensors (logits fp32[Q][N], flag u8[Q][N],
 * mask u8[Q][N], t int64[Q]) -- what TrainerPredictor.evaluate holds (trainer.py:182-187). */
int rl_filtered_rank_dense(int64_t Q, int64_t N, const float *logits, const uint8_t *flag,
                           const uint8_t *mask, const int64_t *t, int64_t *LH, void *stream);

/* Hits@1/3/10, MR, MRR partial sums over rows (L,H) with weight[] (0 drops a duplicate),
 * replaces src/trainer.py:211-232.  harmonic is fp64[N+2] with harmonic[k] = sum_{i<=k} 1/i.
 * sums[5] fp64 are ACCUMULATED (zero them first). */
int rl_rank_metrics(int64_t Q, const int64_t *LH, const double *weight, int32_t expectation,
                    const double *harmonic, double *sums, void *stream);

/* ---- PredictorPlus (src/predictors.py:210-271, src/layers.py:63-126) ------------------------
 * A candidate is a (query, entity) cell whose total path count is non-zero (predictors.py:239);
 * candidates are numbered slot-major, entity-major, lane-minor:
 *   index(slot, e, b) = cand_off[slot*N + e] + popcount(nzmask[slot*N + e] & ((1 << b) - 1)),
 * cand_off = exclusive prefix sum of cand_cnt (done by the caller). */

/* nzmask[S][N] (bit b <=> sum_rule count[e][b] != 0, empty-body rules included) and
 * cand_cnt[S*N] = popcount(nzmask).  Replaces mask / candidate_set of predictors.py:220-239. */
int rl_plus_mask(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                 uint32_t *nzmask, int32_t *cand_cnt, void *stream);

/* Rule-embedding aggregation per candidate, replaces the [C,R_q,H] broadcast of
 * FuncToNodeSum / FuncToNode (layers.py:68-72, 94-99): out_sum[C][H] = sum_rule fp32(count)*emb;
 * with pna != 0 also out_sq (count*emb^2), out_min/out_max over rules with count != 0, their
 * arg rules (rows of emb), degree[C] = sum count + 1.  emb is [n][H] fp32, rule_local[rule id] its
 * row.  cand_query[C] = index of the candidate's query in the call (b_n of predictors.py:240). */
int rl_plus_features(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                     const uint32_t *nzmask, const int64_t *cand_off, const int32_t *q_off,
                     const int32_t *rule_local, const float *emb, int32_t H, int32_t pna,
                     float *out_sum, float *out_sq, float *out_min, float *out_max, int32_t *arg_min,
                     int32_t *arg_max, float *degree, int64_t *cand_query, void *stream);

/* Z[S][N][32] = (candidate ? zc[index] : 0 | -inf) + bias[e] + extra[S][N][32]; replaces
 * predictors.py:257-269.  bias / extra may be NULL. */
int rl_plus_scatter(const rl_graph *g, const rl_slots *s, const uint32_t *nzmask, const int64_t *cand_off,
                    const float *zc, const float *bias, const float *extra, int32_t fill_neg_inf,
                    float *Z, void *stream);
/* dz[index] = G[slot][e][b] at the candidate cells (backward of the scatter). */
int rl_plus_gather(const rl_graph *g, const rl_slots *s, const uint32_t *nzmask, const int64_t *cand_off,
                   const float *G, float *dz, void *stream);

/* Backward of rl_plus_features into the rule embeddings: gA[row][h] += sum_cells fp32(count) *
 * dA[cell][h] (and gB from dB, the squared-sum branch of PNA; dB/gB may be NULL).  ACCUMULATES. */
int rl_plus_backward(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                     const uint32_t *nzmask, const int64_t *cand_off, const int32_t *rule_local, int32_t H,
                     const float *dA, const float *dB, int32_t max_terms, float *gA, float *gB, void *stream);

/* E-step statistics, replaces the per-rule dense tensors of Predictor.compute_H
 * (src/predictors.py:93-112): for slot s, the i-th rule end of the slot's head (i = term index -
 * term_ptr[head*R]) and lane b: sum_cnt[s][i][b] = sum_e count, pos_cnt[s][i][b] = count at lane_t.
 * Both fp64 [S][max_terms][32], zeroed by the caller. */
int rl_rule_stats(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                  int32_t max_terms, double *sum_cnt, double *pos_cnt, void *stream);

/* LSTM rule encoder of PredictorPlus (src/predictors.py:141,201-208: torch.nn.LSTM(H, H, L, batch_first=True)
 * over the embedded [head, body..., pad] tokens, output of the last non-pad position).  x[n][T][H] embedded
 * tokens, len[n] (>= 1) non-pad tokens per rule, weights = HOST array of 4*L device pointers
 * (weight_ih, weight_hh, bias_ih, bias_hh per layer; torch layout [4H][H], gate order i, f, g, o).
 * H in {16, 32}, L <= RL_RNN_MAX_LAYERS.  Forward: out[n][H]; acts[n][L][T][5][H] (i, f, g, o, c) and
 * ih[L][n][T][2H] ([input of layer l at step t | its hidden state of step t-1]) are kept for the backward --
 * zero-filled by the caller, steps behind len stay zero.
 * Backward: dG[L][n][T][4H] (pre-activation gate gradients) and dX[n][T][H], zero-filled by the caller; the
 * weight gradients are the reductions [dW_ih[l] | dW_hh[l]] = dG[l]^T ih[l], db[l] = sum dG[l], left to the
 * caller's (batched) GEMM. */
#define RL_RNN_MAX_LAYERS 4
int rl_lstm_encode_forward(int32_t n, int32_t T, int32_t H, int32_t L, const float *x, const int32_t *len,
                           const float *const *weights, float *acts, float *ih, float *out, void *stream);
int rl_lstm_encode_backward(int32_t n, int32_t T, int32_t H, int32_t L, const int32_t *len,
                            const float *const *weights, const float *acts, const float *dout, float *dG,
                            float *dX, void *stream);
/* The weight-gradient reductions of the encoder: dW[L][4H][2H] += dG[l]^T ih[l] over the M = n*T rows,
 * db[L][4H] += column sums of dG[l] (both zero-filled by the caller; K ~ 1e5 with 64 x 32 outputs is no shape
 * for a library GEMM). */
int rl_lstm_encode_wgrad(int64_t M, int32_t H, int32_t L, const float *dG, const float *ih, float *dW,
                         float *db, void *stream);

/* ---- RotatE entity feature (src/embedding.py:28-70) -----------------------------------------
 * out[S][N][32] = gamma - sum_d |h_b o rot(remb[head]) - e|_d for every entity e; eemb fp32[N][2D]
 * (re | im), remb fp32[R][D] (already doubled with the negated copy, embedding.py:23-26).
 * P is scratch [S][2D][32] (the projected heads, kept for the backward). */
int rl_rotate_scores(const rl_graph *g, const rl_slots *s, int32_t D, float gamma, const float *eemb,
                     const float *remb, float *P, float *out, void *stream);
/* Backward of rl_rotate_scores for G[S][N][32] = d loss / d out: ACCUMULATES into d_eemb[N][2D] and
 * d_remb[R][D]; dP is zeroed scratch [S][2D][32]. */
int rl_rotate_backward(const rl_graph *g, const rl_slots *s, int32_t D, float gamma, const float *eemb,
                       const float *remb, const float *P, const float *G, float *dP, float *d_eemb,
                       float *d_remb, void *stream);

/* One Adam step with torch.optim.Adam's arithmetic (run_predictorplus.py:51; weight_decay is L2, i.e.
 * added to the gradient); step is the 1-based step count.  Optional: the trainer keeps working with any
 * torch optimizer, this is what rnnlogic_b200.optim.Adam launches. */
int rl_adam_step(int64_t n, float *param, const float *grad, float *exp_avg, float *exp_avg_sq, float lr,
                 float beta1, float beta2, float eps, float weight_decay, int64_t step, void *stream);

/* Entity-major <-> reference layout: out[b][e] = Z[slot][e][b] for b < nq (fp32 [nq][N]). */
int rl_slot_to_dense(int32_t N, int32_t nq, const float *Z_slot, float *out, int64_t out_stride,
                     void *stream);
int rl_mask_to_dense(int32_t N, int32_t nq, const uint32_t *nzmask_slot, uint8_t *out,
                     int64_t out_stride, void *stream);

/* ---- the scoring half on candidate cells (rl_cells.cu, rl_tail_tc.cu): no [S][N][32] matrix ---- */

/* Number the cells: cand_off, cell_key, cell_ent, slot_ncell, counters[0..1] from the candidate words nzmask that
 * k_numeric left (the frontier must be expanded without sort buffers, bucket_cnt == NULL; RL_ERR_ARG otherwise);
 * the cells of empty-body rules are added to nzmask here.  counters[0] counts every cell, also those beyond cap.
 * Replaces torch.nonzero(mask) (src/predictors.py:239) without a host sync. */
int rl_cells_build(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                   const rl_cells *c, void *stream);

/* acc[0] = max_e bias[e], acc[1] = sum_e exp(bias[e] - acc[0]) (doubles, DEVICE); acc[2] is scratch of
 * rl_cells_softmax_ce.  Once per parameter update. */
int rl_bias_stats(int32_t N, const float *bias, double *acc, void *stream);

/* Predictor (src/predictors.py:58-65): zc[cell] = sum_rule w_rule * fp32(count), without the bias.  One THREAD per
 * item (non-zero row of a rule-end node) in the order k_numeric appended them: it reads the counts of the queries in
 * the item's lane mask and adds w * fp32(count) to their cells (zc[cap] is cleared first); no sort, no per-warp walk
 * of ragged lists. */
int rl_predictor_item_scores(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                            const rl_cells *c, const float *w, float *zc, void *stream);

/* log(softmax + 1e-8) cross-entropy against the smoothed multi-hot target (src/trainer.py:84,88-89) with the
 * logits given as cell scores zc plus bias[e] for EVERY entity (bias != NULL; predictors.py:257-262), or as
 * the cell scores alone with -inf elsewhere (bias == NULL; predictors.py:267-269).  Same outputs as
 * rl_softmax_ce (group_loss, group_tsum; stats [S][32][4] and slot_sums [3*S] are scratch).  Gc != NULL:
 * Gc[cell] = grad_scale * dloss/dlogit and, with a bias, grad_bias[N] += grad_scale * dloss/dbias
 * (rank-one term + cell and target corrections). */
int rl_cells_softmax_ce(const rl_graph *g, const rl_slots *s, const rl_cells *c, const rl_answers *ans,
                        float smoothing, const float *bias, double *acc, const float *zc, int32_t n_groups,
                        const int32_t *group_ptr, float grad_scale, float *stats, float *slot_sums,
                        float *group_loss, float *group_tsum, float *Gc, float *grad_bias, void *stream);

/* Predictor backward: grad_w[rule] += sum over the rule's non-zero counts of Gc[cell] * fp32(count) (one atomic per
 * item and rule). */
int rl_predictor_item_backward(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                              const rl_cells *c, const float *Gc, float *grad_w, void *stream);

/* Filtered rank (src/trainer.py:189-201) from cell scores: (L,H) int64[S*32][2].  With a bias the entities
 * outside a query's cells are counted by binary search in sorted_bias (bias sorted ascending);
 * counters int32[S*64] is scratch. */
int rl_cells_rank(const rl_graph *g, const rl_slots *s, const rl_cells *c, const rl_answers *known,
                  const float *bias, const float *sorted_bias, const float *zc, int32_t *counters, int64_t *LH,
                  void *stream);

/* Z[S][N][32] += zc at the cells / Gc = G at the cells (dense entity features such as RotatE; the [B,N] scores of
 * the reference's forward()). */
int rl_cells_add_to_dense(const rl_graph *g, const rl_slots *s, const rl_cells *c, const float *zc, float *Z, void *stream);
int rl_cells_gather_dense(const rl_graph *g, const rl_slots *s, const rl_cells *c, const float *G, float *Gc, void *stream);

/* PredictorPlus sum aggregate per cell (src/layers.py:68-72), hidden_dim 16, emb[num_rules][16] indexed by the global
 * rule id: F[cell][16] = sum fp32(count) * emb[rule], one thread per (item, quarter of the hidden vector), 16-byte
 * vector atomics (F[cap][16] is cleared first).  The PNA statistics come from rl_pna_item_stats. */
int rl_plus_item_features(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                         const rl_cells *c, const float *emb, int32_t H, float *F, void *stream);

/* grad_emb[rule][16] += sum over the rule's non-zero counts of fp32(count) * dF[cell][16]. */
int rl_plus_item_backward(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr,
                         const rl_cells *c, int32_t H, const float *dF, float *grad_emb, void *stream);

/* Dense tail of PredictorPlus on the cells (src/layers.py:73-75, src/predictors.py:253-255), H = 16, J = 128:
 * zc[cell] = W2 . relu(W1 [relu(LN(W0 F + b0)), rel[head]] + b1) + b2  (rl_tail_tc.cu).  The Linear(2H,128) of the
 * score MLP and both of its backward products run on the tensor cores (tcgen05.mma, fp32 accumulators in TMEM) with
 * split operands (3xTF32 forward; exact bf16 x 3 against the 0/1 ReLU-bit matrix backward), so the logits keep the
 * 1e-5 bar.  The forward leaves relu_bits[cell][4] (which hidden units are active); the backward uses them instead of
 * recomputing the hidden layer, ACCUMULATES every weight gradient in-kernel (layouts of the parameters), writes
 * dF[cell][16] and needs rl_tail_scratch_floats(R) floats of scratch. */
int64_t rl_tail_scratch_floats(int32_t R);
/* front_done != 0: F already holds the aggregator's Linear output y (the PNA front, rl_pna_front_forward); then W0 is
 * not used, the backward writes dY[cell][16] instead of dF (and no gW0); gb0 still receives sum dy (the Linear's bias). */
int rl_tail_forward(const rl_cells *c, const int32_t *slot_head, int32_t H, int32_t J, const float *F, const float *W0,
                    const float *b0, const float *gamma, const float *beta, const float *W1, const float *b1,
                    const float *W2, const float *b2, const float *rel_emb, float *zc, uint32_t *relu_bits,
                    int32_t front_done, void *stream);
int rl_tail_backward(const rl_cells *c, const int32_t *slot_head, int32_t R, int32_t H, int32_t J, const float *F,
                     const float *W0, const float *b0, const float *gamma, const float *beta, const float *W1,
                     const float *b1, const float *W2, const float *b2, const float *rel_emb, const float *Gc,
                     const uint32_t *relu_bits, float *dF, float *dY, float *gW0, float *gb0,
                     float *ggamma, float *gbeta, float *gW1, float *gb1, float *gW2, float *gb2, float *grel,
                     float *scratch, int32_t front_done, void *stream);

/* ---- rule discovery (rl_miner.cu; miner/rnnlogic.cpp:350-382, 505-589) ----
 * Every relation path of <= max_len hops from h to its FIRST visit of t, for every triple (h, r, t) of
 * tri[n_triples][3] with that triple removed from the graph, without the trivial rule r <- r; h == t yields the empty
 * body.  adj_ptr[N+1] / adj_rel / adj_dst = out-edges by source entity over all relations (DEVICE).  table[cap] (cap a
 * power of two, filled with 0xFF bytes by the caller) receives the DISTINCT rules as 64-bit keys
 *     head << (b*max_len+3) | length << (b*max_len) | body[i] << (b*(max_len-1-i)),   b = rel_bits,
 * whose ascending order is the order of the reference's rule list (head relation, then std::set<Rule> order:
 * length, body; rnnlogic.cpp:118-133, 575-585).  flags[0] != 0 on return:
 * the table was too small.  rel_bits * (max_len + 1) + 3 must be <= 63, max_len <= 6. */
int rl_mine_rules(int32_t n_triples, const int32_t *tri, const int32_t *adj_ptr, const int32_t *adj_rel, const int32_t *adj_dst,
                  int32_t max_len, int32_t rel_bits, unsigned long long *table, int64_t cap, int32_t *flags, void *stream);

/* ---- PNA aggregator (FuncToNode, src/layers.py:89-126) on the cells, hidden_dim 16 (rl_pna.cu) ---- */
typedef struct rl_pna {                 /* per-cell statistics, arrays of rl_cells.cap cells (DEVICE) */
    float *s1;                          /* [cap][16] sum count * emb      (layers.py:94) */
    float *s2;                          /* [cap][16] sum count * emb^2    (layers.py:95) */
    float *deg;                         /* [cap]     sum count (the reference's degree is this + 1, layers.py:92) */
    unsigned long long *mnk;            /* [cap][16] min over rules with count != 0: order key of emb << 32 | rule */
    unsigned long long *mxk;            /* [cap][16] max ...:                        order key of emb << 32 | ~rule */
} rl_pna;
/* statistics from the item list (arrays are initialised here) */
int rl_pna_item_stats(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr, const rl_cells *c,
                      const float *emb, const rl_pna *p, void *stream);
/* Y[cell][16] = Linear(12H,H)([mean, min, max, std] (x) [1, s, 1/s]) (layers.py:100-124; W [16][192], b [16]);
 * FEAT[cap][64] and SC[cap] are kept for the backward; qscr = 2*S*32 floats of scratch. */
int rl_pna_front_forward(const rl_slots *s, const rl_cells *c, const rl_pna *p, const float *W, const float *b, float *qscr,
                         float *Y, float *FEAT, float *SC, void *stream);
/* dY[cell][16] -> dstat[cell][64] = [dS1 | dS2 | dMin | dMax]; gW[16][192] += dY^T update */
int rl_pna_front_backward(const rl_cells *c, const rl_pna *p, const float *W, const float *dY, const float *FEAT,
                          const float *SC, float *dstat, float *gW, void *stream);
/* grad_emb[rule][16] += count * dS1 + 2 count emb dS2 (+ dMin / dMax at the arg rules: first rule in file order on ties) */
int rl_pna_item_backward(const rl_graph *g, const rl_rules *r, const rl_slots *s, const rl_frontier *fr, const rl_cells *c,
                         const float *emb, const rl_pna *p, const float *dstat, float *grad_emb, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* RNNLOGIC_B200_H */
