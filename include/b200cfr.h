/* b200cfr.h — C ABI of the B200-native vectorized CFR engine.
 *
 * Drop-in boundary for the solver hot path of kmurf1999/RustSolver.  The reference has no
 * FFI of its own (mccfr/cfr are private methods, src/solver/cfr.rs:299,481); these entry
 * points are what a `cc`/bindgen block in src/solver would bind to replace
 *   MCCFRTrainer::init   (src/solver/cfr.rs:159-184)  -> rs_create
 *   MCCFRTrainer::train  (src/solver/cfr.rs:188-297)  -> rs_iterate (+ rs_discount)
 *   Infoset::get_strategy / get_final_strategy (src/solver/infoset.rs:83-123)
 *                                                     -> rs_read_infoset / rs_average_strategy
 *   MCCFRTrainer::calc_br (src/solver/cfr.rs:629-638) -> rs_best_response
 *   ICardAbstraction::get_cluster / get_size (src/solver/card_abstraction.rs:71-72)
 *                                                     -> rs_card_table / rs_num_rows
 * See INTEGRATION.md for the Rust-side stub.
 *
 * Conventions: every call returns 0 on success, <0 on error (message via rs_last_error());
 * nothing panics or aborts across the ABI.  The caller owns every input array; the engine
 * copies during rs_create and never retains host pointers.  Outputs go to caller buffers
 * with explicit capacities.  One host thread per handle (thread-compatible).  There is no
 * CPU fallback: rs_create fails if no sm_100-class CUDA device is usable.
 */
#ifndef B200CFR_H
#define B200CFR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* error codes */
#define RS_OK 0
#define RS_ERR_INVALID -1    /* bad argument / malformed tree (reference: panic!) */
#define RS_ERR_CUDA -2       /* CUDA runtime error or no device */
#define RS_ERR_NCCL -3       /* NCCL error */
#define RS_ERR_CAPACITY -4   /* output buffer too small */
#define RS_ERR_UNSUPPORTED -5

/* node types (src/solver/nodes.rs:47-52) */
#define RS_NODE_ACTION 0
#define RS_NODE_TERMINAL 1
#define RS_NODE_PUBLIC_CHANCE 2
#define RS_NODE_PRIVATE_CHANCE 3
/* terminal types (src/solver/nodes.rs:17-21) */
#define RS_TERM_ALLIN 0
#define RS_TERM_SHOWDOWN 1
#define RS_TERM_UNCONTESTED 2
/* betting rounds (src/solver/state.rs:7-22) */
#define RS_ROUND_FLOP 0
#define RS_ROUND_TURN 1
#define RS_ROUND_RIVER 2

/* Tree<GameTreeNode> (src/solver/tree.rs:12-24) flattened: node id = arena index. */
typedef struct rs_tree {
    uint32_t n_nodes;
    const uint8_t* type;          /* [n_nodes] RS_NODE_* */
    const int32_t* parent;        /* [n_nodes] -1 for the root */
    const uint32_t* child_offset; /* [n_nodes+1] CSR into children, action order */
    const uint32_t* children;     /* [child_offset[n_nodes]] */
    const uint8_t* player;        /* ActionNode.player      (nodes.rs:8) */
    const uint32_t* an_index;     /* ActionNode.index       (nodes.rs:7) */
    const uint8_t* round_idx;     /* ActionNode.round_idx   (nodes.rs:9) */
    const uint32_t* value;        /* TerminalNode.value     (nodes.rs:35) */
    const uint8_t* ttype;         /* TerminalNode.ttype     (nodes.rs:36) */
    const uint8_t* last_to_act;   /* TerminalNode.last_to_act (nodes.rs:37) */
} rs_tree;

/* hand_ranges after remove_invalid_combos (src/solver/cfr.rs:161-163): (c0,c1) pairs,
 * card = 4*rank + suit.  Unweighted like the reference (HoleCards has no weight). */
typedef struct rs_ranges {
    uint32_t n_hands[2];
    const uint8_t* hands[2]; /* [n_hands[p]][2] */
} rs_ranges;

/* card abstraction per round_idx (src/solver/card_abstraction.rs:62-66) */
#define RS_ABS_NONE 0        /* one row per live hand (lossless, no suit merging) */
#define RS_ABS_ISOMORPHIC 1  /* ISOMORPHIC: canonical suit-isomorphic index (card_abstraction.rs:186-214) */
#define RS_ABS_CLUSTER_ARR 2 /* EMD / OCHS: cluster_arr[canonical index] (card_abstraction.rs:216-298) */
#define RS_ABS_BUCKET_TABLE 3 /* caller-supplied bucket key per (board, hand) */
typedef struct rs_round_abstraction {
    uint32_t kind;
    const uint32_t* cluster_arr; /* RS_ABS_CLUSTER_ARR: contents of round_N_{emd,ochs}.dat (LE u32) */
    uint64_t cluster_arr_len;
    const uint32_t* bucket_table[2]; /* RS_ABS_BUCKET_TABLE: [n_boards(round)][n_hands[p]] keys */
} rs_round_abstraction;
typedef struct rs_abstraction {
    uint32_t n_rounds; /* = number of betting rounds in the tree (card_abs.len(), cfr.rs:167-172) */
    rs_round_abstraction rounds[3];
} rs_abstraction;

#define RS_NCCL_ID_BYTES 128
typedef struct rs_config {
    uint64_t board_mask;       /* Options.board_mask (options.rs:17) */
    int32_t device;            /* CUDA device ordinal */
    /* board sharding over one process per GPU (SURVEY §8e): rank r owns a contiguous slice of
     * the first dealt-card level; world_size 1 = single GPU */
    int32_t rank;
    int32_t world_size;
    uint8_t nccl_id[RS_NCCL_ID_BYTES]; /* from rs_nccl_unique_id on rank 0, broadcast by the host */
    /* shard the boards of the ROOT round's children by subgame instead (config 5 style) is done
     * by creating one engine per subgame batch: see rs_create_batch */
    uint32_t flags;            /* RS_FLAG_* */
    uint32_t threads_per_block; /* 0 = default */
    /* train() discount schedule (cfr.rs:190-194,248-262); 0 interval = off */
    uint64_t discount_interval;
    uint64_t discount_cap;
} rs_config;
#define RS_FLAG_NO_GRAPH 1u     /* launch kernels directly instead of replaying a CUDA graph */
#define RS_FLAG_NO_CHAIN_SPLIT 2u /* keep one task per node on rounds with one or two boards (default: such rounds are
                                     chains of dependent tasks and their node tasks are split so that each level of
                                     the chain only waits for what it needs; results are identical either way) */
#define RS_FLAG_STREET_KERNEL 4u /* walk the final betting round with the fused street kernel (one CTA per (board, street
                                    segment); terminals valued four reach rows at a time by list walks with running sums,
                                    csrc/street_kernel.cu) instead of the per-(node, board) dataflow tasks.  Same values up
                                    to fp32 rounding.  Lossy (bucketed) final rounds and nodes wider than 5 actions always
                                    take the task path */
#define RS_FLAG_SHARD_ISOLATED 8u /* world_size > 1 without peers: the rank walks only its own slice of the first dealt-card
                                     level (rank r of world_size) and never exchanges; the other ranks' boards contribute zero
                                     to the chance-node sums.  No NCCL communicator is created.  This is public-chance
                                     sub-sampling without an importance weight: used to solve / check a slice of a subgame
                                     that is too large to hold (config 4 on 2 of its 49 turn cards) */
#define RS_FLAG_ALL (RS_FLAG_NO_GRAPH | RS_FLAG_NO_CHAIN_SPLIT | RS_FLAG_STREET_KERNEL | RS_FLAG_SHARD_ISOLATED) /* rs_create rejects other bits */

typedef struct rs_engine rs_engine;

typedef struct rs_stats {
    uint64_t iterations;            /* completed iterations (both players traversed, cfr.rs:216-226) */
    uint64_t updates_per_iteration; /* infoset-action cells updated per iteration on THIS rank */
    uint64_t updates_per_iteration_global;
    double device_ms;               /* CUDA-event time spent inside rs_iterate */
    uint64_t kernel_launches;       /* kernels launched (or graph-replayed) by rs_iterate */
    uint64_t table_bytes;           /* regret + strategy_sum bytes resident on this rank */
    uint32_t n_rounds;
    uint32_t n_boards[3];           /* global boards per round_idx */
    uint32_t n_boards_local[3];
    uint32_t n_hands[2];
    uint64_t n_combos;              /* generate_all_hole_card_combos().len() (cfr.rs:73-98) */
} rs_stats;

const char* rs_last_error(void);
int rs_version(void);
/* number of usable CUDA devices, 0 when none (never fails) */
int rs_device_count(void);
/* fills RS_NCCL_ID_BYTES bytes; call on rank 0 and broadcast */
int rs_nccl_unique_id(uint8_t* out);

/* Board-sharded engines (world_size > 1) exchange the counterfactual values of the shared chance nodes once per
 * traversal (cfr.rs:512-521 sums over the dealt cards).  By default that is an ncclAllReduce between two launches.
 * With the buffers below mapped into every rank the traversal kernel does the exchange itself: each GPU stores its
 * partial sums into its peers' buffers over NVLink and adds the arrived partials in rank order, one launch per
 * traversal.  Every rank exports a handle (a CUDA IPC handle, one process per GPU), the host gathers them, every
 * rank imports all of them in rank order; all ranks must do so at the same point of their call sequence. */
/* Batched suit-isomorphic hand indexing on the device: out[i] = hand_indexer_s::get_index of the (2 + n_board_cards)
 * cards at cards + i * (2 + n_board_cards), hole cards first (indexer init(2, [2, n_board_cards]),
 * card_abstraction.rs:88-90,205).  This is what rs_create uses to build the card tables (generate_maps,
 * card_abstraction.rs:75-184); exported so that the host can index hands in bulk, e.g. to apply a cluster_arr.
 * kernel_ms may be NULL. */
int rs_gpu_index_hands(uint32_t n_board_cards, const uint8_t* cards, size_t n, uint64_t* out, float* kernel_ms);

/* Abstraction generation, the data-parallel part (src/gen_abstraction): distances between hand-strength histograms
 * and the k-means assignment step.  Host buffers in and out; histograms are row-major [n][dim], dim <= 128.
 *   RS_DIST_EMD_1D  emd::emd_1d  (gen_abstraction/emd.rs:54-113), the linear-time EMD approximation
 *   RS_DIST_L2      kmeans::l2_dist (gen_abstraction/kmeans.rs:622-630)
 * rs_kmeans_assign            = Kmeans::predict (kmeans.rs:173-211): cluster[i] = first nearest centre; min_dist,
 *                               inertia (sum of the minima, fp64, point order) and kernel_ms may be NULL
 * rs_histogram_distances      = out[i] = dist(p_i, q_i)
 * rs_kmeans_update_min_dists  = update_min_dists (kmeans.rs:603-619): min_dists[i] = min(min_dists[i], dist(x_i, c)^2)
 * Distances are bit-identical to the fp32 arithmetic of the reference evaluated in its order. */
#define RS_DIST_EMD_1D 0u
#define RS_DIST_L2 1u
int rs_kmeans_assign(const float* points, size_t n, uint32_t dim, const float* centers, uint32_t k, uint32_t dist_kind,
                     uint32_t* cluster, float* min_dist, double* inertia, float* kernel_ms);
int rs_histogram_distances(const float* p, const float* q, size_t n, uint32_t dim, uint32_t dist_kind, float* out);
/* Kmeans::fit_regular (kmeans.rs:497-599): `rounds` rounds (the reference runs 10) of Lloyd's algorithm with its
 * Hamerly-style bounds -- init_s (265-284) and reassign_clusters (285-334) on the device, the centre update on the host
 * in the reference's summation order.  centers [k][dim] in/out (k >= 2), cluster [n] out, inertia (may be NULL) = the
 * reference's final figure, the mean upper bound.  Deterministic where the reference races (its s vector and bounds
 * are restated as written, including s not being reset between rounds). */
int rs_kmeans_fit_regular(const float* points, size_t n, uint32_t dim, float* centers, uint32_t k, uint32_t dist_kind,
                          uint32_t rounds, uint32_t* cluster, float* inertia);
/* generate_histograms (gen_abstraction/main.rs:79-159): the k-means features.  For the canonical hands
 * [first_index, first_index + count) of `round` (0 preflop .. 3 river; indexers of ehs.rs:26-31, un-indexed like
 * main.rs:117-121) draw `samples` random completions of the board (rejection sampling, main.rs:129-140), bin the EHS of
 * the seven cards (get_bin, main.rs:58-70) and divide by the sample count.  The reference looks the EHS up in ehs.dat,
 * a Monte-Carlo table this repository does not have (src/bin/gen_ehs.rs, out of scope); here it is computed exactly
 * on the device: (wins + ties / 2) / 990 against every opponent hole-card combo.  Random stream of hand i: splitmix64
 * from seed + 0x9E3779B97F4A7C15 * (i + 1), card = z % 52, redrawn while taken.  out [count][bins] (bins <= 128);
 * cards_out [count][7] (may be NULL) = the un-indexed hands (first 2 + board cards of every row); kernel_ms may be NULL. */
int rs_generate_histograms(uint32_t round, uint64_t first_index, size_t count, uint32_t samples, uint32_t bins, uint64_t seed,
                           float* out, uint8_t* cards_out, float* kernel_ms);
/* Kmeans::fit_growbatch (kmeans.rs:336-494), the fit gen_emd runs (main.rs:368, batch 10 000).  The reference's loop
 * ends with an unconditional `break` (kmeans.rs:492): ONE pass -- shuffle the data set (SliceRandom::shuffle on the
 * stated splitmix64(seed) stream: for i in (1..n).rev() swap(i, z % (i + 1))), init_s from f32::MAX, assign the first
 * initial_batch_size shuffled points with fresh bounds (assignment_with_bounds, kmeans.rs:212-262, on the device),
 * accumulate them in shuffled order and replace the centres by the means.  centers [k][dim] in/out (k >= 2);
 * batch_index_out [batch] = data-set index of every batch point, cluster_out [batch] = its centre, stats_out [2] =
 * {min_change (kmeans.rs:463-467), inertia (kmeans.rs:473)} as the reference prints them; all three may be NULL. */
int rs_kmeans_fit_growbatch(const float* points, size_t n, uint32_t dim, float* centers, uint32_t k, uint32_t dist_kind,
                            uint32_t initial_batch_size, uint64_t seed, uint32_t* batch_index_out, uint32_t* cluster_out,
                            float* stats_out);
int rs_kmeans_update_min_dists(const float* points, size_t n, uint32_t dim, const float* new_center, uint32_t dist_kind,
                               float* min_dists);
/* Seeding of the centres.  The reference draws from an unspecified `R: Rng`; here the stream is splitmix64(seed),
 * gen_range(0, n) = z % n, a uniform f32 = (z >> 40) * 2^-24, WeightedIndex = the first index whose running f32 sum of
 * the weights exceeds u * total, choose_multiple = a partial Fisher-Yates shuffle.  chosen_out[k] = indices of the
 * points taken as centres, centers_out [k][dim] (may be NULL) = those points.
 * rs_kmeans_init_pp     = Kmeans::init_pp (kmeans.rs:60-90): k-means++, one distance sweep on the device per centre
 * rs_kmeans_init_random = Kmeans::init_random (kmeans.rs:103-166): of n_restarts random sets the most spread out one
 *                         (largest mean pairwise centre distance, the last one on ties) */
int rs_kmeans_init_pp(const float* points, size_t n, uint32_t dim, uint32_t k, uint32_t dist_kind, uint64_t seed, uint32_t* chosen_out,
                      float* centers_out);
int rs_kmeans_init_random(const float* points, size_t n, uint32_t dim, uint32_t k, uint32_t n_restarts, uint32_t dist_kind, uint64_t seed,
                          uint32_t* chosen_out, float* centers_out);

#define RS_EXCHANGE_HANDLE_BYTES 64
int rs_exchange_export(rs_engine* e, uint8_t* out /* RS_EXCHANGE_HANDLE_BYTES */);
int rs_exchange_import(rs_engine* e, const uint8_t* handles /* n_ranks * RS_EXCHANGE_HANDLE_BYTES */, uint32_t n_ranks);
/* rs_exchange_import is all-or-nothing on one rank (a failed mapping leaves that rank on the NCCL path).  The switch
 * must be unanimous: when any rank failed, the others call rs_exchange_disable to return to the NCCL path too. */
int rs_exchange_disable(rs_engine* e);


int rs_create(const rs_tree* tree, const rs_ranges* ranges, const rs_abstraction* abs,
              const rs_config* cfg, rs_engine** out);
/* Batch of independent subgames sharing one tree shape and abstraction kind but with their own
 * boards (BASELINE config 5): board_masks[n_subgames]; ranges are given unfiltered and each
 * subgame drops the combos hitting its own board.  Subgames behave as extra boards of round 0. */
int rs_create_batch(const rs_tree* tree, const rs_ranges* ranges, const rs_abstraction* abs,
                    const rs_config* cfg, const uint64_t* board_masks, uint32_t n_subgames,
                    rs_engine** out);
void rs_destroy(rs_engine* e);

/* train(): run n_iters synchronous full-tree CFR iterations; returns after the device is idle */
int rs_iterate(rs_engine* e, uint64_t n_iters);
/* MCCFR-style iteration: train() samples the run-out of the board for every iteration (generate_hand,
 * cfr.rs:100-143, 209) and traverses only that deal.  Here the host keeps the RNG and passes n_paths sampled
 * run-outs, `dealt[n_paths][n_rounds-1]` cards in deal order; paths must start with distinct cards.  One call =
 * one iteration (player 0 then player 1) over the root street and the sampled boards, for ALL hands at once
 * (public chance sampling); values are importance-weighted by (#possible deals)/(#sampled) so the update is an
 * unbiased estimate of the full iteration's.  On a board-sharded engine the call is collective: every rank passes the
 * SAME paths and walks those whose first card lies in its own slice (the chance-node sums are exchanged as usual).
 * The discount schedule of rs_config applies to these iterations too. */
int rs_iterate_sampled(rs_engine* e, const uint8_t* dealt, uint32_t n_paths);
/* generate_hand's board part (cfr.rs:100-122): n_paths run-outs of n_cards cards each into dealt_out[n_paths][n_cards].
 * Every card is uniform over 0..51 and drawn again while it is on the board or earlier in the same path, as the
 * reference does; distinct_first != 0 also draws again while an earlier path starts with the same card
 * (rs_iterate_sampled needs distinct first cards).  The reference's SmallRng is unspecified; here the stream is
 * splitmix64(seed) and a card is z % 52 with the top of the 64-bit range rejected (exactly uniform).  Host only. */
int rs_sample_runouts(uint64_t seed, uint64_t board_mask, uint32_t n_cards, uint32_t n_paths, int distinct_first, uint8_t* dealt_out);
/* discount sweep of train()'s monitor thread (cfr.rs:248-261): every table *= d */
int rs_discount(rs_engine* e, float d);
/* Bounded waits.  The traversal kernel waits on flags: of its own producer tasks and, with the in-kernel exchange, of
 * the PEER GPUs (rs_exchange_import).  A peer that never launches the same traversal -- a rank that failed, or a
 * rank-asymmetric call: rs_iterate, rs_iterate_sampled, rs_best_response, rs_average_value and rs_profile_iteration
 * are COLLECTIVE on a sharded engine, every rank must make the same calls in the same order -- would leave the others
 * spinning for ever.  Every wait therefore gives up after `ms` milliseconds (default 30 000; 0 = unbounded) or as
 * soon as rs_abort() was called (from any host thread, while the kernel runs): the launching call returns
 * RS_ERR_CUDA, the tables are partly updated and the engine refuses further work (destroy it and create a new one).
 * Ranks on the NCCL path (no rs_exchange_import) block inside ncclAllReduce instead, which this library cannot bound. */
int rs_set_wait_timeout_ms(rs_engine* e, uint64_t ms);
int rs_abort(rs_engine* e);
/* Pruning as train() switches it on for an iteration (cfr.rs:219): a traverser action whose regret is <= threshold
 * is not explored, i.e. its regret is left alone by the update (cfr.rs:352,379-386,419-440); the node value is
 * unaffected (regret matching gives it probability 0).  The reference's -10 000 000 is in units of S = 100
 * (cfr.rs:424): pass -1e5 for the same cut on this engine's unscaled fp32 regrets.  -INFINITY (the default)
 * switches pruning off.  Applies to rs_iterate and rs_iterate_sampled from the next call on. */
int rs_set_prune_threshold(rs_engine* e, float threshold);
/* External sampling for every hand at once -- the opponent arm of mccfr() (cfr.rs:466-475): at an opponent action node
 * each opponent hand draws ONE action from its current strategy (WeightedIndex over get_strategy()) and continues on
 * that child only; the traverser still explores every action (cfr.rs:378-400).  The draw of hand slot h at action node
 * n on (global) board b in traversal number t (counted from this call, both players' traversals) is
 *     key = splitmix64_finalize(seed + 0x9E3779B97F4A7C15 * t)
 *     z   = splitmix64_finalize'(key ^ n << 44 ^ b << 20 ^ h),  u = (z >> 40) / 2^24
 * (the two 64-bit mixers of splitmix64; see xs_uniform in csrc/kernels.cuh), and the action is the first a with
 * u < sigma_0 + ... + sigma_a.  It does not depend on the GPU count, the sharding or the launch schedule.
 *   RS_OPP_FULL               every action with reach * sigma (the vector form of cfr(), the default)
 *   RS_OPP_SAMPLE             the drawn action keeps the hand's whole reach: unbiased external sampling
 *   RS_OPP_SAMPLE_TIMES_SIGMA the drawn action keeps reach * sigma(drawn action): what the reference's code does
 *                             (cfr.rs:474 multiplies cfr_reach by strategy[a_idx] after sampling a_idx)
 * Applies to rs_iterate and rs_iterate_sampled from the next call on (those launches are not graph replays); best
 * response and average-strategy walks are never sampled.  Not available with RS_FLAG_STREET_KERNEL. */
#define RS_OPP_FULL 0u
#define RS_OPP_SAMPLE 1u
#define RS_OPP_SAMPLE_TIMES_SIGMA 2u
int rs_set_opponent_sampling(rs_engine* e, uint32_t mode, uint64_t seed);
/* Update rule of the traverser's table update.  Let t = 1, 2, ... count the rs_iterate iterations since the rule was
 * set or since rs_reset.  In iteration t the traverser rewrites every row of its (round, player) table as
 *     R' = (R > 0 ? fp : fn) * R + (R > prune_threshold ? d_a : 0)      CFR_PLUS only: R' = max(R', 0)
 *     S' = fs * S + sigma_a * w
 * (d_a = cfv_a - cfv_node summed over the row's hands, w = the row's reach mass) with the factors of iteration t - 1
 * (all 1 for t = 1):
 *   RS_RULE_VANILLA   fp = fn = fs = 1 (the default, vanilla CFR)
 *   RS_RULE_DCFR      fp = (t-1)^alpha / ((t-1)^alpha + 1), fn = (t-1)^beta / ((t-1)^beta + 1), fs = ((t-1) / t)^gamma
 *                     (discounted CFR, Brown & Sandholm 2019; 1.5, 0, 2 are the published defaults)
 *   RS_RULE_LCFR      DCFR with alpha = beta = gamma = 1 (linear CFR; the parameters are ignored)
 *   RS_RULE_CFR_PLUS  fp = fn = 1, fs = (t-1) / t, regrets floored at 0 (CFR+; the parameters are ignored)
 * The host computes each factor in double precision and rounds it to fp32.  The discount is applied lazily: a row is
 * multiplied when its owner next updates it, with no extra pass over the tables.  It changes no strategy: regret
 * matching reads only the positive regrets, which share one factor, and the average strategy is normalised.  The stored
 * tables (rs_read_infoset) are the recursion above, i.e. the discounted sums lag one iteration's factor behind.  The
 * discount_interval schedule and rs_discount scale uniformly and compose with every rule.
 * The lazy form needs every row of the traverser's table rewritten in every iteration, which rs_iterate does (with
 * pruning and with sampled opponent actions too).  rs_iterate_sampled does not, so it returns RS_ERR_UNSUPPORTED while a
 * rule other than VANILLA is set; so does this call with such a rule on an engine created with RS_FLAG_STREET_KERNEL.
 * Applies from the next iteration on; rs_reset restarts t at 1 and keeps the rule.  NaN or infinite parameters and
 * unknown kinds are RS_ERR_INVALID.  On a board-sharded engine the call is local (not collective), but every rank must
 * set the same rule.  rs_get_update_rule returns the rule and t of the last iteration run under it (0 before the first);
 * either output may be NULL.  rs_profile_iteration runs an iteration too and advances t like rs_iterate. */
#define RS_RULE_VANILLA 0u
#define RS_RULE_DCFR 1u
#define RS_RULE_LCFR 2u
#define RS_RULE_CFR_PLUS 3u
typedef struct rs_update_rule {
    uint32_t kind; /* RS_RULE_* */
    float alpha, beta, gamma;
} rs_update_rule;
int rs_set_update_rule(rs_engine* e, const rs_update_rule* rule);
int rs_get_update_rule(rs_engine* e, rs_update_rule* out, uint64_t* t_out);
int rs_reset(rs_engine* e);

/* infoset_table[round,player][board][action node] -> [row][n_actions] (README.md:45-47).
 * an_index is ActionNode.index; board_id indexes the round's board table (rs_board_id).
 * Either output may be NULL.  *n_rows_out / *n_actions_out report the slab shape. */
int rs_read_infoset(rs_engine* e, uint32_t an_index, uint32_t board_id, float* regrets,
                    float* strategy_sum, size_t cap_floats, uint32_t* n_rows_out,
                    uint32_t* n_actions_out);
int rs_write_infoset(rs_engine* e, uint32_t an_index, uint32_t board_id, const float* regrets,
                     const float* strategy_sum, size_t n_floats);
/* Infoset::get_final_strategy (infoset.rs:104-123) for every row of the slab */
int rs_average_strategy(rs_engine* e, uint32_t an_index, uint32_t board_id, float* out,
                        size_t cap_floats, uint32_t* n_rows_out, uint32_t* n_actions_out);
/* Infoset::get_strategy (infoset.rs:83-102) for every row of the slab */
int rs_current_strategy(rs_engine* e, uint32_t an_index, uint32_t board_id, float* out,
                        size_t cap_floats, uint32_t* n_rows_out, uint32_t* n_actions_out);
/* Headerless little-endian dump of the average strategy in the style of the reference's abstraction files
 * (gen_abstraction/main.rs:372-380, read back by card_abstraction.rs:227-229): for every action node in
 * ActionNode.index order, for every board of its round this rank owns in board-id order, the fp32 slab
 * [row][n_actions] of Infoset::get_final_strategy (infoset.rs:104-123).  The reference's calc_br / strategy export
 * is a stub (cfr.rs:629-744).  n_floats_out may be NULL. */
int rs_dump_average_strategy(rs_engine* e, const char* path, uint64_t* n_floats_out);

/* board table (README.md:41-43): dealt cards beyond the root board, in deal order -> board id */
int rs_board_id(rs_engine* e, uint32_t round_idx, const uint8_t* dealt, uint32_t n_dealt,
                uint32_t* board_id_out);
/* card table (README.md:36-39): hand slot -> row (0xFFFF = hand hits the board) */
int rs_card_table(rs_engine* e, uint32_t round_idx, uint32_t player, uint32_t board_id,
                  uint16_t* rows_out, size_t cap, uint32_t* n_rows_out);

/* out[p] = value of player p's best response against the other player's average strategy,
 * in the reference's payoff convention (+-pot, cfr.rs:525-556), per deal.
 * exploitability = (out[0] + out[1]) / 2. */
int rs_best_response(rs_engine* e, double out[2]);
/* out[p] = expected value for player p when both play their average strategies */
int rs_average_value(rs_engine* e, double out[2]);
/* counterfactual values at the root for the last traversal of `player` in rs_iterate */
int rs_root_values(rs_engine* e, uint32_t player, float* out, size_t cap);

int rs_stats_get(rs_engine* e, rs_stats* out);

/* Per-hand reach weights of `player`'s range at the root (n = n_hands[player]; default 1.0 = the
 * reference's unweighted HandRange, cfr.rs:124).  Copied host->device on the engine's stream; the
 * next rs_iterate sees them.  This is the per-step host input of a re-solve loop. */
int rs_set_range_weights(rs_engine* e, uint32_t player, const float* weights, size_t n);

/* Kernel-level profile of ONE iteration launched kernel by kernel (no graph) with a CUDA event pair
 * around every launch on the engine's stream.  The iteration is a real one (tables are updated). */
#define RS_KERNEL_TRAVERSAL 0 /* persistent task kernel: the rounds above the final one (or one phase of them);
                                 the whole traversal when the final round is not eligible for the street kernel */
#define RS_KERNEL_STREET 1    /* fused final-street kernel: every board and street segment of the last betting round */
#define RS_KERNEL_ALLREDUCE 3
typedef struct rs_kernel_time {
    uint32_t kind;      /* RS_KERNEL_* */
    uint32_t phase;     /* RS_KERNEL_TRAVERSAL: 0 = down pass above the final round, 1 = gathers + up pass,
                           2 = the part of a sharded traversal after the all-reduce */
    uint32_t traverser;
    uint32_t grid;      /* CTAs launched */
    float ms;           /* CUDA-event duration */
    uint64_t table_bytes; /* algorithmic infoset-table bytes of this launch: 16 B per traverser cell
                             (regret + strategy_sum read+write) + 4 B per opponent cell (regret read) */
    uint64_t vector_bytes; /* reach / value vectors read or written in HBM by this launch */
} rs_kernel_time;
int rs_profile_iteration(rs_engine* e, rs_kernel_time* out, size_t cap, uint32_t* n_out);

/* Tuning aid: per task kind [count, wait cycles, body cycles, total cycles] accumulated by builds compiled with
 * -DRS_TASK_TIMING (all zeros otherwise); out32 holds 96 words: 8 kinds x 4 counters, then per (kind, round)
 * [earliest start, latest end] in globaltimer ns. */
int rs_debug_task_timing(rs_engine* e, unsigned long long* out32, int reset);

/* ---- host-only plan introspection (no GPU needed): integer parity surface ---- */
typedef struct rs_plan rs_plan;
int rs_plan_create(const rs_tree* tree, const rs_ranges* ranges, const rs_abstraction* abs,
                   const rs_config* cfg, const uint64_t* board_masks, uint32_t n_subgames,
                   rs_plan** out);
void rs_plan_destroy(rs_plan* p);
int rs_plan_stats(const rs_plan* p, rs_stats* out);
int rs_plan_board_id(const rs_plan* p, uint32_t round_idx, const uint8_t* dealt, uint32_t n_dealt,
                     uint32_t* board_id_out);
int rs_plan_card_table(const rs_plan* p, uint32_t round_idx, uint32_t player, uint32_t board_id,
                       uint16_t* rows_out, size_t cap, uint32_t* n_rows_out);
/* element offset of slab (an_index, board_id) inside its (round,player) table, and its shape */
int rs_plan_infoset_offset(const rs_plan* p, uint32_t an_index, uint32_t board_id,
                           uint64_t* offset_out, uint32_t* n_rows_out, uint32_t* n_actions_out);
/* showdown ordering of `player`'s live hands on a final-round board: hand slots, weakest first,
 * and for each slot its strength-class id (equal id = tie) */
int rs_plan_showdown_order(const rs_plan* p, uint32_t player, uint32_t board_id,
                           uint16_t* order_out, uint32_t* class_out, size_t cap,
                           uint32_t* n_live_out);

/* The final betting round as the fused street kernel sees it (csrc/street.h): out = {eligible, segments, max reach rows
 * per segment, max value slots, max showdown quads, max mass-only quads, opponent-node ops, traverser-node ops}.  When
 * the round is not eligible rs_last_error() says why (bucketed tables, a node wider than 5 actions, the flag). */
/* The board-local index tables the traversal kernel evaluates terminals with (csrc/tasks.h: HandRec and the cl_pos entry
 * format), for host-side checks: hrec_words_out [Hpad][4] = `player` as traverser, cl_pos_out [2 * Hpad] = `player` as
 * opponent, slot_of_pos_out [Hpad] = hand slot at every board-local position; dims_out = {Hpad, live hands}.  Any output
 * pointer may be NULL; call once with all NULL to size the buffers. */
int rs_plan_local_tables(const rs_plan* p, uint32_t round_idx, uint32_t player, uint32_t board_id, uint32_t* hrec_words_out,
                         uint16_t* cl_pos_out, uint16_t* slot_of_pos_out, uint32_t dims_out[2]);
/* Host-side proof obligation of the traversal kernel's scheduler: tickets are handed out in order and an instance waits
 * for its producers, so the execution order (ticket -> instance slot; a large final round is walked parent board by parent
 * board, force_board_major != 0 applies that whatever the size) must run every producer before its consumers.  Rebuilds the
 * order exactly as rs_create does and checks it against a host mirror of the dispatcher's dependency resolution.
 * RS_OK = deadlock-free; n_moved_out = slots that are not at their task-major ticket.  force_board_major < 0 is the
 * checker's self-test: the reversed order, which must come back as RS_ERR_INVALID. */
int rs_plan_check_execution_order(const rs_plan* p, uint32_t traverser, int force_board_major, uint32_t* n_tickets_out,
                                  uint32_t* n_moved_out);
int rs_plan_street_info(const rs_plan* p, uint32_t traverser, uint32_t out[8]);
/* The list programs that drive the terminal evaluation of `traverser` on a final-round board (csrc/street.h): words
 * [l_steps][52 * 4] of the pieces of the card lists followed by [c_steps][128] of the pieces of the global strength
 * order, and the two per-position words (cards, pieces, identical combo) of the traverser's hands, hinfo[Hpad][2].
 * dims_out = {l_steps, c_steps, Hpad of the traverser, Hpad of the opponent}.  words_out == NULL: only the sizes. */
int rs_plan_street_program(const rs_plan* p, uint32_t traverser, uint32_t board_id, uint32_t* words_out, size_t cap,
                           uint32_t* n_words_out, uint32_t* hinfo_out, size_t hinfo_cap, uint32_t dims_out[4]);

#ifdef __cplusplus
}
#endif
#endif /* B200CFR_H */
