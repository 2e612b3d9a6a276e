/* smz.h — C ABI of the B200-native batched Stochastic-MuZero search engine.
 *
 * Drop-in boundary for the search path of DHDev0/Stochastic-muzero:
 *   monte_carlo_tree_search.py:75-349  (Monte_carlo_tree_search / Node / MinMaxStats / Player_cycle)
 *   muzero_model.py:802-909            (the five *_function_inference calls one simulation makes)
 * The reference has no FFI; these entry points are what a binding for that path would call
 * (see INTEGRATION.md for the ctypes stub that replaces `mcts.run` at self_play.py:46, :85, :419).
 *
 * Conventions
 *   - plain C, no exceptions cross the boundary; every call returns 0 (SMZ_OK) or a negative
 *     SMZ_E_* code, with a thread-local message available from smz_last_error().
 *   - pointers named *_dev are CUDA device pointers owned by the CALLER (e.g. torch tensors'
 *     data_ptr()); pointers named *_host are host memory.  The engine owns only its arena, which is
 *     allocated once in smz_create and never grows; smz_simulate never allocates.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises
 *     implicitly.  One engine per (device, stream); an engine is NOT thread-safe, mirroring the
 *     reference whose run() mutates self.* (monte_carlo_tree_search.py:313-349).
 */
#ifndef SMZ_H_
#define SMZ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMZ_ABI_VERSION 2

enum {
  SMZ_OK = 0,
  SMZ_E_INVALID_ARG = -1,
  SMZ_E_CUDA = -2,
  SMZ_E_CAPACITY = -3,
  SMZ_E_STATE = -4
};

/* where the per-simulation network outputs come from */
enum {
  SMZ_NET_EXTERNAL = 0, /* caller supplies policy/value/reward (tape replay, host-model callback)   */
  SMZ_NET_FP32 = 1,     /* fused fp32 CUDA-core MLP step (parity mode, 1e-5 vs the reference)       */
  SMZ_NET_BF16 = 2,     /* fused bf16 tcgen05/TMEM MLP step, fp32 accumulate (throughput mode)      */
  SMZ_NET_TC32 = 4,     /* fused tcgen05/TMEM MLP step at the reference's precision: every fp32 operand split into
                         * fp16 hi + lo, three products per K-step into one fp32 accumulator (1e-5 vs the reference,
                         * like SMZ_NET_FP32, at tensor-core speed); |activations| must stay below 65504            */
  SMZ_NET_F16 = 5,      /* the same chain on plain fp16 operands (one product per K-step, fp32 accumulate): throughput
                         * mode with 11-bit significands instead of bf16's 8; same range limit as SMZ_NET_TC32          */
  SMZ_NET_VISION = 3    /* vision (ResNet-v2, neural_network_vision_model.py) family, fp32 CUDA cores:
                         * obs_dim must be 3*98*98 (the reference fixes the model input, muzero_model.py:336),
                         * hidden state 3x7x7, state_dim/hidden_dim/num_hidden_layers = S/H/L of the MLP
                         * heads and residual trunks, chance_dim == action_dim                           */
};

/* where uniform draws come from */
enum {
  SMZ_RNG_PHILOX = 0, /* device Philox4x32-10 keyed by (seed, global tree id), see oracle/mcts_oracle.py */
  SMZ_RNG_TAPE = 1    /* caller-supplied doubles in consumption order (record/replay parity tests)      */
};

typedef struct smz_engine smz_engine;

/* Search + model shape.  The nine search fields are the ctor arguments of the reference
 * (monte_carlo_tree_search.py:76-85; JSON section "monte_carlo_tree_search", self_play.py:639-647). */
typedef struct smz_config {
  int32_t abi_version;       /* SMZ_ABI_VERSION */
  int32_t device;            /* CUDA device ordinal */
  int32_t max_trees;         /* B: concurrent trees this engine can hold */
  int32_t num_simulations;   /* N */
  int32_t action_dim;        /* A: width of prediction policy (root + dynamics-expanded nodes) */
  int32_t chance_dim;        /* C: width of afterstate-prediction policy (== A in the reference) */
  int32_t max_action_sample; /* maxium_action_sample: children per non-root node = min(this, width) */
  int32_t pb_c_base;
  double pb_c_init;
  double discount;           /* rounded to float32 before use (numpy weak-scalar semantics, T1/T4) */
  double root_dirichlet_alpha;
  double root_exploration_fraction;
  /* MLP shape (muzero_model.py ctor: observation/state_space_dimensions, hidden_layer_dimensions,
   * number_of_hidden_layer).  Ignored when net_mode == SMZ_NET_EXTERNAL. */
  int32_t obs_dim;           /* flattened observation width, 1..8192 for the MLP modes (the first layer streams its K
                              * through the tensor / CUDA cores in slices of 128); 3*98*98 for SMZ_NET_VISION */
  int32_t state_dim;         /* S: hidden-state width and categorical-support size */
  int32_t hidden_dim;        /* H */
  int32_t num_hidden_layers; /* L (weight-tied, neural_network_mlp_model.py:31-37) */
  int32_t net_mode;          /* SMZ_NET_* */
  int32_t rng_mode;          /* SMZ_RNG_* */
  int32_t lanes_per_tree;    /* 0 = auto; else 2,4,8,16,32 (threads cooperating on one tree) */
  int32_t record;            /* 1: keep per-simulation network outputs + dirichlet for smz_read_record */
  uint64_t seed;             /* Philox key */
  uint64_t tree_id_offset;   /* global id of local tree 0 (shard-invariant RNG across GPUs) */
} smz_config;

/* Sizes derived from a config (for callers that allocate I/O buffers). */
typedef struct smz_dims {
  int32_t nodes_per_tree;    /* 1 + A + N*Kmax */
  int32_t max_children;      /* Kmax = max(min(K,A), min(K,C)) */
  int32_t policy_stride;     /* floats per policy row in every policy buffer = max(A, C) */
  int32_t hidden_stride;     /* floats per hidden-state row (S rounded up to 64) */
  int32_t hidden_slots;      /* N + 1 */
  int32_t path_stride;       /* N + 2 */
  int32_t lanes_per_tree;
  int32_t reserved;
  uint64_t weight_blob_floats; /* size of the fp32 weight blob smz_set_weights expects (0 if external) */
  uint64_t arena_bytes;
} smz_dims;

/* One tree copied out in arena order (host memory owned by the caller, nodes_per_tree entries each).
 * Node 0 is the root, nodes 1..A its children (node 1 + a = action a); a node expanded by simulation s owns the
 * children block starting at 1 + A + s*Kmax.  A root child whose action was illegal (smz_root_legal) is a sentinel:
 * key -1, prior 0, child_base 0, never visited. */
typedef struct smz_tree_host {
  int32_t* visit;
  float* value_sum;
  float* reward;
  float* prior;        /* float32 priors (non-root children) */
  int32_t* child_base; /* 0 = not expanded */
  int32_t* key;        /* action / chance-code index of this node in its parent's policy */
  double* root_prior;  /* A entries: float64 priors of the root children (after Dirichlet mixing) */
  float minmax[2];     /* MinMaxStats.minimum / .maximum */
  int32_t n_uniforms;  /* uniform draws consumed so far */
  int32_t root_to_play; /* as stored: root_to_play_dev[tree] wrapped into [0, n_phases) */
} smz_tree_host;

int smz_create(const smz_config* cfg, smz_engine** out);
int smz_destroy(smz_engine* e);
int smz_get_dims(const smz_engine* e, smz_dims* out);
const char* smz_last_error(void);

/* Exploration prefactor table t[n] = sqrt(n) * (log((n + base + 1)/base) + init) for parent visit
 * counts n = 0..N+1 — the left-associated head of `np.sqrt(N) * pb_c * prior` (monte_carlo_tree_search.py:
 * 236-237).  The engine fills it with the C library's sqrt()/log(); a host that needs bit-equality with
 * numpy on the same machine passes its own table (n_entries must be N + 2). */
int smz_set_pbc_table(smz_engine* e, const double* table_host, int32_t n_entries);

/* Player_cycle (monte_carlo_tree_search.py:38-72) flattened per depth.  For each of n_phases
 * possible root_to_play values p and each depth d in [0, N+1]: sign[p*(N+2)+d] = +1/-1 multiplier of
 * the backed-up value (:302-305), to_play[p*(N+2)+d] = Node.to_play at that depth.  Default: one
 * phase, sign +1, to_play 0. */
int smz_set_player_tables(smz_engine* e, const int8_t* sign_host, const int32_t* to_play_host,
                          int32_t n_phases);

/* fp32 weight blob (host or device memory, `on_device` says which); layout in oracle/net_oracle.py
 * docstring and DESIGN.md §weights: torch Linear W[out,in] row-major then b[out], nets in the order
 * repr, pred, adyn, apred, dyn, enc.  The engine repacks it into its padded fp32 / bf16 tile images. */
int smz_set_weights(smz_engine* e, const float* blob, uint64_t n_floats, int32_t on_device, void* stream);

/* New Philox key / global tree-id base for the following searches (each move of each game must see
 * fresh draws).  Stream-ordered; does not invalidate the captured simulation graph. */
int smz_set_seed(smz_engine* e, uint64_t seed, uint64_t tree_id_offset, void* stream);

/* Which nodes of the tree are chance nodes.  The kind of a node at depth d is (d >> 1) & 1 (1 = chance) under
 * SMZ_PATTERN_REFERENCE, the reference's F,F,T,T,F,F,... (monte_carlo_tree_search.py:211, :333-345), and d & 1 under
 * SMZ_PATTERN_PAPER, the Stochastic MuZero alternation F,T,F,T,...: the root's children are afterstates, so
 * afterstate_dynamics is applied to states and dynamics to afterstates, pUCT runs over actions and sampling over
 * chance codes.  In both patterns a leaf whose parent is a decision node is evaluated by the afterstate pair and gets
 * min(K, C) children, any other by the dynamics pair (min(K, A) children and a reward); a chance child keeps its
 * parent's to_play, a decision child gets the next player.  Any other value returns SMZ_E_INVALID_ARG.
 * The setting applies from the next smz_root, which copies it into the arena; a search already rooted keeps its
 * pattern.  Default: SMZ_PATTERN_REFERENCE.  A caller that supplies its own smz_set_player_tables must build the
 * to_play / sign tables with the same pattern (the per-depth player step follows the node kinds). */
enum {
  SMZ_PATTERN_REFERENCE = 0,
  SMZ_PATTERN_PAPER = 1
};
int smz_set_node_pattern(smz_engine* e, int32_t pattern);

/* Search policy at decision nodes.  SMZ_SEARCH_PUCT (default) is the reference's pUCT with Dirichlet noise at the root
 * (smz_root / smz_root_legal).  SMZ_SEARCH_GUMBEL is Gumbel MuZero (Danihelka et al., "Policy improvement by planning
 * with Gumbel", ICLR 2022), rooted by smz_root_gumbel and read out by smz_read_gumbel:
 *   - per decision node, over its existing children i (the root: its legal children) with prior p_i (float64 at the
 *     root, float32 below), visit count N_i and q_i = reward + discount * value() in float32 (pUCT's value term before
 *     min-max normalisation), and the node's own network value v: v_mix = (v + sum N * (sum_{N_i>0} p_i q_i) /
 *     (sum_{N_i>0} p_i)) / (sum N + 1) (v when sum N = 0); completed value cq_i = q_i if N_i > 0 else v_mix;
 *     r_i = (cq_i - min cq) / max(max cq - min cq, 1e-8); sigma_i = (c_visit + max N) * c_scale * r_i.  float64, in
 *     this order, sums in ascending child order;
 *   - interior decision nodes: argmax of pi'_i - N_i / (1 + sum N), pi' = p_i exp(sigma_i - max sigma) / sum_j ...;
 *   - root: one Gumbel g_a per legal action per search; logit_a = log p_a - max_b log p_b; the children whose visit
 *     count equals the Sequential Halving schedule T[min(m, |L|)][sum N] compete on max(-1e9, g_a + logit_a + sigma_a);
 *   - ties go to the smaller action, and no decision node draws a uniform; chance nodes and the expansions keep the
 *     reference's draws; no Dirichlet noise is mixed.
 * max_considered in [1, 32] (m, default 16), c_visit >= 0 (default 50), c_scale >= 0 (default 0.1), both finite;
 * anything else, or another policy value, returns SMZ_E_INVALID_ARG.  The setting applies from the next root: in Gumbel
 * mode smz_root / smz_root_legal return SMZ_E_STATE, in pUCT mode smz_root_gumbel does.  A search already rooted keeps
 * its policy; switching drops the captured smz_simulate graph. */
enum {
  SMZ_SEARCH_PUCT = 0,
  SMZ_SEARCH_GUMBEL = 1
};
int smz_set_search(smz_engine* e, int32_t policy, int32_t max_considered, double c_visit, double c_scale);

/* The Sequential Halving schedules of every budget b in [0, num_simulations], as the Gumbel search uses them (host
 * memory, no engine, no GPU): out int32[num_simulations + 1][33][max(num_simulations, 1)], entry (b, n, i) = the visit
 * count the root child of simulation i must have when n actions are considered and the budget is b (i < b; the rest 0). */
int smz_sequential_halving_table(int32_t num_simulations, int32_t* out);

/* Per-tree simulation budgets and exploration flags of the NEXT root step (smz_root, smz_root_legal or smz_root_gumbel),
 * which must root the same n_trees.  budget_dev: int32[n_trees] in [0, N], or NULL (every tree N); explore_dev:
 * uint8[n_trees] (0 / non-zero), or NULL (every tree follows the root step's `train`).  Both are copied on `stream`: the
 * caller's buffers may be reused once the call is enqueued.  A root step not preceded by this call uses N and `train`
 * for every tree.
 * Tree b then behaves bit for bit as the reference's search with num_simulations = budget[b]: same arena, same draws,
 * same min-max bounds, record entries and read-out.  For s >= budget[b] it takes no part in simulation s: no descent,
 * no draw, no row for the network step, no expansion, no backup, no record entry, no depth statistic.  Per tree:
 *   - the exploration flag replaces `train` for that tree's root noise: Dirichlet in pUCT mode, Gumbels in Gumbel mode
 *     (a tree with the flag off is a train = 0 search, with it on a train = 1 search);
 *   - pUCT: no Dirichlet noise for a tree whose budget is 0 (:215-216 per tree); as with train = 0, no noise is drawn
 *     or recorded for a tree without noise;
 *   - Gumbel: the root follows the Sequential Halving schedule of its own budget, T_budget[min(m, |L|)][sum N]
 *     (smz_sequential_halving_table); a budget-0 tree still draws its Gumbels.
 * A budget outside [0, N] raises error flag 4 (smz_read_roots) and that tree is searched with N.  Budgets live in an
 * arena column written by the root step: searches with different budgets replay the same captured smz_simulate graph.
 * smz_simulate(n) still runs n simulation steps; a caller that knows the largest budget runs only that many (a step in
 * which no tree takes part costs its launches only: every network kernel leaves at once when it has no rows). */
int smz_set_root_budgets(smz_engine* e, int32_t n_trees, const int32_t* budget_dev, const uint8_t* explore_dev,
                         void* stream);

/* Tape inputs (rng_mode == SMZ_RNG_TAPE): uniforms_dev is double[n_trees][stride]. */
int smz_set_uniform_tape(smz_engine* e, const double* uniforms_dev, int32_t stride);

/* ---- one search (= Monte_carlo_tree_search.run for n_trees independent observations) ----------- */

/* Root step (monte_carlo_tree_search.py:315-323).  Either obs_dev (float[n_trees][obs_dim], internal
 * network: representation + prediction) or root_policy_dev (float[n_trees][policy_stride], softmaxed,
 * external network) must be given.  root_to_play_dev: int32[n_trees] or NULL (all 0); values are wrapped into
 * [0, n_phases) like Player_cycle.global_step() does (monte_carlo_tree_search.py:55-58).
 * train != 0 mixes Dirichlet noise into the root priors (skipped when N == 0, :215-216);
 * dirichlet_dev: double[n_trees][A] recorded noise, or NULL to draw it on the device. */
int smz_root(smz_engine* e, int32_t n_trees, const float* obs_dev, const float* root_policy_dev,
             const int32_t* root_to_play_dev, int32_t train, const double* dirichlet_dev, void* stream);

/* smz_root with the root of each tree restricted to the legal actions of its position.  legal_dev: uint32[n_trees]
 * (bit a set = action a is legal; A <= 32), or NULL for every action (then this is smz_root).  A tree's root behaves
 * exactly as the reference's root would if its action space were L = the set bits in ascending order: the policy is
 * compacted to policy[L] before normalisation and the draws of root expansion, children are created for L only,
 * Dirichlet noise covers L only (device noise: Gamma draws for the legal actions in ascending order; given noise:
 * the entries at L are used), and the root's pUCT consumes one draw per legal child.  Illegal actions keep their
 * arena slot 1 + a with key -1 (see smz_export_tree), and read out as 0 visits, 0 reward and prior 0.0; smz_select_
 * actions applies its rule to the legal children and never returns an illegal action.  A mask that is empty or has
 * a bit >= A set raises error flag 3 (smz_read_roots) and that tree is searched with every action legal.  The mask
 * is read by the kernels this call enqueues only: the captured smz_simulate graph stays valid. */
int smz_root_legal(smz_engine* e, int32_t n_trees, const float* obs_dev, const float* root_policy_dev,
                   const int32_t* root_to_play_dev, const uint32_t* legal_dev, int32_t train,
                   const double* dirichlet_dev, void* stream);

/* Root step of a Gumbel search (smz_set_search(SMZ_SEARCH_GUMBEL)): smz_root_legal's arguments without Dirichlet noise,
 * plus root_value_dev float[n_trees], the network value of each root — required with root_policy_dev, NULL with obs_dev
 * (the internal network's value is used).  train == 0 sets every Gumbel to 0; with train != 0 (also with N == 0)
 * gumbel_dev is double[n_trees][A] recorded Gumbels (entries at illegal actions are ignored), or NULL to draw them on
 * the device: -log(-log u), u = uniform #rank of Philox stream 3 keyed by (seed, global tree id), rank = position of
 * the action among the legal ones, so the draws do not depend on how trees are sharded.  The legal mask behaves as in
 * smz_root_legal (flag 3 included). */
int smz_root_gumbel(smz_engine* e, int32_t n_trees, const float* obs_dev, const float* root_policy_dev,
                    const float* root_value_dev, const int32_t* root_to_play_dev, const uint32_t* legal_dev,
                    int32_t train, const double* gumbel_dev, void* stream);

/* n_sims full simulations (:325-347) with the internal network (net_mode FP32/BF16). */
int smz_simulate(smz_engine* e, int32_t n_sims, void* stream);

/* ---- fine-grained steps (test hooks, and the external-network loop) ---------------------------- */

/* pUCT / chance descent of simulation `sim` (:262-267).  Optional outputs, each [n_trees] or NULL:
 * leaf_parent_slot (hidden-state slot of search_path[-2]), leaf_action (history[-1]),
 * leaf_branch (0 = afterstate pair :339-342, 1 = dynamics pair :333-337).  A tree without simulation `sim` (its budget
 * is used up, smz_set_root_budgets) gets leaf_parent_slot -1; its other outputs are unspecified, and
 * smz_expand_backup ignores its inputs. */
int smz_select(smz_engine* e, int32_t sim, int32_t* leaf_parent_slot_dev, int32_t* leaf_action_dev,
               int32_t* leaf_branch_dev, void* stream);
/* internal network on the leaves chosen by the last smz_select */
int smz_net_step(smz_engine* e, int32_t sim, void* stream);
/* The tree step exactly as smz_simulate's captured loop runs it between two network steps: expansion + backup
 * of simulation `sim` on the outputs of smz_net_step, fused with the descent of simulation `sim + 1`
 * (sim + 1 < N).  Stand-alone launch (no programmatic dependency): bench.py times the real kernel with it. */
int smz_backup_select(smz_engine* e, int32_t sim, void* stream);
/* expansion + backup of simulation `sim` (:289-308).  With policy_dev == NULL the outputs of
 * smz_net_step are used; else policy_dev float[n_trees][policy_stride] (softmaxed), value_dev /
 * reward_dev float[n_trees]. */
int smz_expand_backup(smz_engine* e, int32_t sim, const float* policy_dev, const float* value_dev,
                      const float* reward_dev, void* stream);

/* Stand-alone network functions on caller rows (parity tests of N1-N6, SURVEY.md §8a).
 * which: 0 repr(obs)->h   1 pred(h)->policy[A],value   2 adyn(h,a)->h'   3 apred(h)->policy[C],value
 *        4 dyn(h,c)->reward,h'   5 enc(obs)->probs[C],code
 * in_dev: float[n_rows][obs_dim] or float[n_rows][hidden_stride]; idx_dev: int32[n_rows] action/code;
 * outputs may be NULL when the function does not produce them. */
int smz_net_eval(smz_engine* e, int32_t which, int32_t n_rows, const float* in_dev, const int32_t* idx_dev,
                 float* hidden_out_dev, float* policy_out_dev, float* value_out_dev, float* reward_out_dev,
                 int32_t* code_out_dev, void* stream);

/* ---- read-out ------------------------------------------------------------------------------------ */

/* Root statistics consumed by Game.store_search_statistics / policy_step (game.py:179-235):
 * visits int32[n][A], root_values float[n] (= Node.value() of the root), priors double[n][A],
 * rewards float[n][A]; error_dev int32[1] = the search's error flag (0 ok, 1 uniform tape exhausted,
 * 2 NaN / all-zero policy met during an expansion — where np.random.choice raises in the reference,
 * monte_carlo_tree_search.py:208/:294, 3 a legal-action mask of smz_root_legal was empty or had a bit >= A set,
 * 4 a budget of smz_set_root_budgets was outside [0, N]), delivered with the same read-out so that the host needs no extra
 * synchronisation to learn about it.  Any pointer may be NULL. */
int smz_read_roots(smz_engine* e, int32_t* visits_dev, float* root_values_dev, double* priors_dev,
                   float* rewards_dev, int32_t* error_dev, void* stream);
/* The step after the search (game.py:179-235), on the device so that B games advance without a host
 * round-trip: stored_policy double[n][A] = visit distribution (priors when fewer than 3 visits,
 * store_search_statistics); policy double[n][A] = visits (priors when <= 1 visit) ** (1/temperature) only
 * if temperature >= 0.3, normalised (softmax_stable); actions int32[n] = sampled from `policy` when
 * temperature > 0.1 or the policy is flat, else first argmax (select_action).  uniforms_dev: double[n]
 * recorded draws, or NULL for device Philox (stream 2).  Any output may be NULL. */
int smz_select_actions(smz_engine* e, double temperature, const double* uniforms_dev, int32_t* actions_dev,
                       double* policy_dev, double* stored_policy_dev, void* stream);
/* Read-out of a Gumbel search: actions_dev int32[n] = argmax over the legal actions with the most visits of
 * g_a + logit_a + sigma_a (with N = 0 a Gumbel-max sample of the prior); improved_policy_dev double[n][A] = softmax
 * over the legal actions of logit_a + sigma_a, 0 for illegal actions (the policy target); gumbels_dev double[n][A] =
 * the search's Gumbels (0 for illegal actions), for replay through smz_root_gumbel.  Any pointer may be NULL.
 * SMZ_E_STATE unless the current search was rooted by smz_root_gumbel. */
int smz_read_gumbel(smz_engine* e, int32_t* actions_dev, double* improved_policy_dev, double* gumbels_dev, void* stream);
/* Network value of every expanded node of a Gumbel search by hidden slot (0 = root, s+1 = node expanded by simulation
 * s): float[n][N+1].  SMZ_E_STATE unless the current search was rooted by smz_root_gumbel. */
int smz_read_raw_values(smz_engine* e, float* out_dev, void* stream);
/* Synchronises `stream`, then copies one tree to host memory. */
int smz_export_tree(smz_engine* e, int32_t tree, smz_tree_host* out, void* stream);
/* Hidden state of a slot (0 = root, s+1 = node expanded by simulation s): float[n][hidden_stride]. */
int smz_read_hidden(smz_engine* e, int32_t slot, float* out_dev, void* stream);
/* record == 1: network outputs of every simulation so a run can be replayed by the CPU oracle.
 * policy float[n][N][policy_stride], value/reward float[n][N], branch int8[n][N],
 * dirichlet double[n][A], root_policy float[n][policy_stride].  Entries of simulations s >= budget[b] of a tree are
 * not written (they hold whatever an earlier search left there). */
int smz_read_record(smz_engine* e, float* policy_dev, float* value_dev, float* reward_dev,
                    int8_t* branch_dev, double* dirichlet_dev, float* root_policy_dev, void* stream);
/* Synchronises `stream`.  Mean leaf depth and kernel-launch count of the last smz_root + smz_simulate, and the
 * number of kernels this engine has launched since smz_create (bench bookkeeping: `gpu_launches`).  The depth is
 * averaged over the simulations actually run, sum over the trees of min(budget, simulations done).  Returns
 * SMZ_E_CAPACITY / SMZ_E_STATE / SMZ_E_INVALID_ARG when the last search raised its error flag 1 / 2 / 3 or 4 (see
 * smz_read_roots). */
int smz_stats(smz_engine* e, double* mean_leaf_depth, int64_t* launches, int64_t* launches_total, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SMZ_H_ */
