/*
 * aqgnn.h -- C ABI of libaqgnn.so, the sm_100a CUDA implementation of the AlphaQuoridorGNN
 * hot path (game_logic legal moves / wall legality, board-graph construction, the
 * pv_network_gnn GCN forward/backward, batched leaf evaluation and lock-step PV-MCTS).
 *
 * The reference (ApproximateCaesar/AlphaQuoridorGNN) is pure Python and has no FFI; the
 * boundary it exposes is the duck-typed BaseNetwork object (BaseNetwork.py:9-54) plus
 * game_logic.State (game_logic.py:15-395).  Each entry point below names the reference
 * function it replaces.  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the name ends in _host;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), allocates
 *     nothing persistent, and keeps no global mutable state (re-entrant per stream);
 *   - return value: 0 = ok, >0 = cudaError_t of the launch, <0 = argument error
 *     (AQ_ERR_*); aq_last_error_string() describes the last failure on this host thread;
 *   - board is 9x9: 81 squares, 64 wall slots, 209 actions (game_logic.py:105-108).
 */
#ifndef AQGNN_H
#define AQGNN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AQ_N 9
#define AQ_SQUARES 81
#define AQ_SLOTS 64
#define AQ_ACTIONS 209
#define AQ_MASK_WORDS 8      /* 256-bit legal mask, bit a = action a */
#define AQ_MAX_LEGAL 136     /* 5 pawn moves + 128 wall actions, rounded up */
#define AQ_FEATURES 6        /* pv_network_gnn.py:17 */
#define AQ_HIDDEN 128        /* pv_network_gnn.py:18 */
#define AQ_HEAD_HIDDEN 64    /* hidden_dim // 2, pv_network_gnn.py:39,47 */
#define AQ_PLIES_FOR_DRAW 116 /* constants.py:20 */

#define AQ_ERR_ARG (-1)
#define AQ_ERR_UNSUPPORTED (-2)

/* Packed game state, 32 bytes.  Mirrors game_logic.State (game_logic.py:15-40):
 *   hwalls bit s  <=> walls[s] == 1,  vwalls bit s <=> walls[s] == 2   (s = 8*row + col)
 *   ppos/pwalls = State.player, epos/ewalls = State.enemy (epos in the ENEMY's own frame),
 *   plies = State.plies_played.  rotate_walls() (game_logic.py:359-364) is a 64-bit
 *   bit reversal in this layout. */
typedef struct AqState {
    uint64_t hwalls;
    uint64_t vwalls;
    uint8_t ppos, pwalls, epos, ewalls;
    uint16_t plies;
    uint16_t flags;    /* reserved, 0 */
    uint64_t reserved; /* reserved, 0 */
} AqState;

#define AQ_VERSION 211 /* bumped with every change of a signature below; the ctypes loader refuses a library of another version */
int aq_version(void);
const char *aq_last_error_string(void);
/* Number of kernels this library has launched in the process so far (monotonic; kernels replayed through a CUDA graph the caller
 * captured are counted once, at capture).  Lets a benchmark report measured launch counts. */
int64_t aq_launch_count(void);

/* State.to_array() rows ("row68": uint8[68] = player[2], enemy[2], walls[64]) <-> AqState.
 * Replaces the python list handling of game_logic.py:96-100. */
int aq_pack_states(const uint8_t *rows68, const int16_t *plies, int64_t B, AqState *out, void *stream);
int aq_unpack_states(const AqState *states, int64_t B, uint8_t *rows68, int16_t *plies, void *stream);

/* State.legal_actions() (game_logic.py:103-117) for B states: legal_actions_pos (120-192),
 * can_place_wall (199-223), the touch-count gate (227-307,327-328) and both path-existence
 * searches (309-348), bit-exact.
 *   mask [B,8] uint32 : bit a set iff action a is legal
 *   pawn [B,8] uint8  : [n_pawn, p0..p4 in the reference's U,D,L,R/jump order (0xFF pad), 0, 0]
 * The ordered action list is pawn[1..n] followed by the wall bits of `mask` in ascending
 * slot order, H before V per slot (game_logic.py:352-355); aq_legal_actions_list emits it. */
int aq_legal_mask(const AqState *states, int64_t B, uint32_t *mask, uint8_t *pawn, void *stream);
/* Same with a caller-provided workspace (the list of path searches that the second kernel of the two-phase form works
 * through): the faster form at every batch size.  aq_legal_mask_ws_bytes(B) is the recommended size; any size >= 4352
 * bytes is valid (states whose searches do not fit the list run them in the first kernel).  ws == NULL selects the
 * one-kernel form, which is what aq_legal_mask runs (the library never allocates).  Results are identical in every form. */
int64_t aq_legal_mask_ws_bytes(int64_t B);
int aq_legal_mask_ws(const AqState *states, int64_t B, uint32_t *mask, uint8_t *pawn, void *ws, int64_t ws_bytes,
                     void *stream);
int aq_legal_actions_list(const uint32_t *mask, const uint8_t *pawn, int64_t B, int16_t *actions /*[B,136], -1 pad*/,
                          int16_t *n_actions /*[B]*/, void *stream);

/* State.next() + is_lose()/is_draw() of the successor (game_logic.py:43-54, 359-391).
 * terminal[b] bit0 = successor.is_lose(), bit1 = successor.is_draw(). terminal may be NULL. */
int aq_state_next(const AqState *states, const int16_t *actions, int64_t B, AqState *out, uint8_t *terminal,
                  void *stream);

/* Board graph + node features (derived from game_logic.py:145-167 and 56-93; the reference has
 * no graph builder -- SURVEY.md section 8a A6).
 *   open_mask [B,81] uint8 : bit k = direction k of MOVEMENT_DIRECTIONS (U,D,L,R) is an edge
 *   dinv      [B,81] f32   : (1 + popcount(open))^-1/2   (gcn_norm with self loops)
 *   x         [B*81,6] f32 : the 6 planes of State.pieces_array read at each square
 *   edge_count[B] int32    : directed edges of board b (may be NULL) */
int aq_build_graph(const AqState *states, int64_t B, uint8_t *open_mask, float *dinv, float *x, int32_t *edge_count,
                   void *stream);
/* PyG-style edge_index for GraphPolicyValueNetwork.forward(x, edge_index, batch)
 * (pv_network_gnn.py:53): edge_offset[B] = exclusive scan of edge_count; src/dst int64[E]. */
int aq_build_edge_index(const uint8_t *open_mask, const int64_t *edge_offset, int64_t B, int64_t *src, int64_t *dst,
                        void *stream);
/* Inverse, for callers that hand us (x, edge_index, batch): rebuild open masks; bad[0] is set to 1 if an edge does not join
 * 4-neighbours of one 9x9 board and to 2 if an edge lacks its reverse (the kernels take a node's own degree where GCNConv's
 * gcn_norm takes the in-degree at the target; the two agree only on symmetric edge lists, which every board graph is). */
int aq_edges_to_open_mask(const int64_t *src, const int64_t *dst, int64_t E, int64_t B, uint8_t *open_mask,
                          int32_t *bad, void *stream);

/* GraphPolicyValueNetwork.forward (pv_network_gnn.py:53-64 + PyG GCNConv/global_mean_pool).
 * params: flat f32[64082] in state_dict order (see aq_param_count / DESIGN.md).
 * Inputs are either `states` (graph built in-kernel) or (x, open_mask) when states == NULL.
 *   policy [B,209] softmax probabilities, value [B] tanh.
 *   saved  NULL for inference, else workspace of aq_gnn_saved_floats(B) floats kept for backward.
 *   precision 0 = fp32 FFMA path, 1 = bf16 tcgen05 tensor-core path (needs packed states). */
int64_t aq_param_count(void);
int64_t aq_gnn_saved_floats(int64_t B);
int aq_gnn_forward(const float *params, const AqState *states, const float *x, const uint8_t *open_mask, int64_t B,
                   float *policy, float *value, float *saved, int precision, void *stream);

/* The two stages of aq_gnn_forward, exposed separately for profiling and tests:
 *   aq_gcn_trunk_forward: graph build + 3 GCN layers + global_mean_pool -> pooled [B,128]
 *   aq_heads_forward:     policy/value MLPs on pooled; legal_mask (may be NULL) applies the
 *                         predict() restriction + renormalisation */
int aq_gcn_trunk_forward(const float *params, const void *prepared, const AqState *states, int64_t B, float *pooled,
                         int precision, void *stream);
int aq_heads_forward(const float *params, const void *prepared, const float *pooled, int64_t B, float *policy,
                     float *value, const uint32_t *legal_mask, int precision, void *stream);

/* Inference weights prepared once per parameter update (the counterpart of the reference's one-time
 * model.eval() / TensorRT compile in BaseNetwork.py:22-32): the bf16 operand tiles of the tensor-core
 * kernels (trunk W1/W2/W3, heads Wp0/Wv0/Wp2) in their shared-memory layout, aq_prepared_bytes() bytes.
 * Every inference entry point takes `prepared` (may be NULL: each CTA then converts the fp32 parameters
 * itself; ignored at precision 0).  The caller must call aq_prepare_inference again after changing
 * params.  Biases and the fp32 value head are always read from params. */
int64_t aq_prepared_bytes(void);
int aq_prepare_inference(const float *params, void *prepared, void *stream);

/* Backward of the above (autograd of train_network.py:93).  dpolicy [B,209], dvalue [B] are the
 * loss gradients w.r.t. the softmax / tanh outputs; grads f32[64082] is OVERWRITTEN with the
 * parameter gradients (flat, same order as params); workspace of aq_gnn_backward_ws_floats(B).
 * precision must equal the precision of the aq_gnn_forward call that filled `saved` (0 = fp32 FFMA,
 * 1 = bf16 tcgen05 trunk forward/backward with fp32 accumulation; heads, loss and Adam stay fp32). */
int64_t aq_gnn_backward_ws_floats(int64_t B);
int aq_gnn_backward(const float *params, const float *saved, const float *dpolicy, const float *dvalue, int64_t B,
                    float *grads, float *workspace, int precision, void *stream);

/* Loss of train_network.py:54-55,85-89: CrossEntropyLoss applied to the softmax OUTPUT (so a
 * second log_softmax; kept literally) + MSELoss, both 'mean' over B_total (= global batch under
 * data parallelism).  Writes loss[0] = policy loss sum over this shard / B_total, loss[1] = value
 * part, and the gradients dpolicy [B,209], dvalue [B]. */
int aq_loss_grad(const float *policy, const float *value, const float *policy_target, const float *value_target,
                 int64_t B, int64_t B_total, float *loss, float *dpolicy, float *dvalue, void *stream);

/* torch.optim.Adam step (train_network.py:56,94; default betas/eps, no weight decay) on the flat
 * buffers. step is the 1-based step count; lr already includes the LambdaLR factor. */
int aq_adam_step(float *params, const float *grads, float *exp_avg, float *exp_avg_sq, int64_t n, int64_t step,
                 float lr, float beta1, float beta2, float eps, float grad_scale, void *stream);

/* Data-parallel optimiser step without NCCL on the path (csrc/dp_comm.cu): one communicator per rank (process) of ONE box.
 *   aq_comm_create  allocates the rank's communication block and returns its 64-byte CUDA IPC handle in handle_out64;
 *   aq_comm_open    maps the other ranks' blocks: handles = world x 64 bytes, entry r from rank r (exchanged by the caller over any
 *                   host channel, e.g. torch.distributed.all_gather_object); not needed when world == 1;
 *   aq_comm_status  out2[0] = optimiser steps completed (device counter), out2[1] = 0 ok / 1 a peer did not arrive within the
 *                   kernel's time-out (the kernel gives up instead of hanging); synchronises `stream`;
 *   aq_comm_set_step sets the device step counter (0 for a fresh optimiser; every rank at the same point) and the running powers
 *                   beta^step the bias corrections are computed from.
 * aq_dp_adam_step: all-reduce (sum over the ranks) of the flat gradient `grads` + torch.optim.Adam step (train_network.py:56,94) in
 * ONE kernel over NVLink peer memory; `grads` holds the sum afterwards; every rank ends with bit-identical parameters.  The step
 * number of the bias corrections is the device counter + 1.  The replacement for torch.distributed.all_reduce + aq_adam_step. */
int aq_comm_create(int rank, int world, void **comm, void *handle_out64);
int aq_comm_open(void *comm, const void *handles);
int aq_comm_destroy(void *comm);
int aq_comm_status(void *comm, int64_t *out2, void *stream);
int aq_comm_set_step(void *comm, int64_t step, float beta1, float beta2, void *stream);
int aq_dp_adam_step(void *comm, float *params, float *grads, float *exp_avg, float *exp_avg_sq, float lr, float beta1, float beta2,
                    float eps, void *stream);
/* Everything of a training step behind the forward pass -- the reference's `loss = CE + MSE; zero_grad(); loss.backward();
 * optimizer.step()` (train_network.py:85-94) with the gradient all-reduce of data parallelism in between -- in four kernels:
 * loss gradient + heads backward, trunk backward, head weight gradients, and slot reduction + all-reduce + Adam (above).
 * saved / workspace / precision as in aq_gnn_forward / aq_gnn_backward; B_total = the global batch the 'mean' losses divide by;
 * loss (may be NULL) receives this rank's {policy, value} loss contributions; grads (may be NULL) the reduced gradient. */
int aq_train_backward_step(void *comm, float *params, const float *saved, const float *policy_target, const float *value_target,
                           int64_t B, int64_t B_total, float *loss, float *grads, float *exp_avg, float *exp_avg_sq, float *workspace,
                           int precision, float lr, float beta1, float beta2, float eps, void *stream);

/* Batched BaseNetwork.predict (BaseNetwork.py:36-40; behaviour pv_network_cnn.py:117-137):
 * legal mask + graph + forward + restriction to legal actions + renormalisation, for B leaves.
 *   priors [B,209]: p[a]/sum_legal p for legal a, 0 elsewhere (sum==0 -> left unnormalised, as
 *                   `policy /= sum if sum else 1`)
 *   value  [B], mask [B,8], pawn [B,8] as in aq_legal_mask. */
int aq_leaf_eval(const float *params, const void *prepared /* or NULL */, const AqState *states, int64_t B, float *priors,
                 float *value, uint32_t *mask, uint8_t *pawn, float *workspace /* aq_leaf_eval_ws_floats(B) */,
                 int precision, void *stream);
int64_t aq_leaf_eval_ws_floats(int64_t B);

/* Same through HOST buffers (pinned or pageable): copies states H2D, runs, copies priors/value/
 * mask/pawn D2H on `stream`, then synchronises the stream.  dev_ws is a device workspace of
 * aq_leaf_eval_host_ws_bytes(B) bytes. */
int64_t aq_leaf_eval_host_ws_bytes(int64_t B);
/* host_ctx (optional, may be NULL): context from aq_host_ctx_create; with it, batches >= 4096 are
 * processed in 2 chunks on two worker streams so that the D2H of the first overlaps the kernels of the second;
 * with pinned host buffers the whole pipeline is replayed as one cached CUDA graph per argument tuple. */
int aq_host_ctx_create(void **ctx);
int aq_host_ctx_destroy(void *ctx);
int aq_leaf_eval_host(const float *params, const void *prepared /* or NULL */, const AqState *states_host, int64_t B,
                      float *priors_host, float *value_host, uint32_t *mask_host, uint8_t *pawn_host, void *dev_ws,
                      int precision, void *host_ctx, void *stream);

/* predict()-shaped output (BaseNetwork.py:36-40, pv_network_cnn.py:128-135: the probabilities of the LEGAL actions
 * only, in state.legal_actions() order) for a batch, as a ragged array:
 *   offsets [B+1] int32 : offsets[b] = number of legal actions of boards < b, offsets[B] = total
 *   compact [total] f32 : board b owns compact[offsets[b] .. offsets[b+1]); capacity B*136 is always enough
 * priors/mask/pawn are the outputs of aq_leaf_eval (or aq_heads_forward + aq_legal_mask). */
int aq_compact_priors(const float *priors, const uint32_t *mask, const uint8_t *pawn, int64_t B, int32_t *offsets,
                      float *compact, void *stream);

/* aq_leaf_eval_host with predict()-shaped output (BaseNetwork.py:36-40, pv_network_cnn.py:128-135): H2D states, kernels, then
 * only the legal actions' probabilities travel back (4 or 2 bytes per legal action instead of 836 per board; the dense path is
 * PCIe-bound).
 *   priors_host  [priors_capacity] : ragged priors, board b at [offsets_host[b], offsets_host[b+1]); f32 (wire = AQ_WIRE_F32: the
 *                                    bits of the dense priors) or IEEE half (AQ_WIRE_F16: the same values rounded to nearest even,
 *                                    |error| <= 2^-12 relative; halves the device -> host bytes).  B*136 entries always suffice;
 *                                    AQ_ERR_ARG from _wait if the capacity is too small
 *   offsets_host [B+1] int32, value_host [B]; mask_host [B,8] / pawn_host [B,8] are optional (NULL: not copied -- predict() itself
 *                                    returns only (policy, value); callers that want the action ids without running
 *                                    legal_actions() on the host ask for them)
 * host_ctx is required (worker stream, events, and the running estimate that sizes the ragged copy -- see gnn_forward.cu).
 * dev_ws: aq_leaf_eval_host_compact_ws_bytes(B) bytes.
 * The call comes in two halves so that a host can keep several batches in flight (one host_ctx + dev_ws + set of host buffers per
 * batch, e.g. three pools of games evaluated round-robin): _submit enqueues the copies and kernels and returns immediately; _wait
 * returns when that context's results are on the host (one event wait; only this batch's own work is waited for, not other work
 * queued on `stream`).  One batch per context at a time.  aq_leaf_eval_host_compact = _submit + _wait. */
#define AQ_WIRE_F32 0
#define AQ_WIRE_F16 1
int aq_leaf_eval_host_compact_submit(const float *params, const void *prepared, const AqState *states_host, int64_t B,
                                     void *priors_host, int64_t priors_capacity, int32_t *offsets_host, float *value_host,
                                     uint32_t *mask_host, uint8_t *pawn_host, void *dev_ws, int precision, int wire,
                                     void *host_ctx, void *stream);
int aq_leaf_eval_host_compact_wait(void *host_ctx);
int64_t aq_leaf_eval_host_compact_ws_bytes(int64_t B);
/* Optional: host buffers laid out as ONE block -- value_host = (char *)offsets_host + out2[0], priors_host = (char *)offsets_host +
 * out2[1] -- are filled by a single device -> host copy per batch (the device keeps its results in the same layout). */
int aq_leaf_eval_host_compact_layout(int64_t B, int64_t *out2);
int aq_leaf_eval_host_compact(const float *params, const void *prepared /* or NULL */, const AqState *states_host, int64_t B,
                              void *priors_host, int64_t priors_capacity, int32_t *offsets_host, float *value_host,
                              uint32_t *mask_host, uint8_t *pawn_host, void *dev_ws, int precision, int wire, void *host_ctx,
                              void *stream);
/* Diagnostics of a host context: out2[0] = batches whose ragged priors needed a second copy (estimate too small),
 * out2[1] = current estimate of legal actions per board x 1024. */
int aq_host_ctx_stats(void *host_ctx, int64_t *out2);

/* Lock-step PV-MCTS over G independent games (pv_mcts.py:20-95: Node.evaluate / next_child_node).
 * ws: device workspace of aq_mcts_ws_bytes(G, max_nodes); max_nodes >= 1 + sims * 133 never overflows.
 * One simulation = aq_mcts_select -> aq_leaf_eval on leaf_states -> aq_mcts_expand_backup.
 *   leaf_kind[g]: 0 = leaf needs the network, 1 = terminal loss (value -1), 2 = terminal draw (0)
 *   aq_mcts_root_counts: visit counts / actions of the root's children in legal_actions() order
 *   (pv_mcts.py:88), n_children[g]; overflow[0] != 0 if any arena was exhausted. */
int64_t aq_mcts_ws_bytes(int64_t G, int64_t max_nodes);
int aq_mcts_reset(void *ws, const AqState *roots, int64_t G, int64_t max_nodes, void *stream);
/* Tree reuse between moves (AlphaGo Zero; the reference has none): destination game g continues the tree of source game
 * src_game[g] (-1 = fresh root).  Walk path[g, 0..path_len) from that game's root: path_len = 1 for the own move, 2 for the own
 * move and the opponent's reply.  If the node reached was visited (n >= 1) and its subtree has at most max_nodes - reserve_nodes
 * nodes, that subtree becomes game g's tree, with w, n, prior, child order and n_children bit-identical.  Otherwise game g starts
 * from a fresh root, exactly as aq_mcts_reset makes it.
 *   roots [G_dst]    the new root states (also used for fresh rows); for a carried row, state_after(src root, path) must
 *                    equal roots[g].  A mismatch, or src_game out of range, makes the row fresh and is counted in status[0]
 *   kept  [G_dst]    nodes carried, 0 = fresh (may be NULL)
 *   src_ws, dst_ws   workspaces laid out for G_src / G_dst games with the same max_nodes; they must not overlap
 * AQ_ERR_ARG for sizes < 1, path_len < 1, reserve_nodes outside [0, max_nodes) or overlapping workspaces. */
int aq_mcts_advance(const void *src_ws, int64_t G_src, void *dst_ws, int64_t G_dst, int64_t max_nodes, const AqState *roots,
                    const int64_t *src_game, const int16_t *path, int path_len, int64_t reserve_nodes, int32_t *kept,
                    int32_t *status, void *stream);
int aq_mcts_select(void *ws, int64_t G, int64_t max_nodes, float c_puct, AqState *leaf_states, int32_t *leaf_kind,
                   void *stream);
int aq_mcts_expand_backup(void *ws, int64_t G, int64_t max_nodes, const float *priors, const float *values,
                          const uint32_t *mask, const uint8_t *pawn, void *stream);
/* aq_mcts_expand_backup of one simulation followed by aq_mcts_select of the next in one launch (same results: a game's next
 * descent depends only on that game's own backup). */
int aq_mcts_expand_select(void *ws, int64_t G, int64_t max_nodes, const float *priors, const float *values, const uint32_t *mask,
                          const uint8_t *pawn, float c_puct, AqState *leaf_states, int32_t *leaf_kind, void *stream);
/* Gumbel root (Gumbel AlphaZero, Danihelka et al. 2022, as DeepMind's mctx gumbel_muzero_policy; the reference has none): the
 * root's children are sampled without replacement by Gumbel-top-k and the simulations spread over them by sequential halving; every
 * node below the root keeps PUCT.  A Gumbel search runs aq_mcts_reset, simulation 1, aq_mcts_gumbel_root, sims - 1 simulations with
 * aq_mcts_select_gumbel / aq_mcts_expand_select_gumbel in place of aq_mcts_select / aq_mcts_expand_select, then
 * aq_mcts_gumbel_result.
 * aq_mcts_gumbel_root gives every root that simulation 1 has expanded and nothing has visited since (root n == 1) and that has
 * no Gumbel state yet its state: per child c of the K children, base_c = float32(g_c + (log p_c - max log p)) with
 * g_c = gumbel_scale * (-log(-log U_c)), U_c in (0, 1) a counter-based draw (splitmix64, keyed by (seed, game_id[g], ply) with its
 * own domain constant: independent of the batch, the row and padding rows); v_hat = the root's value; m = min(considered, K);
 * n = sims - 1 root-child visits.  Calling it again is a no-op for a root that has its state.
 *   game_id [G] int64 (NULL: the row index); root_scores [G,136] f32 (may be NULL): base_c after the call, 0 beyond n_children.
 *   AQ_ERR_ARG for G < 1, a null ws, considered < 1, sims < 1, gumbel_scale < 0 or not finite.
 * The _gumbel select / expand-select leave a root with Gumbel state by the child with the largest max(-1e9, base_c + sigma_c)
 * among those with n_c == considered_visit(m, n, sum of the children's n): mctx's sequential-halving table; sigma_c is mctx's
 * completed-Q transform (mixed value of v_hat and the visited children's Q, min-max rescaled, times (50 + max n) * 0.1).
 * csrc/mcts.cu states the rule and its float64 rounding exactly.  Roots without Gumbel state, and all other nodes, use PUCT.
 * aq_mcts_gumbel_result: policy [G,136] f32 = softmax(log p_c + sigma_c) over the root's children (legal_actions() order, 0 beyond);
 * choice [G] int16 = the child with the largest score among the most visited ones.  Roots without Gumbel state: 0 and -1. */
int aq_mcts_gumbel_root(void *ws, int64_t G, int64_t max_nodes, const int64_t *game_id, uint64_t seed, int32_t ply, int32_t considered,
                        float gumbel_scale, int32_t sims, float *root_scores, void *stream);
int aq_mcts_select_gumbel(void *ws, int64_t G, int64_t max_nodes, float c_puct, AqState *leaf_states, int32_t *leaf_kind,
                          void *stream);
int aq_mcts_expand_select_gumbel(void *ws, int64_t G, int64_t max_nodes, const float *priors, const float *values, const uint32_t *mask,
                                 const uint8_t *pawn, float c_puct, AqState *leaf_states, int32_t *leaf_kind, void *stream);
int aq_mcts_gumbel_result(void *ws, int64_t G, int64_t max_nodes, float *policy /*[G,136]*/, int16_t *choice /*[G]*/, void *stream);
int aq_mcts_root_counts(void *ws, int64_t G, int64_t max_nodes, int32_t *counts /*[G,136]*/,
                        int16_t *actions /*[G,136]*/, int16_t *n_children /*[G]*/, int32_t *overflow, void *stream);
/* Root values of the last search of every game (fresh, carried, noised or Gumbel roots alike), all in double, one warp per game:
 *   root_value [G] = w_root / n_root, from the player to move at the root; NaN if n_root == 0
 *   best_child [G] = the root child with the largest visit count, the first in legal_actions() order on ties (the child that
 *                    temperature 0 plays); -1 without children
 *   best_q     [G] = -(w_b / n_b) of that child b, from the player to move at the root; -inf if n_b == 0 or there are no children
 * AQ_ERR_ARG for G < 1, max_nodes < 1 or a NULL pointer. */
int aq_mcts_root_values(void *ws, int64_t G, int64_t max_nodes, double *root_value /*[G]*/, double *best_q /*[G]*/, int16_t *best_child /*[G]*/,
                        void *stream);
/* Forced playouts and policy target pruning (KataGo: Wu 2019; the reference has neither).  A forced search runs
 * aq_mcts_select_forced / aq_mcts_expand_select_forced in place of aq_mcts_select / aq_mcts_expand_select and reads its counts with
 * aq_mcts_root_counts_pruned in place of aq_mcts_root_counts; both take forced_k >= 0 after c_puct.  With t = n_root - 1 (the sum of
 * the root children's n), P_c the stored prior (noised if the root was noised) and k = (double)forced_k:
 *   n_forced(c) = sqrt(k * P_c * t) in float64;  PUCT(c, m) = the select score with the visit count of U replaced by m
 * The forced select leaves the root (expanded, not terminal) by the first child in legal_actions() order with n_c >= 1 and
 * (double)n_c < n_forced(c), else by PUCT; every other node uses PUCT.  aq_mcts_root_counts_pruned writes what aq_mcts_root_counts
 * writes, except the counts: c* (the first child with the largest n) keeps n_c*; every other child with n_c >= 1 starts from
 * m = n_c and, while m >= 1, (double)(m - 1) >= (double)n_c - n_forced(c) and PUCT(c, m - 1) < PUCT(c*, n_c*), loses one; a child
 * that was reduced and ends with m <= 1 gets 0.  k = 0 is the plain search and the plain counts; the most visited child never
 * changes.  csrc/mcts.cu states the rounding exactly.  AQ_ERR_ARG as the plain entry points, and for forced_k < 0 or not finite. */
int aq_mcts_select_forced(void *ws, int64_t G, int64_t max_nodes, float c_puct, float forced_k, AqState *leaf_states, int32_t *leaf_kind,
                          void *stream);
int aq_mcts_expand_select_forced(void *ws, int64_t G, int64_t max_nodes, const float *priors, const float *values, const uint32_t *mask,
                                 const uint8_t *pawn, float c_puct, float forced_k, AqState *leaf_states, int32_t *leaf_kind, void *stream);
int aq_mcts_root_counts_pruned(void *ws, int64_t G, int64_t max_nodes, float c_puct, float forced_k, int32_t *counts /*[G,136]*/,
                               int16_t *actions /*[G,136]*/, int16_t *n_children /*[G]*/, int32_t *overflow, void *stream);
/* Dirichlet noise on the priors of every expanded, not yet noised root (AlphaZero; the reference has none).
 *   game_id [G] int64 (NULL: the row index), seed / ply: the key of the draw; alpha > 0, 0 <= fraction <= 1
 *   root_priors [G,136] f32 (may be NULL): the root's child priors after the call, legal_actions() order, 0 beyond n_children
 * A root is noised at most once between aq_mcts_reset / aq_mcts_advance and the next one; calling again is a no-op for it.
 * For game g with K = n_children root children, priors p_c in legal_actions() order:
 *   eta ~ Dirichlet(alpha, ..., alpha) over the K children, a pure function of (seed, game_id[g], ply, K, alpha): a counter-based
 *         draw (splitmix64, keyed like the move draw of aq_selfplay_advance with its own domain constant), independent of the
 *         other games of the batch, of the row and of padding rows.  Gamma variates: Marsaglia-Tsang with Box-Muller normals at
 *         shape alpha (alpha >= 1) or alpha + 1 boosted by u^(1/alpha) (alpha < 1), in logs, normalised with the maximum
 *         subtracted; csrc/mcts.cu documents the exact counter layout
 *   p'_c = float32((1 - fraction) * (double)p_c + fraction * eta_c), computed in double and rounded once (fraction 0: p'_c = p_c)
 * Callers noise a search's root once before its first descent that reads the root's children: right after aq_mcts_advance for a
 * carried root, right after simulation 1 (which expands it) for a fresh one; calling before and after simulation 1 does both.
 * The noised priors stay in the tree for the rest of the search.  AQ_ERR_ARG for G < 1, a null ws, alpha <= 0 or not finite,
 * fraction outside [0, 1] or NaN. */
int aq_mcts_root_noise(void *ws, int64_t G, int64_t max_nodes, const int64_t *game_id, uint64_t seed, int32_t ply,
                       float alpha, float fraction, float *root_priors, void *stream);

/* Prefix entry points (playout cap randomization searches a prefix of the batch): each runs the kernel of its plain entry point over
 * games [0, rows) of a workspace laid out for G games, 1 <= rows <= G; games [rows, G) are neither read nor written.  Every other
 * argument, and every per-game array (leaf_states, leaf_kind, priors, values, mask, pawn, game_id, root_priors), is that of the
 * plain entry point, indexed by the game's row.  AQ_ERR_ARG as the plain entry point, and for rows outside [1, G]. */
int aq_mcts_select_rows(void *ws, int64_t G, int64_t rows, int64_t max_nodes, float c_puct, AqState *leaf_states, int32_t *leaf_kind,
                        void *stream);
int aq_mcts_select_forced_rows(void *ws, int64_t G, int64_t rows, int64_t max_nodes, float c_puct, float forced_k, AqState *leaf_states,
                               int32_t *leaf_kind, void *stream);
int aq_mcts_expand_backup_rows(void *ws, int64_t G, int64_t rows, int64_t max_nodes, const float *priors, const float *values,
                               const uint32_t *mask, const uint8_t *pawn, void *stream);
int aq_mcts_expand_select_rows(void *ws, int64_t G, int64_t rows, int64_t max_nodes, const float *priors, const float *values,
                               const uint32_t *mask, const uint8_t *pawn, float c_puct, AqState *leaf_states, int32_t *leaf_kind, void *stream);
int aq_mcts_expand_select_forced_rows(void *ws, int64_t G, int64_t rows, int64_t max_nodes, const float *priors, const float *values,
                                      const uint32_t *mask, const uint8_t *pawn, float c_puct, float forced_k, AqState *leaf_states,
                                      int32_t *leaf_kind, void *stream);
int aq_mcts_root_noise_rows(void *ws, int64_t G, int64_t rows, int64_t max_nodes, const int64_t *game_id, uint64_t seed, int32_t ply,
                            float alpha, float fraction, float *root_priors, void *stream);

/* One ply of G lock-step self-play games after their searches (self_play.py:47-60), two launches:
 *   scores = counts ** (1 / temperature) / sum over the root's children (pv_mcts.py:88-95; temperature 0 = one-hot on
 *            the first maximum, np.argmax); policy[g, action] = score, 0 for the other of the 209 actions (self_play.py:51-54),
 *            float64 if policy_f64 else float32;
 *   action = one draw from scores (self_play.py:57, np.random.choice(legal_actions, p=scores)): inverse CDF in
 *            legal_actions() order of a uniform hashed from (seed, game_id[g], ply); chosen[g] (may be NULL);
 *   the games whose next state (self_play.py:60) is not terminal are written, in order, to next_states / next_game_id
 *   and counted in alive_count[0]; for the others final_flags[game_id] = is_lose | is_draw << 1 of the last state
 *   (game_logic.py:43-50) and final_plies[game_id] = ply + 1.
 * counts / actions / n_children as aq_mcts_root_counts returns them; workspace: aq_selfplay_ws_bytes(G) device bytes. */
int64_t aq_selfplay_ws_bytes(int64_t G);
int aq_selfplay_advance(const AqState *states, const int32_t *counts, const int16_t *actions, const int16_t *n_children,
                        const int64_t *game_id, int64_t G, double temperature, uint64_t seed, int32_t ply, void *policy,
                        int policy_f64, int16_t *chosen, AqState *next_states, int64_t *next_game_id, uint8_t *final_flags,
                        int64_t *final_plies, int32_t *alive_count, void *workspace, void *stream);
/* aq_selfplay_advance with the policy and the move from the search (a Gumbel root: aq_mcts_gumbel_result) instead of counts,
 * temperature and a draw: policy[g, actions[g, c]] = child_policy[g, c] for c < n_children[g], 0 for the other actions; the move is
 * child choice[g] (out of range: the game cannot move and ends as a draw).  Everything else as aq_selfplay_advance. */
int aq_selfplay_advance_chosen(const AqState *states, const float *child_policy /*[G,136]*/, const int16_t *choice /*[G]*/,
                               const int16_t *actions, const int16_t *n_children, const int64_t *game_id, int64_t G, int32_t ply,
                               void *policy, int policy_f64, int16_t *chosen, AqState *next_states, int64_t *next_game_id,
                               uint8_t *final_flags, int64_t *final_plies, int32_t *alive_count, void *workspace, void *stream);
/* Resignation (AlphaGo Zero, Silver et al. 2017; the reference has none): one ply as aq_selfplay_advance when counts is given (then
 * child_policy and choice are NULL), or as aq_selfplay_advance_chosen when child_policy and choice are (then counts is NULL), in which
 * a game may resign.  For game g, with s = max(root_value[g], best_q[g]) as aq_mcts_root_values returns them (NaN if either is):
 *   resign_min [num_games, 2] f64, indexed by game_id: resign_min[game_id[g], ply & 1] = min(itself, s) for every game at every
 *              ply (a NaN s leaves it); column 0 belongs to the first player, column 1 to the second.  The caller initialises it
 *              (+inf).
 *   calibration game: u < calibration with u = (mix64(mix64((seed ^ kResignDomain) + 0x9E3779B97F4A7C15 * (game_id + 1))) >> 11)
 *              * 2^-53 (splitmix64 finaliser, csrc/mcts.cu): a function of (seed, game id) alone, the same at every ply and
 *              independent of the move, noise and Gumbel draws.  Calibration games never resign; they are played to the end.
 *   is_calibration [num_games] u8, indexed by game_id: 1 for a calibration game, 0 otherwise, written for every game at every ply
 *              (the bit the kernel used).
 *   A game that is not a calibration game and has s < v_resign resigns: its policy row is written as without resignation, no
 *   move is played (chosen[g] = -1), and it leaves the batch with final_flags = 1 | 4 (bit 0: the player to move has lost, bit 2:
 *   resigned) and final_plies = ply, the moves played.  A resigned game therefore has final_plies + 1 recorded positions, a game
 *   that ends on the board final_plies; the value targets of both follow from bit 0 and final_plies alike.
 * Every other game gets exactly what aq_selfplay_advance / aq_selfplay_advance_chosen give it.  Two launches.
 * AQ_ERR_ARG as those entries, and for neither or both modes given, a NaN v_resign, calibration outside [0, 1] or a NULL
 * root_value, best_q, resign_min or is_calibration. */
int aq_selfplay_advance_resign(const AqState *states, const int32_t *counts, const float *child_policy, const int16_t *choice,
                               const int16_t *actions, const int16_t *n_children, const int64_t *game_id, int64_t G, double temperature,
                               uint64_t seed, int32_t ply, void *policy, int policy_f64, int16_t *chosen, const double *root_value,
                               const double *best_q, double v_resign, double calibration, double *resign_min /*[num_games,2]*/,
                               uint8_t *is_calibration /*[num_games]*/, AqState *next_states, int64_t *next_game_id, uint8_t *final_flags, int64_t *final_plies,
                               int32_t *alive_count, void *workspace, void *stream);

/* Playout cap randomization (KataGo: Wu 2019, section 3.1; the reference has none): which moves get a full search.  One launch, one
 * CTA.  Rows [0, n) with n = *count (device; NULL: G; clamped to [0, G]) are reordered stably: the full rows first, then the fast
 * rows, each kind in input order; out_states / out_game_id [n] take the reordered rows, out_row [n] int64 the input row of each
 * output row, full_count[0] the number of full rows.  Row i is full iff u < full_prob with
 *   u = (mix64(mix64((seed ^ kPcrDomain) + 0x9E3779B97F4A7C15 * (game_id[i] + 1)) + 0xD1B54A32D192ED03 * (ply + 1)) >> 11) * 2^-53,
 *   kPcrDomain = 0x082EFA98EC4E6C89 (csrc/mcts.cu)
 * a function of (seed, game id, ply) alone, independent of the move, noise, Gumbel and calibration draws; full_prob = 1 makes every
 * row full.  AQ_ERR_ARG for G outside [1, 2^31), full_prob outside [0, 1] or NaN, or a NULL pointer other than count. */
int aq_selfplay_partition(const AqState *states, const int64_t *game_id, int64_t G, const int32_t *count, uint64_t seed, int32_t ply,
                          double full_prob, AqState *out_states, int64_t *out_game_id, int64_t *out_row, int32_t *full_count, void *stream);

/* agents.heuristic_eval (agents.py:22-54) for B states: shortest pawn-path lengths to the goal row for the mover
 * and for the enemy (shortest_path_bfs, agents.py:27-41, with the jump rules of legal_actions_pos; -1 = no path).
 *   dist      [B,2] int16 : {mover, enemy}                                    (may be NULL)
 *   heuristic [B] float64 : (dist_enemy - dist_mover) / MAX_DIST_FROM_GOAL (= 116//2 - 10 = 48, agents.py:11)   (may be NULL)
 *   leaf48    [B] int32   : 48 x the depth-0 value of agents.alpha_beta (agents.py:69-75): is_lose -> -48,
 *                           is_draw -> 0, else dist_enemy - dist_mover                                          (may be NULL) */
int aq_shortest_paths(const AqState *states, int64_t B, int16_t *dist, double *heuristic, int32_t *leaf48, void *stream);

/* One level of the negamax recursion of agents.alpha_beta / alpha_beta_action (agents.py:58-107) over a batch of
 * parents: value[p] = max over children c in [child_offset[p], child_offset[p+1]) of -child_value[c];
 * best[p] = index (within the parent) of the FIRST child attaining it, -1 if none; parents with
 * fixed[p] != INT32_MIN keep fixed[p] (terminal nodes).  fixed and best may be NULL. */
int aq_negamax_backup(const int32_t *child_value, const int64_t *child_offset, int64_t P, const int32_t *fixed,
                      int32_t *value, int32_t *best, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* AQGNN_H */
