"""Policy-Value Monte Carlo Tree Search -- drop-in for reference pv_mcts.py, batched over games.

Same public names (PV_EVALUATE_COUNT, pv_mcts_policy, pv_mcts_action, boltzman).  The tree lives on
the GPU (csrc/mcts.cu): G games are searched in lock-step, so the leaf of every game at simulation k
forms one batch for the network (batched leaf evaluation = model.predict for G states at once,
pv_mcts.py:47).  The reference has no virtual loss, no Dirichlet noise and no tree reuse
(pv_mcts.py:81 builds a fresh root per move), so each game's search is exactly the reference's.
Tree reuse between moves (AlphaGo Zero: the child of the played move becomes the next root with its
statistics) is opt-in, BatchedMCTS(..., tree_reuse=True); the default keeps the reference's fresh root.
Dirichlet noise on the root priors (AlphaZero self-play exploration) is opt-in too,
BatchedMCTS(..., dirichlet_alpha=0.3); the default searches with the network's priors.
So is the Gumbel root of Gumbel AlphaZero, BatchedMCTS(..., gumbel_considered=16): sequential halving over Gumbel-top-k sampled
root children and a completed-Q improved policy; the default keeps PUCT at the root.
Forced playouts with policy target pruning (KataGo), BatchedMCTS(..., forced_k=2.0), give every visited root child at least
sqrt(k * P * sum N) visits and take the surplus back out of the counts the search returns; the default returns the plain counts.
Playout cap randomization (KataGo), search(..., fast_sims=50, full_rows=F), gives rows [0, F) the full search and the others a
cheap one of fast_sims simulations without root noise; the default gives every row the full search.
"""
import math
from copy import deepcopy

import numpy as np
import torch

from . import _lib
from . import game_logic as gl

# Prepare parameters
PV_EVALUATE_COUNT = 50  # Number of simulations per inference (pv_mcts.py:18)
C_PUCT = 1.25           # pv_mcts.py:71
MAX_CHILDREN = 133      # 5 pawn moves + 128 wall placements
GRAPH_CHUNK = 25        # simulations per launch of the chunk graph (BatchedMCTS.search)


def _padded(n):
    """Batch size a search of n rows runs at when it pads (network evaluator, graphs on, n > 256): the next multiple of 256."""
    return n if n <= 256 or n % 256 == 0 else n + 256 - n % 256


def network_evaluator(model):
    """Evaluator protocol: packed states uint8[G,32] -> dict(priors f32[G,209] (legal-masked,
    renormalised), value f32[G], mask int32[G,8], pawn uint8[G,8])."""
    return lambda packed: model.predict_batch(packed)


class BatchedMCTS:
    """Lock-step PV-MCTS over G independent root states.

    `evaluator` is either a GNNNetwork (leaf evaluation = aq_leaf_eval into preallocated buffers; the simulation
    step -- select, legal mask, GNN trunk, heads, expand+backup -- is captured in CUDA graphs of GRAPH_CHUNK steps
    and of one step, and a search replays those) or any callable following the evaluator protocol (eager loop).

    tree_reuse=True (AlphaGo Zero; the reference has none): a search may continue the tree of the previous one
    (search(..., src_row, path)).  `sims` is then required: each game's arena holds 1 + 2 * sims * MAX_CHILDREN nodes, room
    for one carried search and one new one, and two workspaces are used in turn (the previous search's tree is read from one
    while the next is built in the other).

    dirichlet_alpha (AlphaZero; the reference has none): each search mixes eta ~ Dirichlet(dirichlet_alpha) into its root's child
    priors, p' = (1 - noise_fraction) * p + noise_fraction * eta (aq_mcts_root_noise), once, before the first descent that reads
    them: a carried root right after it is carried, a fresh root right after simulation 1 expands it.  The draw is keyed by
    search(..., noise_seed, game_id, ply).  None (the default) runs exactly the search without noise.

    gumbel_considered (Gumbel AlphaZero, Danihelka et al. 2022, as mctx's gumbel_muzero_policy; the reference has none): the root
    samples min(gumbel_considered, K) of its K children without replacement (Gumbel-top-k, Gumbel noise scaled by gumbel_scale) and
    spreads the search's sims - 1 root-child visits over them by sequential halving; every node below the root keeps PUCT.  After
    the search, last_policy f32[G,136] holds the improved policy softmax(logits + sigma(completed Q)) over the root's children and
    last_choice int16[G] the child to play (aq_mcts_gumbel_root / _result, csrc/mcts.cu).  The draw is keyed by search(...,
    noise_seed, game_id, ply).  It cannot be combined with tree_reuse (the schedule starts from a root without child visits) or with
    dirichlet_alpha (the Gumbel draw is the root's exploration).  None (the default) runs exactly the PUCT search.

    forced_k (forced playouts and policy target pruning, KataGo: Wu 2019; the reference has none): the root's descent takes the
    first child in legal_actions() order that has been visited but has fewer than n_forced = sqrt(forced_k * P * t) visits (P its
    prior, noised if the root was, t the sum of the root children's visits), else the PUCT arg-max; every node below the root keeps
    PUCT (aq_mcts_select_forced).  The counts a search returns are then pruned (aq_mcts_root_counts_pruned): every child but the
    most visited one loses the visits, up to n_forced, that PUCT would not have given it against that child, and a child left with
    one visit goes to 0.  The most visited child keeps its count, so temperature 0 and root_values() see the same move.  It pairs
    with dirichlet_alpha (the forced visits then explore the noise without training on it) and tree_reuse (carried visits count in
    t), not with gumbel_considered.  forced_k=0 is the plain search; None (the default) runs exactly it.

    search(..., fast_sims, full_rows) (playout cap randomization, KataGo: Wu 2019, section 3.1; the reference has none): rows
    [0, full_rows) get the full search of `sims` new simulations with the configured root noise, and the other rows a fast search of
    fast_sims new simulations without root noise; a fast row's result is exactly that of this searcher's search with
    dirichlet_alpha=None and fast_sims simulations.  Fast rows keep the select rule and the counts of the searcher: with forced_k they
    force root playouts and return pruned counts too (KataGo turns forced playouts off for its cheap searches; here one select rule
    serves every row of a launch, and without noise the rule finds little to force).  Every tree is started (reset or advance), the
    full rows' roots are noised before and after simulation 1, then phase A runs fast_sims simulations on every row and phase B the
    other sims - fast_sims on the full rows alone, through the prefix entry points (aq_mcts_*_rows); the counts are read for every
    row.  When the search pads (network evaluator, graphs, more than 256 rows), its rows are laid out as [full rows | copies of the
    last full root up to the padded size of the full-row count | fast rows | padding], so that phase B is replayed from graphs
    captured for a few sizes; outputs, last_kept and root_values() are in the caller's order all the same.  It cannot be combined
    with gumbel_considered, whose schedule depends on the budget."""

    def __init__(self, evaluator, sims=None, c_puct=C_PUCT, device=None, use_graph=True, tree_reuse=False, dirichlet_alpha=None,
                 noise_fraction=0.25, gumbel_considered=None, gumbel_scale=1.0, forced_k=None):
        if tree_reuse and not sims:
            raise ValueError("BatchedMCTS(tree_reuse=True) needs `sims` at construction: it sizes the node arena")
        if dirichlet_alpha is not None and not (math.isfinite(dirichlet_alpha) and dirichlet_alpha > 0):
            raise ValueError(f"dirichlet_alpha must be a finite number > 0 (or None), not {dirichlet_alpha!r}")
        if not 0.0 <= noise_fraction <= 1.0:
            raise ValueError(f"noise_fraction must be in [0, 1], not {noise_fraction!r}")
        if gumbel_considered is not None:
            if isinstance(gumbel_considered, bool) or int(gumbel_considered) != gumbel_considered or gumbel_considered < 1:
                raise ValueError(f"gumbel_considered must be an integer >= 1 (or None), not {gumbel_considered!r}")
            if not (math.isfinite(gumbel_scale) and gumbel_scale >= 0):
                raise ValueError(f"gumbel_scale must be a finite number >= 0, not {gumbel_scale!r}")
            if tree_reuse:
                raise ValueError("gumbel_considered cannot be combined with tree_reuse: the Gumbel schedule starts from a root without "
                                 "child visits")
            if dirichlet_alpha is not None:
                raise ValueError("gumbel_considered cannot be combined with dirichlet_alpha: the Gumbel draw is the root's exploration")
            if forced_k is not None:
                raise ValueError("gumbel_considered cannot be combined with forced_k: the Gumbel schedule sets the root's visits")
        if forced_k is not None and (isinstance(forced_k, bool) or not (math.isfinite(forced_k) and forced_k >= 0)):
            raise ValueError(f"forced_k must be a finite number >= 0 (or None), not {forced_k!r}")
        self.model = evaluator if hasattr(evaluator, "flat_parameters") else None
        self.evaluator = network_evaluator(evaluator) if hasattr(evaluator, "predict_batch") else evaluator
        self.sims = sims
        self.c_puct = float(c_puct)
        self.device = gl._dev(device)
        self.use_graph = use_graph
        self.tree_reuse = bool(tree_reuse)
        self.dirichlet_alpha = None if dirichlet_alpha is None else float(dirichlet_alpha)
        self.noise_fraction = float(noise_fraction)
        self.gumbel_considered = None if gumbel_considered is None else int(gumbel_considered)
        self.gumbel_scale = float(gumbel_scale)
        self.forced_k = None if forced_k is None else float(forced_k)
        self._mode = "puct" if self.forced_k is None else "forced"   # step mode of the simulations (a Gumbel search: of its first)
        self.last_policy = None  # gumbel_considered: f32[G,136] improved policy of the last search, else None
        self.last_choice = None  # gumbel_considered: int16[G] child chosen by the last search, else None
        self._ws = [None, None] if self.tree_reuse else [None]
        self._last = None     # tree_reuse: (workspace slot, G) of the previous search, the source a next search can continue
        self._last_rows = None  # tree_reuse: the workspace row of each caller row of the previous search when it is not that row
        self.last_kept = None  # tree_reuse: int32[G] nodes carried into each row by the last search (0 = fresh root), else None
        self._root = None      # (workspace, G, real rows, max_nodes) of the last search: what root_values() reads
        self._root_rows = None  # the workspace row of each caller row of the last search when it is not that row (None: row r is row r)
        self._buf = {}
        self._graphs = {}
        self._warm = set()   # step modes (the last item of a graph key: "puct", "gumbel" or "forced") whose lazy initialisation an
                             # eager step has done

    def _workspace(self, G, max_nodes, slot=0):
        L = _lib.load()
        need = L.aq_mcts_ws_bytes(G, max_nodes)
        if self._ws[slot] is None or self._ws[slot].numel() < need:
            self._ws[slot] = torch.empty((need,), dtype=torch.uint8, device=self.device)
            self._graphs.clear()  # graphs hold raw pointers into the old workspace
        return self._ws[slot]

    def _buffers(self, G):
        if G not in self._buf:
            dev = self.device
            if len(self._buf) >= 16:  # self-play shrinks G almost every ply: bound the cache; the captured graphs hold raw
                self._buf.clear()     # pointers into these buffers, so both caches are dropped together
                self._graphs.clear()
            self._buf[G] = {
                "leaf": torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device=dev),
                "kind": torch.empty((G,), dtype=torch.int32, device=dev),
                "priors": torch.empty((G, gl.NUM_ACTIONS), dtype=torch.float32, device=dev),
                "value": torch.empty((G,), dtype=torch.float32, device=dev),
                "mask": torch.empty((G, 8), dtype=torch.int32, device=dev),
                "pawn": torch.empty((G, 8), dtype=torch.uint8, device=dev),
                "pooled": torch.empty((max(1, _lib.load().aq_leaf_eval_ws_floats(G)),), dtype=torch.float32, device=dev),  # leaf-eval workspace
            }
        return self._buf[G]

    def _step(self, ws, G, max_nodes, buf, evaluate, st, steps=1, gumbel=False, forced=False, rows=None):
        """`steps` simulations for all games: select, then `steps` leaf evaluations out = evaluate(stream) (terminal leaves are
        evaluated too and ignored by the backup) joined by the fused expand + backup + next select, then the last expand + backup.
        gumbel: the selects leave a Gumbel root by the Gumbel rule; forced: the root by the forced-playout rule (forced_k).
        rows: the simulations run for games [0, rows) only, through the prefix entry points (aq_mcts_*_rows)."""
        L, P = _lib.load(), _lib.ptr
        if forced:
            k = (self.forced_k,)
            select, expand_select = ((L.aq_mcts_select_forced, L.aq_mcts_expand_select_forced) if rows is None else
                                     (L.aq_mcts_select_forced_rows, L.aq_mcts_expand_select_forced_rows))
        else:
            k = ()
            select, expand_select = ((L.aq_mcts_select_gumbel, L.aq_mcts_expand_select_gumbel) if gumbel else
                                     (L.aq_mcts_select, L.aq_mcts_expand_select) if rows is None else
                                     (L.aq_mcts_select_rows, L.aq_mcts_expand_select_rows))
        expand_backup = L.aq_mcts_expand_backup if rows is None else L.aq_mcts_expand_backup_rows
        dims = (G,) if rows is None else (G, rows)
        _lib.check(select(P(ws), *dims, max_nodes, self.c_puct, *k, P(buf["leaf"]), P(buf["kind"]), st), "aq_mcts_select")
        for i in range(steps):
            out = evaluate(st)
            leaves = (P(ws), *dims, max_nodes, P(out["priors"]), P(out["value"]), P(out["mask"]), P(out["pawn"]))
            if i + 1 < steps:
                _lib.check(expand_select(*leaves, self.c_puct, *k, P(buf["leaf"]), P(buf["kind"]), st), "aq_mcts_expand_select")
            else:
                _lib.check(expand_backup(*leaves, st), "aq_mcts_expand_backup")

    def _simulate(self, n, step, key, st):
        """n simulations; step(stream, k) enqueues k of them.  With a graph key (network evaluator) and use_graph, they are replays of
        CUDA graphs captured for the key; else one eager step per simulation."""
        if self.use_graph and key is not None:
            if key[-1] not in self._warm and n:
                # the searcher's first step of a mode runs outside capture: lazy initialisation (module load, function attributes)
                # must not happen inside one; a failure here is a real error and propagates
                step(st, 1)
                n = n - 1
                self._warm.add(key[-1])
                torch.cuda.synchronize(self.device)
            graphs = self._graphs.get(key)
            if graphs is None:
                if len(self._graphs) >= 32:
                    self._graphs.clear()
                graphs = self._graphs[key] = {}
            # GRAPH_CHUNK simulations back to back in one graph (+ a one-step graph for the remainder, captured only when there is
            # one): a search is a handful of graph launches instead of one per simulation -- a launch costs the host 10-100 us
            # depending on the box, the step 75 us of GPU time at 4,096 games
            for k in ((GRAPH_CHUNK,) if n >= GRAPH_CHUNK else ()) + ((1,) if n % GRAPH_CHUNK else ()):
                if k not in graphs:
                    graphs[k] = _lib.capture_graph(self.device, lambda cst: step(cst, k), "the MCTS simulation step")
                    if graphs[k] is None:
                        self.use_graph = False
                        self._graphs.clear()
                        break
            if self.use_graph:
                for _ in range(n // GRAPH_CHUNK):
                    graphs[GRAPH_CHUNK].replay()
                for _ in range(n % GRAPH_CHUNK):
                    graphs[1].replay()
                return
        for _ in range(n):
            step(st, 1)

    @torch.no_grad()
    def search_async(self, roots, sims=None, src_row=None, path=None, noise_seed=None, game_id=None, ply=0, fast_sims=None, full_rows=None):
        """search() without the synchronisation: returns (counts, actions, n_children, status int32[3] on the device); the caller
        passes status.tolist() to check_status() when it synchronises anyway."""
        sims = sims or self.sims or PV_EVALUATE_COUNT
        L, P = _lib.load(), _lib.ptr
        dev = self.device
        roots = roots.to(dev).contiguous()
        G_real = roots.shape[0]
        if src_row is not None:
            if not self.tree_reuse:
                raise ValueError("search(src_row=...) continues a tree: construct the searcher with tree_reuse=True")
            if self._last is None:
                raise ValueError("search(src_row=...) needs a previous search of this searcher to continue")
            if path is None:
                raise ValueError("search(src_row=...) needs the path of actions from each source root")
        if self.tree_reuse and sims > self.sims:
            raise ValueError(f"this searcher's node arena holds {self.sims} simulations per search, not {sims}")
        pcr = fast_sims is not None
        if pcr:
            if isinstance(fast_sims, bool) or int(fast_sims) != fast_sims or not 1 <= fast_sims <= sims:
                raise ValueError(f"fast_sims must be an integer in [1, sims = {sims}] (or None), not {fast_sims!r}")
            if self.gumbel_considered is not None:
                raise ValueError("fast_sims cannot be combined with gumbel_considered: the Gumbel schedule depends on the budget")
            full = G_real if full_rows is None else full_rows
            if isinstance(full, bool) or int(full) != full or not 0 <= full <= G_real:
                raise ValueError(f"full_rows must be an integer in [0, {G_real}] (or None), not {full_rows!r}")
            fast_sims, full = int(fast_sims), int(full)
        elif full_rows is not None:
            raise ValueError("search(full_rows=...) splits full and fast searches: it needs fast_sims")
        if G_real == 0:
            self.last_kept = self.last_policy = self.last_choice = None
            self._root, self._root_rows = (None, 0, 0, 0), None
            return (torch.empty((0, gl.MAX_LEGAL), dtype=torch.int32, device=dev), torch.empty((0, gl.MAX_LEGAL), dtype=torch.int16, device=dev),
                    torch.empty((0,), dtype=torch.int16, device=dev), torch.zeros((3,), dtype=torch.int32, device=dev))
        # Self-play and the arena drop finished games, so the number of roots shrinks by a few almost every ply.  Batches above 256
        # are padded to the next multiple of 256 with copies of the last root (searched and discarded; games are independent, so the
        # real ones are unaffected): workspaces, buffers and the captured CUDA graph of the simulation step are then reused across
        # plies instead of being rebuilt for every distinct size.
        rows = None   # the workspace row of each caller row, when it is not that row
        pads = self.model is not None and self.use_graph and G_real > 256
        if pcr and pads:
            # [full rows | copies of the last full root up to _padded(full) | fast rows | copies of the last root up to a multiple of
            # 256]: the full-row prefix that phase B searches has a padded size too, so its graphs are reused across plies as well
            full_pad = _padded(full)
            G = _padded(full_pad + G_real - full)
            if G > G_real:
                rows = torch.cat([torch.arange(full, device=dev), torch.arange(full_pad, full_pad + G_real - full, device=dev)])
                src = torch.full((G,), G_real - 1, dtype=torch.int64, device=dev)
                src[:full_pad] = full - 1
                src[rows] = torch.arange(G_real, device=dev)
                roots = roots[src].contiguous()
            full = full_pad
        elif pads and G_real % 256:
            roots = torch.cat([roots, roots[-1:].expand(256 - G_real % 256, -1)]).contiguous()
        G = roots.shape[0]

        def pad(t, fill):   # a per-game argument for the padded rows: they start fresh (src_row -1) and draw the noise of game 0
            if rows is not None:
                out = t.new_full((G,) + t.shape[1:], fill)
                out[rows] = t
                return out
            return (torch.cat([t, t.new_full((G - G_real,) + t.shape[1:], fill)]) if G > G_real else t).contiguous()

        def real(t):        # the caller's rows of a per-game output
            return t[:G_real] if rows is None else t[rows]

        max_nodes = 1 + (2 * self.sims if self.tree_reuse else sims) * MAX_CHILDREN
        slot = 0 if self._last is None else 1 - self._last[0]
        ws = self._workspace(G, max_nodes, slot)
        buf = self._buffers(G)
        # [arena overflow, NaN leaf value, inconsistent tree-reuse rows]
        status = torch.zeros((3,), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            st = _lib.stream_ptr(dev)
            if src_row is not None:
                src_slot, G_src = self._last
                src = src_row.to(device=dev, dtype=torch.int64).reshape(G_real)
                if self._last_rows is not None:   # caller rows of the previous search -> its workspace rows (out of range stays so)
                    n_prev = self._last_rows.shape[0]
                    src = torch.where(src < 0, src, torch.where(src < n_prev, self._last_rows[src.clamp(0, n_prev - 1)], src - n_prev + G_src))
                src = pad(src, -1)
                path = pad(path.to(device=dev, dtype=torch.int16).reshape(G_real, -1), 0)
                kept = torch.empty((G,), dtype=torch.int32, device=dev)
                _lib.check(L.aq_mcts_advance(P(self._ws[src_slot]), G_src, P(ws), G, max_nodes, P(roots), P(src), P(path), path.shape[1],
                                             sims * MAX_CHILDREN, P(kept), P(status[2:]), st), "aq_mcts_advance")
                self.last_kept = real(kept)
            else:
                _lib.check(L.aq_mcts_reset(P(ws), P(roots), G, max_nodes, st), "aq_mcts_reset")
                self.last_kept = None
            if self.tree_reuse:
                self._last, self._last_rows = (slot, G), rows
            if self.model is not None:
                from .pv_network_gnn import PRECISIONS
                flat = self.model.flat_parameters()
                prec = PRECISIONS[self.model.precision]
                # bf16 operand tiles, refreshed in place if the parameters changed since the last search
                prep = self.model.prepared_weights() if prec == 1 else None
                key = (G, max_nodes, ws.data_ptr(), flat.data_ptr(), prep.data_ptr() if prep is not None else 0, prec, self._mode)

                def evaluate_rows(n):
                    def evaluate(s):
                        _lib.check(L.aq_leaf_eval(P(flat), P(prep), P(buf["leaf"]), n, P(buf["priors"]), P(buf["value"]), P(buf["mask"]),
                                                  P(buf["pawn"]), P(buf["pooled"]), prec, s), "aq_leaf_eval")
                        return buf
                    return evaluate
                evaluate = evaluate_rows(G)
            else:
                key, evaluate = None, lambda s: self.evaluator(buf["leaf"])
            step = lambda s, k: self._step(ws, G, max_nodes, buf, evaluate, s, k, forced=self.forced_k is not None)
            if self.dirichlet_alpha is not None or self.gumbel_considered is not None:
                seed = (int(torch.randint(0, 2 ** 63 - 1, (1,)).item()) if noise_seed is None else int(noise_seed)) & (2 ** 64 - 1)
                gid = None if game_id is None else pad(game_id.to(device=dev, dtype=torch.int64).reshape(G_real), 0)
            self.last_policy = self.last_choice = None
            if pcr:
                # Phase A: fast_sims simulations of every row; phase B: sims - fast_sims more of the full rows [0, full) alone.  Only the
                # full rows are noised, at the same two points as a search without playout cap randomization.
                for n in ((1, fast_sims - 1) if self.dirichlet_alpha is not None else (fast_sims,)):
                    if self.dirichlet_alpha is not None and full:
                        _lib.check(L.aq_mcts_root_noise_rows(P(ws), G, full, max_nodes, P(gid), seed, int(ply), self.dirichlet_alpha,
                                                             self.noise_fraction, None, st), "aq_mcts_root_noise_rows")
                    self._simulate(n, step, key, st)
                if full and sims > fast_sims:
                    evaluate_b = evaluate_rows(full) if self.model is not None else lambda s: self.evaluator(buf["leaf"][:full])
                    step_b = lambda s, k: self._step(ws, G, max_nodes, buf, evaluate_b, s, k, forced=self.forced_k is not None, rows=full)
                    self._simulate(sims - fast_sims, step_b, None if key is None else key[:-1] + (full, self._mode + "-rows"), st)
            elif self.gumbel_considered is not None:
                # simulation 1 expands the root, aq_mcts_gumbel_root draws its Gumbel state, the other sims - 1 descend by its rule
                self._simulate(1, step, key, st)
                _lib.check(L.aq_mcts_gumbel_root(P(ws), G, max_nodes, P(gid), seed, int(ply), self.gumbel_considered, self.gumbel_scale,
                                                 sims, None, st), "aq_mcts_gumbel_root")
                gstep = lambda s, k: self._step(ws, G, max_nodes, buf, evaluate, s, k, gumbel=True)
                self._simulate(sims - 1, gstep, None if key is None else key[:-1] + ("gumbel",), st)
                policy = torch.empty((G, gl.MAX_LEGAL), dtype=torch.float32, device=dev)
                choice = torch.empty((G,), dtype=torch.int16, device=dev)
                _lib.check(L.aq_mcts_gumbel_result(P(ws), G, max_nodes, P(policy), P(choice), st), "aq_mcts_gumbel_result")
                self.last_policy, self.last_choice = policy[:G_real], choice[:G_real]
            elif self.dirichlet_alpha is None:
                self._simulate(sims, step, key, st)
            else:
                # aq_mcts_root_noise skips a root that is unexpanded or noised already, so noising before and after simulation 1 is the
                # whole rule: the first call noises a carried root, the second a fresh root, which simulation 1 expanded
                for n in (1, sims - 1):
                    _lib.check(L.aq_mcts_root_noise(P(ws), G, max_nodes, P(gid), seed, int(ply), self.dirichlet_alpha, self.noise_fraction,
                                                    None, st), "aq_mcts_root_noise")
                    self._simulate(n, step, key, st)
            counts = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int32, device=dev)
            actions = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int16, device=dev)
            n = torch.empty((G,), dtype=torch.int16, device=dev)
            if self.forced_k is None:
                _lib.check(L.aq_mcts_root_counts(P(ws), G, max_nodes, P(counts), P(actions), P(n), P(status[:1]), st),
                           "aq_mcts_root_counts")
            else:
                _lib.check(L.aq_mcts_root_counts_pruned(P(ws), G, max_nodes, self.c_puct, self.forced_k, P(counts), P(actions), P(n),
                                                        P(status[:1]), st), "aq_mcts_root_counts_pruned")
            if self.model is not None:
                status[1:2].copy_(torch.isnan(buf["value"]).any().reshape(1))
        self._root, self._root_rows = (ws, G, G_real, max_nodes), rows
        return real(counts), real(actions), real(n), status

    @torch.no_grad()
    def root_values(self):
        """The search's evaluation of each root of the last search, on the device and without a synchronisation (aq_mcts_root_values):
        (root_value float64[G], best_q float64[G]), both from the player to move at the root.  root_value = w / n of the root (NaN
        if it has no visit); best_q = -(w / n) of its most visited child, the first in legal_actions() order on ties (the move
        temperature 0 plays), -inf if that child has no visit or the root no children.  With tree_reuse the carried visits count."""
        if self._root is None:
            raise ValueError("root_values() reads the last search of this searcher: run a search first")
        ws, G, G_real, max_nodes = self._root
        dev = self.device
        root_value = torch.empty((G,), dtype=torch.float64, device=dev)
        best_q = torch.empty((G,), dtype=torch.float64, device=dev)
        if G:
            best_child = torch.empty((G,), dtype=torch.int16, device=dev)
            P = _lib.ptr
            with torch.cuda.device(dev):
                _lib.check(_lib.load().aq_mcts_root_values(P(ws), G, max_nodes, P(root_value), P(best_q), P(best_child), _lib.stream_ptr(dev)),
                           "aq_mcts_root_values")
        if self._root_rows is not None:
            return root_value[self._root_rows], best_q[self._root_rows]
        return root_value[:G_real], best_q[:G_real]

    @staticmethod
    def check_status(status):
        """status: the three flags search_async returns, as host integers."""
        if status[0]:
            raise _lib.AqError("MCTS node arena overflow")
        if status[2]:
            raise _lib.AqError(f"tree reuse: {status[2]} row(s) named a source game out of range or a root that is not the position "
                               "the path leads to from the source root")
        if status[1]:
            raise _lib.AqError("the network returned NaN for a leaf: with precision 'bf16' that is how an activation beyond the fp16 range of the "
                               "aggregation operand is reported (gnn_tc2.cu); evaluate this network with precision 'fp32'")

    def search(self, roots, sims=None, src_row=None, path=None, noise_seed=None, game_id=None, ply=0, fast_sims=None, full_rows=None):
        """roots: packed uint8[G,32] (non-terminal states).  Runs `sims` simulations per game
        (pv_mcts.py:84) and returns (counts int32[G,136], actions int16[G,136], n_children int16[G]):
        visit counts of the root's children in State.legal_actions() order (pv_mcts.py:88).

        With tree_reuse, src_row int64[G] (row of the previous search, -1 = fresh root) and path int16[G, k] (k = 1: the move
        played from that row's root; 2: and the reply) continue the previous search's trees: row g keeps the subtree below the
        path's end when that node was visited and its subtree leaves room for `sims` more simulations, else it starts fresh.
        The counts then include the carried visits; last_kept gives the nodes carried per row.

        With dirichlet_alpha, the root noise of row g is drawn from (noise_seed, game_id[g], ply): game_id int64[G] (None = the row
        index) names the game, so a game's noise does not depend on the other rows; noise_seed None draws one from torch's generator.

        With forced_k, the counts are the pruned counts (aq_mcts_root_counts_pruned); the tree keeps the visits it made.

        With fast_sims (playout cap randomization), rows [0, full_rows) (None: all) get the full search above and the other rows a
        fast one: exactly the search of this searcher with dirichlet_alpha=None and fast_sims simulations.  See the class docstring."""
        counts, actions, n, status = self.search_async(roots, sims, src_row, path, noise_seed, game_id, ply, fast_sims, full_rows)
        self.check_status(status.tolist())   # one synchronisation for both flags
        return counts, actions, n


class _SearcherCache(dict):
    """The searchers kept on a network object.  A copy or a pickle of the network starts with none: node arenas, captured graphs and
    raw pointers belong to the object they were made for."""

    def __deepcopy__(self, memo):
        return _SearcherCache()

    def __reduce__(self):
        return (_SearcherCache, ())


def searcher_for(evaluator, sims, device=None, tree_reuse=False, dirichlet_alpha=None, noise_fraction=0.25, gumbel_considered=None,
                 gumbel_scale=1.0, forced_k=None):
    """The BatchedMCTS of a network for `sims` simulations, kept on the network object: its node arenas (3.5 GB at 4,096 games x
    200 simulations), leaf buffers and captured graphs are reused by every later self-play / arena / policy call on that network
    instead of being allocated and captured again.  Evaluators that are plain callables get a fresh searcher."""
    dev = gl._dev(device)
    opts = dict(tree_reuse=tree_reuse, dirichlet_alpha=dirichlet_alpha, noise_fraction=noise_fraction, gumbel_considered=gumbel_considered,
                gumbel_scale=gumbel_scale, forced_k=forced_k)
    if not hasattr(evaluator, "flat_parameters"):
        return BatchedMCTS(evaluator, sims, device=dev, **opts)
    cache = evaluator.__dict__.setdefault("_searchers", _SearcherCache())
    key = (int(sims), str(dev), bool(tree_reuse), None if dirichlet_alpha is None else float(dirichlet_alpha),
           None if dirichlet_alpha is None else float(noise_fraction), None if gumbel_considered is None else int(gumbel_considered),
           None if gumbel_considered is None else float(gumbel_scale), None if forced_k is None else float(forced_k))
    if key not in cache:
        if len(cache) >= 4:
            cache.clear()
        cache[key] = BatchedMCTS(evaluator, sims, device=dev, **opts)
    return cache[key]


def policy_from_counts(counts, temperature):
    """pv_mcts.py:88-95 for a batch: counts [G,136] -> float64 probabilities [G,136] (0 beyond the
    root's children)."""
    c = counts.to(torch.float64)
    if temperature == 0:  # most-visited child, first maximum (np.argmax)
        pol = torch.zeros_like(c)
        pol[torch.arange(c.shape[0], device=c.device), torch.argmax(counts, dim=1)] = 1.0
        return pol
    x = c ** (1.0 / temperature)
    return x / x.sum(dim=1, keepdim=True)


def pv_mcts_policy_batch(model, packed_roots, temperature, sims=None, device=None):
    """Batched pv_mcts_policy: -> (policy float64[G,136], actions int16[G,136], n_children int16[G])."""
    mcts = searcher_for(model, sims or PV_EVALUATE_COUNT, device)
    counts, actions, n = mcts.search(packed_roots)
    return policy_from_counts(counts, temperature), actions, n


def pv_mcts_policy(model, state, temperature, device=None):
    """Use PUCT-based Monte Carlo Tree Search to return an improved policy (distribution over legal
    actions), compared to the prior policy provided by the neural network (pv_mcts.py:20-95)."""
    rows, plies = gl.rows_from_states([state])
    packed = gl.pack_rows(rows, plies, device)
    pol, _, n = pv_mcts_policy_batch(model, packed, temperature, PV_EVALUATE_COUNT, device)
    k = int(n[0])
    out = pol[0, :k].cpu().numpy()
    return out if temperature == 0 else out.tolist()


# Action selection with Monte Carlo Tree Search
def pv_mcts_action(model, temperature=0, device=None):
    """Returns a function of the game state that selects an action based on PV-MCTS (pv_mcts.py:98-103)."""
    def pv_mcts_action(state):
        policy = pv_mcts_policy(model, deepcopy(state), temperature, device)
        return np.random.choice(state.legal_actions(), p=policy)
    return pv_mcts_action


# Boltzmann distribution
def boltzman(xs, temperature):
    """Boltzmann distribution (pv_mcts.py:106-109)"""
    xs = [x ** (1 / temperature) for x in xs]
    return [x / sum(xs) for x in xs]
