"""CPU restatement of the Gumbel root (Gumbel AlphaZero, Danihelka et al. 2022; DeepMind mctx gumbel_muzero_policy) on top of the
reference-literal search of oracle/mcts_oracle.py.

The reference has no Gumbel root.  This restates aq_mcts_gumbel_root, the Gumbel rule of aq_mcts_select_gumbel and
aq_mcts_gumbel_result (csrc/mcts.cu) in numpy float64, each operation rounded as the kernels round it:
  key    = mix64(mix64((seed ^ GUMBEL_DOMAIN) + GOLDEN * (game_id + 1)) + PLY_MUL * (ply + 1))
  U_c    = ((mix64(key + GOLDEN * (c + 1)) >> 11) + 0.5) * 2^-53                                    in (0, 1)
  g_c    = gumbel_scale * (-log(-log U_c))
  base_c = float32(g_c + (log p_c - max log p))                          stored once, right after simulation 1 expanded the root
  v_mix  = (v_hat + N * (S_pq / S_p)) / (N + 1)  over the visited children, pt = max(p, FLT_MIN), sums in warp order
  sigma  = ((50 + max n) * 0.1) * (cq - min cq) / max(max cq - min cq, 1e-8),  cq = -(w / n) if visited else v_mix
  score  = max(-1e9, base + sigma)
The root descent takes the first argmax of the score over the children whose visit count is considered_visit(m, n, sum of visits)
(mctx's sequential-halving table); the result is softmax(log p + sigma) and the first argmax over the most visited children.
log / exp may differ from the GPU's in the last bit: base is rounded to float32 (the same on both sides unless a value lies within
that bit of a float32 rounding boundary), and the improved policy is compared within one float32 ulp.
"""
import math

import numpy as np

from oracle import mcts_oracle as mo

from mcts_noise_oracle import GOLDEN, M64, PLY_MUL, mix64, warp_sum

GUMBEL_DOMAIN = 0x13198A2E03707344
FLT_MIN = np.float32(np.finfo(np.float32).tiny)
MAXVISIT_INIT, VALUE_SCALE = 50.0, 0.1


def sequence_of_considered_visits(m, n):
    """mctx seq_halving.get_sequence_of_considered_visits, literally."""
    if m <= 1:
        return tuple(range(n))
    log2max = int(math.ceil(math.log2(m)))
    sequence = []
    visits = [0] * m
    num_considered = m
    while len(sequence) < n:
        num_extra_visits = max(1, int(n / (log2max * num_considered)))
        for _ in range(num_extra_visits):
            sequence.extend(visits[:num_considered])
            for i in range(num_considered):
                visits[i] += 1
        num_considered = max(2, num_considered // 2)
    return tuple(sequence[:n])


def considered_visit(m, n, k):
    """Entry k of sequence_of_considered_visits(m, n), continued past n - 1 by the same phases, as the kernel computes it."""
    if m <= 1:
        return k
    log2max = (m - 1).bit_length()
    nc, base = m, 0
    while True:
        extra = max(1, n // (log2max * nc))
        if k < extra * nc:
            return base + k // nc
        k -= extra * nc
        base += extra
        nc = max(2, nc // 2)


def gumbel_key(seed, game_id, ply):
    gid = np.asarray(game_id, dtype=np.int64).astype(np.uint64)
    with np.errstate(over="ignore"):
        a = np.uint64((int(seed) ^ GUMBEL_DOMAIN) & M64) + np.uint64(GOLDEN) * (gid + np.uint64(1))
        return mix64(mix64(a) + np.uint64(PLY_MUL * (int(ply) + 1) & M64))


def gumbel_uniform(seed, game_id, ply, K):
    """U_c [N, K] in (0, 1) for the games of game_id (int array [N])."""
    key = gumbel_key(seed, game_id, ply)
    c = np.arange(K, dtype=np.uint64)
    with np.errstate(over="ignore"):
        bits = mix64(key[:, None] + np.uint64(GOLDEN) * (c[None, :] + np.uint64(1)))
    return ((bits >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def gumbel_draw(seed, game_id, ply, K, scale=1.0):
    """g [N, K]; scale is the float32 the ABI takes."""
    return float(np.float32(scale)) * -np.log(-np.log(gumbel_uniform(seed, game_id, ply, K)))


def logits(priors):
    with np.errstate(divide="ignore"):
        return np.log(np.asarray(priors, np.float32).astype(np.float64))


def base_scores(priors, g):
    """float32(g + (log p - max log p)) [K]."""
    lg = logits(priors)
    return (g + (lg - lg.max())).astype(np.float32)


def sigma(w, n, priors, v_hat):
    """sigma(completed Q) [K] of the root children with values w (float64), visits n (int), priors p (float32)."""
    w, n = np.asarray(w, np.float64), np.asarray(n, np.int64)
    vis = n > 0
    q = np.zeros(len(n))
    q[vis] = -(w[vis] / n[vis])
    pt = np.where(vis, np.maximum(np.asarray(priors, np.float32), FLT_MIN).astype(np.float64), 0.0)
    N = int(n.sum())
    sp = warp_sum(pt[None, :])[0]
    spq = warp_sum(np.where(vis, pt * q, 0.0)[None, :])[0]
    v_mix = (float(v_hat) + float(N) * (spq / sp if N > 0 else 0.0)) / float(N + 1)
    cq = np.where(vis, q, v_mix)
    lo, hi = cq.min(), cq.max()
    return ((MAXVISIT_INIT + float(n.max())) * VALUE_SCALE) * ((cq - lo) / max(hi - lo, 1e-8))


def scores(base, sig):
    return np.maximum(-1e9, np.asarray(base, np.float32).astype(np.float64) + sig)


def pick(sc, n, visits):
    """First argmax of sc over the children with n == visits; 0 when there is none (jnp.argmax over all -inf)."""
    cand = np.flatnonzero(np.asarray(n) == visits)
    return int(cand[np.argmax(np.asarray(sc)[cand])]) if len(cand) else 0


def improved_policy(priors, sig):
    """softmax(log p + sigma) [K], the sum in warp order."""
    z = logits(priors) + sig
    e = np.exp(z - z.max())
    return e / warp_sum(e[None, :])[0]


class _GumbelRoot(mo._Node):
    """The root node of a Gumbel search: next_child_node is the Gumbel rule, every node below it keeps the reference's PUCT."""
    __slots__ = ("base", "v_hat", "m", "budget")

    def __init__(self, state, p):
        super().__init__(state, p)
        self.base = None   # float32 [K] once the Gumbel state is drawn

    def child_stats(self):
        ch = self.child_nodes
        return ([c.w for c in ch], [c.n for c in ch], np.array([c.p for c in ch], np.float32))

    def sigma(self):
        w, n, p = self.child_stats()
        return sigma(w, n, p, self.v_hat)

    def next_child_node(self):
        if self.base is None:
            return super().next_child_node()
        n = [c.n for c in self.child_nodes]
        cv = considered_visit(self.m, self.budget, sum(n))
        return self.child_nodes[pick(scores(self.base, self.sigma()), n, cv)]


class GumbelSearch:
    """One search with a Gumbel root: simulation 1 expands the root, init() draws its Gumbel state, sims - 1 more follow."""

    def __init__(self, state, considered, scale=1.0):
        self.root = _GumbelRoot(state, 0)
        self.considered, self.scale = considered, scale

    def init(self, seed, game_id, ply, sims):
        r = self.root
        if r.base is not None or not r.child_nodes or r.n != 1:
            return
        _, _, p = r.child_stats()
        r.base = base_scores(p, gumbel_draw(seed, [game_id], ply, len(p), self.scale)[0])
        r.v_hat, r.m, r.budget = float(r.w), min(self.considered, len(p)), sims - 1

    def search(self, predict, sims, seed=0, game_id=0, ply=0):
        for i in range(sims):
            self.root.evaluate(predict)
            if i == 0:
                self.init(seed, game_id, ply, sims)

    def counts(self):
        return [c.n for c in self.root.child_nodes] if self.root.child_nodes else []

    def actions(self):
        return self.root.state.legal_actions() if self.root.child_nodes else []

    def result(self):
        """(improved policy float64 [K], chosen child index)."""
        r = self.root
        sig = r.sigma()
        n = self.counts()
        return improved_policy(r.child_stats()[2], sig), pick(scores(r.base, sig), n, max(n))
