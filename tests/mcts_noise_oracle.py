"""CPU restatement of Dirichlet noise on the search root (AlphaZero), on top of the reference-literal search of oracle/mcts_oracle.py.

The reference has no root noise.  ``dirichlet`` restates the counter-based draw of aq_mcts_root_noise (csrc/mcts.cu) in numpy
float64 with the same counter layout, so a draw here and on the GPU differ only by the last-bit rounding of log / exp / cos:
  key     = mix64(mix64((seed ^ NOISE_DOMAIN) + GOLDEN * (game_id + 1)) + PLY_MUL * (ply + 1))
  U(c, j) = ((mix64(key + GOLDEN * (c * DRAWS + j + 1)) >> 11) + 1) * 2^-53                 in (0, 1]
  gamma   : Marsaglia-Tsang at shape alpha (alpha >= 1) or alpha + 1 boosted by U(c, 0)^(1/alpha) (alpha < 1), attempt i using
            U(c, 3i+1), U(c, 3i+2) (Box-Muller) and U(c, 3i+3) (acceptance); ATTEMPTS attempts, then log G = log d
  eta     = exp(log gamma - max) / S, S summed in the order of the GPU warp (lane partial sums, then an xor butterfly).
``NoisedSearch`` applies it to a ReuseSearch the way BatchedMCTS does: once per search, before the first descent that reads the
root's children (before simulation 1 for a carried root, after it for a fresh one).  Noised priors are stored as np.float32, so
the PUCT arithmetic stays float32 under NEP 50, as with the network's priors.
"""
import numpy as np

from mcts_reuse_oracle import ReuseSearch

M64 = (1 << 64) - 1
GOLDEN = 0x9E3779B97F4A7C15
PLY_MUL = 0xD1B54A32D192ED03
NOISE_DOMAIN = 0x243F6A8885A308D3
ATTEMPTS = 16
DRAWS = 1 + 3 * ATTEMPTS
LANES, SLOTS = 32, 5   # warp width and children per lane (136 = 5 * 32 rounded up from 133)


def mix64(z):
    """splitmix64 finaliser on uint64 arrays (wrapping arithmetic)."""
    z = np.asarray(z, dtype=np.uint64)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def noise_key(seed, game_id, ply):
    """uint64[N] keys of games game_id (int array) at one ply."""
    gid = np.asarray(game_id, dtype=np.int64).astype(np.uint64)
    with np.errstate(over="ignore"):
        a = np.uint64((int(seed) ^ NOISE_DOMAIN) & M64) + np.uint64(GOLDEN) * (gid + np.uint64(1))
        return mix64(mix64(a) + np.uint64(PLY_MUL * (int(ply) + 1) & M64))


def uniform(key, K, j):
    """U(c, j) for every key [N] and child c < K -> float64 [N, K]."""
    c = np.arange(K, dtype=np.uint64)
    with np.errstate(over="ignore"):
        bits = mix64(key[:, None] + np.uint64(GOLDEN) * (c[None, :] * np.uint64(DRAWS) + np.uint64(j + 1)))
    return ((bits >> np.uint64(11)) + np.uint64(1)).astype(np.float64) * 2.0 ** -53


def log_gamma(key, K, alpha):
    """log gamma_c [N, K] of the Dirichlet draw."""
    alpha = float(np.float32(alpha))
    boost = alpha < 1.0
    a = alpha + 1.0 if boost else alpha
    d = a - 1.0 / 3.0
    k = 1.0 / np.sqrt(9.0 * d)
    lg = np.full((key.shape[0], K), np.log(d))
    todo = np.ones(lg.shape, dtype=bool)
    for i in range(ATTEMPTS):
        if not todo.any():
            break
        x = np.sqrt(-2.0 * np.log(uniform(key, K, 3 * i + 1))) * np.cos(6.283185307179586 * uniform(key, K, 3 * i + 2))
        t = 1.0 + k * x
        with np.errstate(invalid="ignore", divide="ignore"):
            v = t * t * t
            rhs = ((0.5 * x * x + d) - d * v) + d * np.log(v)
            ok = todo & (t > 0.0) & (np.log(uniform(key, K, 3 * i + 3)) < rhs)
            lg = np.where(ok, np.log(d * v), lg)
        todo &= ~ok
    if boost:
        lg = lg + np.log(uniform(key, K, 0)) / alpha
    return lg


def warp_sum(e):
    """Sum over the last axis (K <= 160) in the order of the GPU warp: lane l adds children l, l + 32, ... from 0.0, then an xor
    butterfly over the 32 lane sums."""
    n, K = e.shape
    pad = np.zeros((n, LANES * SLOTS))
    pad[:, :K] = e
    s = np.zeros((n, LANES))
    for slot in range(SLOTS):
        s = s + pad[:, slot * LANES:(slot + 1) * LANES]
    lanes = np.arange(LANES)
    for m in (16, 8, 4, 2, 1):
        s = s + s[:, lanes ^ m]
    return s[:, 0]


def dirichlet(seed, game_id, ply, K, alpha):
    """eta [N, K] float64 for the games of `game_id` (int array [N]) at one ply, K children each."""
    key = noise_key(seed, game_id, ply)
    lg = log_gamma(key, K, alpha)
    e = np.exp(lg - lg.max(axis=1, keepdims=True))
    return e / warp_sum(e)[:, None]


def noised_priors(priors, eta, fraction):
    """float32((1 - fraction) * p + fraction * eta) in double, rounded once; fraction is the float32 the ABI takes."""
    f = float(np.float32(fraction))
    return ((1.0 - f) * np.asarray(priors, np.float32).astype(np.float64) + f * eta).astype(np.float32)


class NoisedSearch(ReuseSearch):
    """ReuseSearch with root noise: noise(...) is a no-op once the root has been noised, until advance() sets a new root."""

    def __init__(self, state, alpha, fraction=0.25):
        super().__init__(state)
        self.alpha, self.fraction, self.noised = alpha, fraction, False

    def advance(self, path, capacity, reserve):
        self.noised = False
        return super().advance(path, capacity, reserve)

    def noise(self, seed, game_id, ply):
        ch = self.root.child_nodes
        if self.noised or ch is None:   # not expanded yet
            return
        self.noised = True
        if not ch:
            return
        eta = dirichlet(seed, [game_id], ply, len(ch), self.alpha)[0]
        for c, p in zip(ch, noised_priors([c.p for c in ch], eta, self.fraction)):
            c.p = p

    def search(self, predict, sims, seed=0, game_id=0, ply=0):
        self.noise(seed, game_id, ply)
        for i in range(sims):
            self.root.evaluate(predict)
            if i == 0:
                self.noise(seed, game_id, ply)

