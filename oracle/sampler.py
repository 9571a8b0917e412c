"""ORACLE (test infrastructure -- imported only by tests/, __graft_entry__.smoke() and bench.py's CPU legs).

CPU restatement of the in-kernel action sampler of merlin_env_policy_step (include/merlin_b200.h).  The reference
samples with torch.distributions.Categorical(logits).sample() and stores .log_prob(a) (src/actor_critic.py act();
src/ppo.py:70-86; src/fomaml.py:65-84); torch's generator stream cannot be reproduced by a fused kernel, so the draw is
SPECIFIED by the product and restated here independently (pure-Python integer arithmetic for Philox, vectorised on
uint64 arrays in uniform_batch, numpy float32 for the inverse CDF):

    u      = (Philox4x32-10(counter = (env, draw, 0, 0), key = (seed_lo, seed_hi))[0] >> 8) * 2**-24
    action = first a with cumsum(exp(l - max(l)))[a] > u * sum(exp(l - max(l)))          (float32, left to right)
    logp   = (l[action] - max(l)) - log(sum)

Philox4x32-10: Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC'11 (Random123).  Pinned by
the Random123 known-answer vectors in tests/test_host_logic.py.  exp/log differ in the last ulp between libm and the
GPU's expf/logf: tests compare log-probabilities with a tolerance and skip actions whose draw lies within that
tolerance of a CDF boundary.  `reference_f64` is the float64 distribution every draw must be consistent with.
"""
from __future__ import annotations

import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF


def philox4x32_10(counter, key):
    """counter: 4 ints, key: 2 ints (all uint32) -> 4 uint32 words."""
    c0, c1, c2, c3 = [int(c) & MASK for c in counter]
    k0, k1 = [int(k) & MASK for k in key]
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & MASK, p1 & MASK, ((p0 >> 32) ^ c3 ^ k1) & MASK, p0 & MASK
        k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
    return c0, c1, c2, c3


def uniform(seed, env, draw):
    """The float32 uniform in [0, 1) env `env` uses for its draw number `draw`."""
    x = philox4x32_10((env, draw, 0, 0), (seed & MASK, (seed >> 32) & MASK))[0]
    return np.float32(x >> 8) * np.float32(1.0 / 16777216.0)


def philox4x32_10_batch(counter, key):
    """`philox4x32_10` on arrays: counter = 4 uint32 arrays (broadcast together), key = 2 ints.  uint64 arithmetic,
    where the product of two uint32 words is exact.  Returns 4 uint64 arrays holding the uint32 output words."""
    m32, s32 = np.uint64(MASK), np.uint64(32)
    c0, c1, c2, c3 = (a & m32 for a in np.broadcast_arrays(*(np.asarray(c, np.uint64) for c in counter)))
    k0, k1 = (np.uint64(int(k) & MASK) for k in key)
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c0, np.uint64(M1) * c2
        c0, c1, c2, c3 = ((p1 >> s32) ^ c1 ^ k0) & m32, p1 & m32, ((p0 >> s32) ^ c3 ^ k1) & m32, p0 & m32
        k0, k1 = (k0 + np.uint64(W0)) & m32, (k1 + np.uint64(W1)) & m32
    return c0, c1, c2, c3


def uniform_batch(seed, envs, draws):
    """`uniform` for arrays of env indices and draw numbers (broadcast together) -> float32 of their shape."""
    x = philox4x32_10_batch((envs, draws, 0, 0), (seed & MASK, (seed >> 32) & MASK))[0]
    return (x >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)


def sample_batch(logits, seed, draws, greedy=False):
    """logits float32[N, A], draws int[N] (draw number of each env) -> (actions int64[N], logp float32[N],
    margin float64[N]).  margin = distance of u*sum to the nearest CDF boundary relative to sum (a draw with a tiny
    margin may legitimately differ by one action between exp implementations); 1 in greedy mode (first maximum)."""
    l = np.asarray(logits, dtype=np.float32)
    N, A = l.shape
    rows = np.arange(N)
    with np.errstate(invalid="ignore", over="ignore"):
        m = l.max(axis=1, keepdims=True)
        ex = np.exp((l - m).astype(np.float32)).astype(np.float32)
        cum = np.cumsum(ex, axis=1, dtype=np.float32)  # float32, left to right, as the kernel accumulates
        s = cum[:, -1]
        if greedy:
            a = np.argmax(l, axis=1)
            margin = np.ones(N)
        else:
            target = (uniform_batch(seed, rows, draws) * s).astype(np.float32)
            above = cum > target[:, None]
            a = np.where(above.any(axis=1), above.argmax(axis=1), A - 1)
            gap = np.abs(cum[:, :-1].astype(np.float64) - target[:, None].astype(np.float64))
            margin = gap.min(axis=1) / s.astype(np.float64) if A > 1 else np.ones(N)
        logp = ((l[rows, a] - m[:, 0]).astype(np.float32) - np.log(s).astype(np.float32)).astype(np.float32)
    return a.astype(np.int64), logp, margin


def reference_f64(logits, u, tol=1e-5):
    """The plain float64 categorical distribution of `logits` [N, A] (-inf = probability 0) and the actions a draw
    `u` [N] may pick: cdf float64[N, A], logp64 float64[N, A] (log_softmax; -inf where the probability is 0) and
    allowed bool[N, A] = p[a] > 0 and cdf[a-1] <= u + tol and cdf[a] > u - tol.  `tol` covers the float32 rounding of the
    kernel's exp / sum / u * sum, so every action a float32 inverse CDF can legitimately pick is allowed."""
    l = np.asarray(logits, dtype=np.float64)
    u = np.asarray(u, dtype=np.float64).reshape(-1, 1)
    z = l - l.max(axis=1, keepdims=True)
    ex = np.exp(z)
    tot = ex.sum(axis=1, keepdims=True)
    p = ex / tot
    with np.errstate(divide="ignore"):
        logp64 = z - np.log(tot)
    cdf = np.cumsum(p, axis=1)
    below = np.concatenate([np.zeros((l.shape[0], 1)), cdf[:, :-1]], axis=1)
    allowed = (p > 0) & (below <= u + tol) & (cdf > u - tol)
    return cdf, logp64, allowed
