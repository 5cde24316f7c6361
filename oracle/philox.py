"""numpy restatement of the device Philox draws (csrc/common.cuh: Philox, u53).

TEST INFRASTRUCTURE ONLY (see oracle/oracle.py).  Philox4x32-10 (Salmon et al. 2011, the
Random123 `philox4x32` with 10 rounds) over arrays of counters, and the two ways the library
turns its output into draws:

- `policy_draws`: the epsilon-greedy draws of the DQN Q head when the caller supplies none
  (csrc/dqn.cu: dqn_head_kernel, csrc/gemm_sm100_epilogue.inc: EPI_QHEAD);
- `env_draws`: the packet (start, target, size) draws of the batched Routing env when no
  host draws are set (csrc/routing_env.cu: draw()).

Parity status: PINNED against the Random123 known-answer vectors in
tests/test_oracle_philox.py.
"""
import numpy as np

_M0, _M1 = 0xD2511F53, 0xCD9E8D57
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_MASK = 0xFFFFFFFF

# policy draws: counter word 3 is the step's high word XOR this constant, the key is the seed XOR this one
POLICY_STEP_HI_XOR = 0x5BD1E995
POLICY_KEY_XOR = 0xA5A5A5A5DEADBEEF


def _u32(x):
    return np.asarray(x, dtype=np.uint64) & np.uint64(_MASK)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counters (c0, c1, c2, c3) under key (k0, k1); every argument broadcasts.
    Returns four uint32 arrays (r0, r1, r2, r3)."""
    c0, c1, c2, c3, k0, k1 = np.broadcast_arrays(*(_u32(x) for x in (c0, c1, c2, c3, k0, k1)))
    c0, c1, c2, c3, k0, k1 = (x.copy() for x in (c0, c1, c2, c3, k0, k1))
    m0, m1, mask = np.uint64(_M0), np.uint64(_M1), np.uint64(_MASK)
    for _ in range(10):
        p0 = m0 * c0  # 32 x 32 -> 64 bits: exact in uint64
        p1 = m1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0 = (k0 + np.uint64(_W0)) & mask
        k1 = (k1 + np.uint64(_W1)) & mask
    return tuple(x.astype(np.uint32) for x in (c0, c1, c2, c3))


def u53(a, b):
    """common.cuh u53: a uniform double in [0, 1) from the top 27 bits of `a` and the top 26 bits of `b`."""
    a, b = np.asarray(a, dtype=np.uint32), np.asarray(b, dtype=np.uint32)
    return ((a >> np.uint32(5)).astype(np.float64) * 67108864.0 + (b >> np.uint32(6)).astype(np.float64)) / 9007199254740992.0


def umulhi(r, n):
    """__umulhi(r, n) for 32-bit r and n: an index in [0, n)."""
    return ((np.asarray(r, dtype=np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


def _key(seed):
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return seed & _MASK, seed >> 32


def policy_draws(rows, n_act, seed, step):
    """The device epsilon-greedy draws of rows 0..rows-1 (or of the row indices in `rows`, an array):
    counter (row lo, row hi, step lo, step hi ^ 0x5bd1e995), key seed ^ 0xA5A5A5A5DEADBEEF.
    Returns (rand_action int64 in [0, n_act), rand_u float64 in [0, 1)); a row acts at random where u < epsilon."""
    r = np.arange(rows, dtype=np.uint64) if np.isscalar(rows) else np.asarray(rows, dtype=np.uint64)
    step = int(step) & 0xFFFFFFFFFFFFFFFF
    k0, k1 = _key(int(seed) ^ POLICY_KEY_XOR)
    out = philox4x32_10(r & np.uint64(_MASK), r >> np.uint64(32), step & _MASK, (step >> 32) ^ POLICY_STEP_HI_XOR, k0, k1)
    return umulhi(out[0], n_act), u53(out[1], out[2])


def env_draws(B, A, N, seed, step):
    """The device packet draws of a batched Routing call: tables [B, A] in the slot format of
    Routing.set_draws (slot s feeds the s-th respawn of env b in packet-id order).  Counter
    (slot, env b, step lo, step hi), key seed; `step` is the env's call counter at that call
    (Routing._calls: reset and step both count).  Returns (start int32, target int32, size float64)."""
    slot = np.arange(A, dtype=np.uint64)[None, :]
    b = np.arange(B, dtype=np.uint64)[:, None]
    step = int(step) & 0xFFFFFFFFFFFFFFFF
    k0, k1 = _key(seed)
    r0, r1, r2, r3 = philox4x32_10(slot, b, step & _MASK, step >> 32, k0, k1)
    return umulhi(r0, N).astype(np.int32), umulhi(r1, N).astype(np.int32), u53(r2, r3)
