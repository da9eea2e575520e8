"""The minibatch option of the update (Algo_PPO(n_minibatches=B), DESIGN.md §4 "Minibatches") restated in numpy: the bucket
b(car, g, e) of Philox stream 3 and the plan of mhppo_minibatch_plan (bucket-major column lists, offsets, counts).  The
checks here hold the restatement to its definition and need no GPU; tests/test_minibatch_gpu.py holds the kernels and
Algo_PPO to it.  The reference has no minibatches, so the restatement lives here and not in oracle/.

Stream 3 of the policy-noise contract (DESIGN.md §2 "RNG contract", next to streams 1 and 2 of oracle/ppo_oracle.py's
policy_normal / policy_uniform): counter = (epoch*C + car, 3 | iteration << 8, g_lo, g_hi), key = the env seed; in that epoch
the (car, env) column of global env id g goes to bucket (w0 * B) >> 32."""
import numpy as np
import pytest
from scipy import stats

from oracle import ppo_oracle as PO
from oracle.refshim import philox as PH


def minibatch_bucket(epoch, car, C, env_id, seed, B, iteration=0):
    """b(car, g, e) of stream 3, vectorised over car / env_id."""
    w = PO.philox_blocks(np.asarray(epoch, np.uint64) * np.uint64(C) + np.asarray(car, np.uint64), 3 | (iteration << 8), env_id, seed)
    return ((w[0] * np.uint64(B)) >> np.uint64(32)).astype(np.int64)


def buckets(C, N, env_id0, seed, iteration, epoch, B):
    """b(car, g, e) of every column, [C][N]."""
    g = env_id0 + np.arange(N, dtype=np.int64)
    return minibatch_bucket(epoch, np.arange(C)[:, None], C, g[None, :], seed, B, iteration)


def minibatch_plan(route, exist, act_d, seed, env_id0, iteration, epochs, B):
    """What mhppo_minibatch_plan writes.  route / exist [C][N], act_d [C][N].  Returns (lists, offsets, counts):
    lists [E][3] python lists of column ids m = car*N + n (cross, wait, existing; bucket-major, ascending m within a bucket),
    offsets int64 [E][3][B+1], counts int64 [E][5][B]."""
    C, N = route.shape
    route, exist, act_d = (np.asarray(a).reshape(-1) for a in (route, exist, act_d))
    ex = exist != 0
    sels = (route == 0, route == 1, ex, ex & (act_d == 0), ex & (act_d == 1))
    lists, offsets, counts = [], np.zeros((epochs, 3, B + 1), np.int64), np.zeros((epochs, 5, B), np.int64)
    for e in range(epochs):
        b = buckets(C, N, env_id0, seed, iteration, e, B).reshape(-1)
        row = []
        for s, sel in enumerate(sels):
            m = np.nonzero(sel)[0]
            counts[e, s] = np.bincount(b[m], minlength=B)
            if s < 3:
                row.append(m[np.argsort(b[m], kind="stable")])
                offsets[e, s, 1:] = np.cumsum(counts[e, s])
        lists.append(row)
    return lists, offsets, counts


def test_bucket_matches_definition():
    """The vectorised restatement against the scalar Philox of the RNG contract, word 0 scaled by B."""
    rng = np.random.default_rng(0)
    for seed in (0, 1, 77, 2 ** 40 + 3):
        for _ in range(20):
            C, e, it = int(rng.integers(1, 9)), int(rng.integers(0, 12)), int(rng.integers(0, 5000))
            car, g, B = int(rng.integers(0, C)), int(rng.integers(0, 2 ** 33)), int(rng.integers(1, 1025))
            w0 = PH.philox4x32_10((e * C + car, 3 | (it << 8), g & 0xFFFFFFFF, g >> 32), (seed & 0xFFFFFFFF, seed >> 32))[0]
            assert minibatch_bucket(e, car, C, g, seed, B, it) == (w0 * B) >> 32


def test_one_bucket_is_all_zeros():
    for C, N in ((1, 26), (4, 257)):
        assert not buckets(C, N, 5, 9, 3, 2, 1).any()


def test_bucket_streams_differ():
    """Stream 3 is not streams 1 / 2, and epochs and iterations draw different buckets."""
    b = buckets(4, 4096, 0, 7, 0, 0, 64)
    assert (b != buckets(4, 4096, 0, 7, 0, 1, 64)).mean() > 0.9
    assert (b != buckets(4, 4096, 0, 7, 1, 0, 64)).mean() > 0.9
    w1 = PO.philox_blocks(np.arange(4)[:, None], 1, np.arange(4096)[None, :], 7)[0]
    assert (b != ((w1 * np.uint64(64)) >> np.uint64(32)).astype(np.int64)).mean() > 0.9


@pytest.mark.parametrize("B", [1, 7, 64])
def test_plan_at_one_bucket_is_nonzero_order_and_sharding(B):
    """At B = 1 the lists are the compacted torch.nonzero lists; for any B, the plan of envs [r*n, (r+1)*n) with env_id0 = r*n
    is the matching part of the plan of all envs (same buckets, same order within a bucket)."""
    rng = np.random.default_rng(B)
    C, N, R, E = 4, 300, 3, 3
    n = N // R
    route = rng.choice(np.array([-1, 0, 1], np.int8), (C, N))
    exist = (route >= 0).astype(np.int8)
    act_d = rng.integers(0, 2, (C, N)).astype(np.float32)
    L, off, cnt = minibatch_plan(route, exist, act_d, 11, 0, 4, E, B)
    if B == 1:
        for e in range(E):
            for s, sel in enumerate((route == 0, route == 1, exist != 0)):
                assert np.array_equal(L[e][s], np.nonzero(sel.reshape(-1))[0])
    total = np.zeros_like(cnt)
    for r in range(R):
        sl = slice(r * n, (r + 1) * n)
        Ls, offs, cs = minibatch_plan(route[:, sl], exist[:, sl], act_d[:, sl], 11, r * n, 4, E, B)
        total += cs
        for e in range(E):
            for s in range(3):
                for b in range(B):
                    mine = Ls[e][s][offs[e, s, b]:offs[e, s, b + 1]]
                    glob = L[e][s][off[e, s, b]:off[e, s, b + 1]]
                    env = glob % N
                    part = glob[(env >= r * n) & (env < (r + 1) * n)]
                    assert np.array_equal((mine // n) * N + mine % n + r * n, part)
    assert np.array_equal(total, cnt)                   # the all-reduced counts of the shards are the counts of the whole


@pytest.mark.parametrize("B", [2, 7, 16, 64, 1024])
def test_bucket_sizes_are_uniform(B):
    """131 072 envs x 4 cars: the bucket sizes pass a chi-square test of uniformity at p > 1e-4, in several epochs."""
    C, N = 4, 131072
    for e in (0, 9):
        sizes = np.bincount(buckets(C, N, 0, 4, 17, e, B).reshape(-1), minlength=B)
        assert sizes.sum() == C * N
        chi2 = ((sizes - C * N / B) ** 2 / (C * N / B)).sum()
        assert stats.chi2.sf(chi2, B - 1) > 1e-4, (B, e, chi2)
