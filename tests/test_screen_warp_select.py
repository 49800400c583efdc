"""CPU check of the selection logic of the two mma.sync screening shapes (csrc/dune_screen_mma_kernel.cuh), transcribed to numpy:
tau (the M-th smallest upper-bound key) and the candidate set {lower bound <= tau}.

  dune_screen_mma_kernel   4 warps per item: pass p, warp w, lane -> point 128 p + 32 w + own(lane); M REDUX rounds per warp over its
                           keys, then M rounds over the 4 M survivors; candidates appended through a shared counter
  dune_screen_warp_kernel  1 warp per item: tile j, lane -> point 32 j + own(lane); M REDUX rounds over all the lane's keys; candidates
                           compacted tile by tile with __ballot_sync + __popc(ballot & lanes below)

On random bounds -- with ties, and clouds of n < 32, 33, 500 and 1000 points -- both give the same tau and the same candidate set, and
the ballot compaction writes every candidate exactly once to positions 0 .. count-1."""
import numpy as np
import pytest

KCAND = 32


def orderable(d):
    u = np.asarray(d, np.float32).view(np.uint32).astype(np.uint64)
    out = np.where(u & 0x80000000, (~u) & 0xFFFFFFFF, u | 0x80000000)
    return np.where(np.isnan(d), 0xFFFFFFFF, out).astype(np.uint64)


def unique_key(k, idx, bits):
    mask = (1 << bits) - 1
    return ((np.minimum(k, 0xFFFFF000) + mask + 1) & ~np.uint64(mask) & 0xFFFFFFFF) | np.uint64(idx)


def own(lane):
    return 8 * (lane & 3) + (lane >> 2)


def keys_of(d, eps, n, bits):
    i = np.arange(len(d))
    return np.where(i < n, unique_key(orderable(d + eps), i, bits), 0xFFFFFFFF).astype(np.uint64)


def redux_rounds(q, M):
    """q: (lanes, slots) keys of one warp; M rounds of (min over lane, __reduce_min_sync, remove); returns the M minima."""
    q = q.copy()
    out = []
    for _ in range(M):
        md = q.min()
        out.append(md)
        q[q == md] = 0xFFFFFFFF
    return np.array(out, np.uint64)


def cta_shape(d, eps, n, M, kP):
    bits = 9 if kP <= 4 else 10
    key = keys_of(d, eps, n, bits)
    lanes = np.arange(32)
    surv = []
    for w in range(4):
        idx = np.array([[128 * p + 32 * w + own(l) for p in range(kP)] for l in lanes])
        surv.append(redux_rounds(key[idx], M))
    tau = redux_rounds(np.concatenate(surv)[None, :], M)[-1]
    lb = orderable(d - eps)
    i = np.arange(len(d))
    cand = np.nonzero((i < n) & (key != 0xFFFFFFFF) & (lb <= tau))[0]
    return tau, set(cand.tolist()), len(cand)


def warp_shape(d, eps, n, M, kP):
    bits = 9 if kP <= 4 else 10
    key = keys_of(d, eps, n, bits)
    lanes = np.arange(32)
    idx = np.array([[32 * j + own(l) for j in range(4 * kP)] for l in lanes])
    q = np.where(idx < n, key[idx], 0xFFFFFFFF)
    tau = redux_rounds(q, M)[-1]
    lb = orderable(d - eps)
    lst, nc = {}, 0
    for j in range(4 * kP):
        if 32 * j >= n:
            continue
        i = 32 * j + own(lanes)
        take = (i < n) & (lb[i] <= tau)
        bal = sum(1 << int(l) for l in lanes[take])
        for l in lanes[take]:
            pos = nc + bin(bal & ((1 << int(l)) - 1)).count("1")
            if pos < KCAND:
                assert pos not in lst
                lst[pos] = int(i[l])
        nc += bin(bal).count("1")
    if nc <= KCAND:
        assert sorted(lst) == list(range(nc))
    return tau, set(lst.values()), nc


@pytest.mark.parametrize("n", [7, 31, 33, 100, 500, 512, 513, 1000, 1024])
@pytest.mark.parametrize("ties", [False, True])
def test_one_warp_selection_equals_four_warp_merge(n, ties):
    rng = np.random.default_rng(n * 2 + ties)
    kP = 4 if n <= 512 else 8
    P = 128 * kP
    M = 10
    for trial in range(6):
        d = rng.uniform(0.0, 3.0, P).astype(np.float32)
        if ties:  # few distinct distances: equal upper bounds, told apart only by the index bits
            d = np.round(d * 2) / 2
        eps = np.float32(rng.choice([1e-3, 2e-2, 0.3])) * np.ones(P, np.float32)
        if trial % 2:
            eps = (eps * rng.uniform(0.5, 1.5, P)).astype(np.float32)
        d[n:] = rng.uniform(-5, 5, P - n)  # rows beyond n carry garbage: they must never count
        t_old, s_old, c_old = cta_shape(d, eps, n, M, kP)
        t_new, s_new, c_new = warp_shape(d, eps, n, M, kP)
        assert t_old == t_new
        assert c_old == c_new
        if c_new <= KCAND:
            assert s_old == s_new
        assert all(i < n for i in s_new)
        if n >= M:
            assert c_new >= M  # the M points of smallest upper bound are always candidates
