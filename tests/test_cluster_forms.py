"""Average-linkage clustering (AHC) of many buckets in one call, against the oracle.

On the device a bucket takes one of five replay forms, chosen by its point count after the isolated-pair mask and by
whether the speculative component pass flagged one of its components (bkid_api.cuh cluster_ahc):

    unflagged,  < 512 points       ahc_replay_rank (shared memory)
    unflagged, >= 512 points       ahc_rg_* (global-memory rank form: radix sorts by bucket, one warp per tie group)
    flagged,    < 900 points       ahc_replay_smem, first launch
    flagged,  900 .. 4095 points   ahc_replay_smem, second launch
    flagged,  >= 4096 points       ahc_bucket_exact

The ladder below holds a bucket on each side of every boundary, degenerate buckets between them, tiny filler buckets
(so there are more than 256 and the bucket-keyed radix sorts take two digit passes), and two large same-chromosome
buckets whose mask sorts take the multi-CTA partition and the heapsort fallback.  The oracle clusters with the component
model (oracle.cc orc_model_ahc_tree): the literal O(N^3) form is out of reach beyond ~1 500 points, and the model is
checked against it here on every rung up to that size.  The model also predicts which components the device flags, so
the CPU side knows which form each bucket takes, and the GPU tests check that prediction against the count the library
prints with BKID_DEBUG_TIMING=1."""
import os
import re
import sys
import types

import numpy as np
import pytest

W = 1243.15                                  # cluster distance used across the suite
THR = int(W)                                 # (long) threshold of the AHC and the mask
NT = 20                                      # targets: 21 x 21 bucket names
NAMES = ["c%02d" % t for t in range(NT)]
TLEN = [250_000_000] * NT
RG_LO, SMEM_HI, EXACT_LO = 512, 900, 4096    # form boundaries in cluster_ahc
N_FILLERS = 300
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# (name, post-mask points or None when the size is whatever the construction gives, predicted flagged)
RUNGS = [
    ("u2", 2, False), ("empty", 0, False), ("u3", 3, False), ("one", 1, False), ("u511", 511, False),
    ("f4", 4, True), ("u512", 512, False), ("two", 2, False), ("u513", 513, False), ("f899", 899, True),
    ("copies", None, False), ("f900", 900, True), ("u4100", 4100, False), ("f901", 901, True), ("empty2", 0, False),
    ("f4095", 4095, True), ("u9000", 9000, False), ("f4096", 4096, True), ("deep", None, False), ("f9000", 9000, True),
    ("owner", None, False),
]


def _O():
    import oracle_py as O
    return O


def _tiefree(seed, n):
    """n points in clusters of 3..9 with random integer offsets in a 700 x 700 box; the clusters' x and y ranges are
    disjoint, so the mask only drops what sits at the ends of the sort orders"""
    rng = np.random.RandomState(seed)
    k = n // 3 + 2
    size = rng.randint(3, 10, k)
    cy = rng.permutation(k) * 30000 + 1_000_000
    c = np.repeat(np.arange(k), size)[:n]
    x = c * 30000 + 1_000_000 + rng.randint(0, 700, n)
    y = cy[c] + rng.randint(0, 700, n)
    return x.astype(np.uint32), y.astype(np.uint32)


def _lattice(seed, n):
    """n points in clusters of 6..14 on a 50-spaced 4 x 4 lattice: exact distance ties and duplicates everywhere"""
    rng = np.random.RandomState(seed)
    k = n // 6 + 2
    size = rng.randint(6, 15, k)
    cy = rng.permutation(k) * 30000 + 1_000_000
    c = np.repeat(np.arange(k), size)[:n]
    x = c * 30000 + 1_000_000 + rng.randint(0, 4, n) * 50
    y = cy[c] + rng.randint(0, 4, n) * 50
    return x.astype(np.uint32), y.astype(np.uint32)


def _sparse(seed, n):
    """n points in a 2 500 x 2 500 box: some isolated, some not (for buckets the mask leaves one or two points of)"""
    rng = np.random.RandomState(seed)
    return (rng.randint(0, 2500, n) + 1_000_000).astype(np.uint32), (rng.randint(0, 2500, n) + 1_000_000).astype(np.uint32)


def _fit(gen, target, flagged, seed0):
    """the first seed (from seed0) and point count for which gen gives `target` points after the mask and the predicted
    flag equals `flagged`"""
    O = _O()
    for seed in range(seed0, seed0 + 200):
        n = target + 2
        for _ in range(12):
            x, y = gen(seed, n)
            keep = O.remove_isolated(x, y, W)
            if len(keep) == target:
                break
            n = max(1, n + target - len(keep))
        else:
            continue
        if len(keep) != target:
            continue
        if target >= 2 and (O.ahc_flags(x[keep], y[keep], W)[0] > 0) != flagged:
            continue
        return x, y
    raise AssertionError("no seed gives %d points, flagged=%s" % (target, flagged))


def _copies():
    """40 translated copies of one tie-free 16-point shape: every prefix-max distance of the shape's merge events is shared
    by >= 33 components of the bucket, so the global rank form gets tie groups of more than 32 events"""
    O = _O()
    for seed in range(100):
        rng = np.random.RandomState(1000 + seed)
        sx = rng.randint(0, 700, 16); sy = rng.randint(0, 700, 16)
        if O.ahc_flags(sx.astype(np.uint32), sy.astype(np.uint32), W)[0]:
            continue
        i = np.repeat(np.arange(40), 16)
        x = (np.tile(sx, 40) + i * 30000 + 1_000_000).astype(np.uint32)
        y = (np.tile(sy, 40) + i * 30000 + 5_000_000).astype(np.uint32)
        keep = O.remove_isolated(x, y, W)
        if O.ahc_flags(x[keep], y[keep], W)[0] == 0:
            return x, y
    raise AssertionError("no tie-free shape")


def _near_sorted(keys):
    """a same-chromosome bucket whose first mask pass leaves the points with y = keys in x order, every tenth of them
    twice: each kept point S has a left x-neighbour 1 away with a far y and a right x-neighbour with its own y but far
    in x, and both helpers fall to the mask; every tenth S also has a twin T 1..5 to its right with the same y.  So the
    second mask sort (by y) sorts `keys` nearly as they are -- the near-sorted keys of a real bucket
    (tests/golden/make_depth_exhausted_keys.py) exhaust the introsort depth there -- and the first sort has over
    3 x len(keys) elements (multi-CTA partition).  The twins survive the whole mask and cluster in two-point components,
    with a handful of distinct merge distances: large tie groups for the global rank form."""
    m = len(keys)
    base = 1_000_000 + np.arange(m, dtype=np.int64) * 10000
    k = keys.astype(np.int64)
    x = [base, base + 1, base + 5000]
    y = [k + 100_000_000, k, k]
    t = np.arange(0, m, 10)
    x.append(base[t] + 2 + (t // 10) % 5); y.append(k[t])
    return np.concatenate(x).astype(np.uint32), np.concatenate(y).astype(np.uint32)


def _golden_keys():
    g = np.load(os.path.join(GOLDEN, "depth_exhausted_sort_keys.npz"))
    return g["sort2"], g["sort3"]


def _rung_points(i, name, target, flagged):
    if name == "copies":
        return _copies()
    k2, k3 = _golden_keys()
    if name == "deep":
        return _near_sorted(k2)
    if name == "owner":
        return _near_sorted(np.concatenate([k2, k3.astype(np.int64) + 50_000_000, k2[:11000].astype(np.int64) + 100_000_000]))
    if name == "one":
        return _fit(_sparse, 1, False, 1000 * i)
    if flagged:
        return _fit(_lattice, target, True, 1000 * i)
    return _fit(_tiefree, target, False, 1000 * i)


def _bucket_ranks():
    O = _O()
    rank = np.zeros((NT + 1) ** 2, np.int32)
    O.olib().orc_bucket_rank_table(NT, O._names(types.SimpleNamespace(target_names=NAMES)), rank)
    return rank


def _pairs(buckets, seed):
    """PAIR_DTYPE table of [(p1_tid, p2_tid, x, y)], rows shuffled; inside a bucket the points keep their order (orig)"""
    from breakid_b200.api import PAIR_DTYPE
    rank = _bucket_ranks()
    rng = np.random.RandomState(seed)
    n = sum(len(b[2]) for b in buckets)
    p = np.zeros(n, PAIR_DTYPE)
    o = 0
    for t1, t2, x, y in buckets:
        s = slice(o, o + len(x))
        p["p1_tid"][s] = t1; p["p2_tid"][s] = t2
        p["bucket"][s] = rank[(t1 + 1) * (NT + 1) + (t2 + 1)]
        p["p1_chr_pos"][s] = x; p["p2_chr_pos"][s] = y
        o += len(x)
    p["p1_pos"] = p["p1_chr_pos"]; p["p2_pos"] = p["p2_chr_pos"]
    p["name_lo"] = rng.randint(0, 2 ** 63, n, dtype=np.int64).astype(np.uint64); p["name_hi"] = np.arange(n, dtype=np.uint64)
    p["p1_flag"] = 1 | rng.randint(0, 2, n) * 0x10; p["p2_flag"] = 1 | rng.randint(0, 2, n) * 0x10
    p["p1_strand"] = np.where(p["p1_flag"] & 0x10, ord("-"), ord("+")); p["p2_strand"] = np.where(p["p2_flag"] & 0x10, ord("-"), ord("+"))
    p["p1_mapq"] = 60; p["p2_mapq"] = 60
    p["cluster"] = -1
    p["orig"] = np.arange(n, dtype=np.uint32)
    return p[rng.permutation(n)]


class Ladder:
    def __init__(self):
        self.rungs = []          # (name, target, flagged, x, y)
        for i, (name, target, flagged) in enumerate(RUNGS):
            x, y = _rung_points(i, name, target, flagged)
            self.rungs.append((name, target, flagged, x, y))
        rng = np.random.RandomState(77)
        self.fillers = [_tiefree(50_000 + i, int(rng.randint(4, 9))) for i in range(N_FILLERS)]
        # tid pairs in ascending name order, so the ladder's buckets keep their order on both sides; the two big buckets
        # are same-chromosome ones
        names = [(a, b) for a in range(-1, NT) for b in range(-1, NT) if a != b]
        same = iter([(t, t) for t in range(NT)])
        self.tids = []
        k = 0
        for name, *_ in self.rungs:
            if name in ("deep", "owner"):
                self.tids.append(next(same))
            else:
                self.tids.append(names[k]); k += 1
        self.filler_tids = names[k:k + N_FILLERS]
        assert len(self.filler_tids) == N_FILLERS

    def buckets(self, only=None):
        out = [(t[0], t[1], r[3], r[4]) for t, r in zip(self.tids, self.rungs) if only is None or r[0] == only]
        if only is None:
            out += [(t[0], t[1], x, y) for t, (x, y) in zip(self.filler_tids, self.fillers)]
        return out

    def predicted_flagged_components(self, only=None):
        O = _O()
        f = 0
        for _, _, x, y in self.buckets(only):
            keep = O.remove_isolated(x, y, W)
            if len(keep) >= 2:
                f += O.ahc_flags(x[keep], y[keep], W)[0]
        return f


@pytest.fixture(scope="module")
def ladder():
    return Ladder()


# ------------------------------------------------------------------------------------------------ CPU
def test_rungs_hit_their_sizes(ladder):
    O = _O()
    sizes = {}
    for name, target, flagged, x, y in ladder.rungs:
        m = len(O.remove_isolated(x, y, W))
        sizes[name] = m
        if target is not None:
            assert m == target, (name, m)
    # every form on both sides of its boundary
    assert sizes["u511"] < RG_LO <= sizes["u512"] < sizes["u513"] and sizes["u9000"] >= EXACT_LO
    assert sizes["f899"] < SMEM_HI <= sizes["f900"] and sizes["f4095"] < EXACT_LO <= sizes["f4096"]
    assert sizes["copies"] >= RG_LO
    assert len(ladder.buckets()) > 256
    assert all(len(O.remove_isolated(x, y, W)) < RG_LO for x, y in ladder.fillers)
    for name in ("deep", "owner"):
        x = [r for r in ladder.rungs if r[0] == name][0][3]
        assert len(x) > 49152, name
    assert len([r for r in ladder.rungs if r[0] == "owner"][0][3]) > 190_000


def test_predictor_marks_rungs_as_designed(ladder):
    O = _O()
    for name, target, flagged, x, y in ladder.rungs:
        keep = O.remove_isolated(x, y, W)
        f = O.ahc_flags(x[keep], y[keep], W)[0] if len(keep) >= 2 else 0
        assert (f > 0) == flagged, (name, f)
    # three points cannot be flagged: the only merged node's row has one entry, so there is no tie to break
    rng = np.random.RandomState(3)
    for _ in range(200):
        x = (rng.randint(0, 3, 3) * 50).astype(np.uint32); y = (rng.randint(0, 3, 3) * 50).astype(np.uint32)
        assert O.ahc_flags(x, y, W) == (0, 0)


def test_copies_share_one_shape(ladder):
    """>= 33 components of the copies rung are the same shape after the mask (tie groups of > 32 events)"""
    O = _O()
    x, y = [r[3:] for r in ladder.rungs if r[0] == "copies"][0]
    keep = O.remove_isolated(x, y, W)
    xs, ys = x[keep].astype(np.int64), y[keep].astype(np.int64)
    copy = (xs - 1_000_000) // 30000
    shapes = {}
    for c in np.unique(copy):
        m = copy == c
        shapes.setdefault(tuple(sorted(zip(xs[m] - c * 30000, ys[m] - c * 30000))), []).append(c)
    assert max(len(v) for v in shapes.values()) >= 33


def test_deep_bucket_exhausts_introsort_depth_in_second_mask_sort(ladder):
    """the second sort of the mask on the 'deep' bucket hits the heapsort fallback (the is_heap kernel on the device)"""
    O = _O()
    sys.path.insert(0, GOLDEN)
    from make_depth_exhausted_keys import mask_pass
    x, y = [r[3:] for r in ladder.rungs if r[0] == "deep"][0]
    v = mask_pass(O.sort_perm(x).astype(np.int64), x, y, THR)
    k2 = np.ascontiguousarray(y[v])
    assert len(x) > 49152 and len(k2) > len(_golden_keys()[0])
    h0 = O.heapsort_count()
    assert np.array_equal(O.sort_perm(k2, model=True), O.sort_perm(k2))
    assert O.heapsort_count() > h0


def test_model_equals_literal_ahc_on_small_rungs(ladder):
    O = _O()
    n_checked = {True: 0, False: 0}
    for name, target, flagged, x, y in ladder.rungs:
        keep = O.remove_isolated(x, y, W)
        if len(keep) > 1500 or len(keep) < 2:
            continue
        xs, ys = x[keep], y[keep]
        a = O.cluster(0, xs, ys, W); b = O.cluster(0, xs, ys, W, model=True)
        assert all(np.array_equal(p, q) for p, q in zip(a[:2], b[:2])) and a[2] == b[2], name
        n_checked[flagged] += 1
    assert n_checked[True] >= 4 and n_checked[False] >= 5


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gpu():
    import torch
    from breakid_b200 import api
    from breakid_b200.dist import GpuEngine
    c = api.Context(TLEN, NAMES, device=0)
    yield GpuEngine(c, torch.device("cuda", 0))
    c.close()


def _run_device(eng, pairs, mode):
    import torch
    eng.set_pairs(torch.from_numpy(pairs.view(np.uint8).reshape(-1, 64).copy()).cuda())
    eng.cluster(W, mode)


def _expected(pairs, mode):
    """stage-1 survivors, stage-2 members and the cluster summaries, from the oracle"""
    import torch
    from oracle_engine import OracleEngine
    O = _O()
    oe = OracleEngine(types.SimpleNamespace(target_names=NAMES, target_len=np.array(TLEN, np.uint32)), ahc_model=True)
    oe.set_pairs(torch.from_numpy(pairs.view(np.uint8).reshape(-1, 64).copy()))
    oe.cluster(W, mode)
    sp = oe.pairs                                  # sorted like the device's table: orig there = index here
    s1, s2 = [], []
    bounds = np.flatnonzero(np.diff(sp["bucket"])) + 1
    for k, (s, e) in enumerate(zip(np.r_[0, bounds], np.r_[bounds, len(sp)])):
        x, y = sp["p1_chr_pos"][s:e], sp["p2_chr_pos"][s:e]
        keep = O.remove_isolated(x, y, W)
        s1 += [(s + i, k, -1) for i in keep]
        if len(keep) >= 2:
            ci, cl, _ = O.cluster(mode, x[keep], y[keep], W, model=True)
            s2 += [(s + keep[i], k, c) for i, c in zip(ci, cl)]
    return np.array(s1, np.int64).reshape(-1, 3), np.array(s2, np.int64).reshape(-1, 3), oe.clusters().numpy()


def _cols(p):
    return np.stack([p["orig"].astype(np.int64), p["bucket"].astype(np.int64), p["cluster"].astype(np.int64)], 1)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_ladder_in_one_call_matches_oracle(ladder, gpu, mode):
    pairs = _pairs(ladder.buckets(), seed=mode)
    _run_device(gpu, pairs, mode)
    e1, e2, ecl = _expected(pairs, mode)
    g1 = _cols(gpu.ctx.fetch_pairs(1))
    g2 = _cols(gpu.ctx.fetch_pairs(2))
    assert np.array_equal(g1[:, :2], e1[:, :2])
    if mode == 1:                                  # -fast: compared after the (bucket, cluster, member) lexsort
        g2 = g2[np.lexsort((g2[:, 0], g2[:, 2], g2[:, 1]))]
        e2 = e2[np.lexsort((e2[:, 0], e2[:, 2], e2[:, 1]))]
    assert len(e2) > 20000
    assert np.array_equal(g2, e2)
    gcl = gpu.clusters().cpu().numpy()
    assert gcl.shape == ecl.shape and gcl.shape[0] > 1000
    assert gcl.tobytes() == ecl.tobytes()


_FLAG_LINE = re.compile(r"ncomp (\d+) flagged (\d+) \(points (\d+)\) max comp (\d+) merges (\d+) points (\d+) buckets (\d+)")


def flagged_witness(text):
    """[(ncomp, flagged components, points, buckets)] of every AHC call whose BKID_DEBUG_TIMING output is in `text`"""
    return [(int(m[0]), int(m[1]), int(m[5]), int(m[6])) for m in _FLAG_LINE.findall(text)]


@pytest.mark.gpu
def test_each_rung_takes_its_predicted_form(ladder, gpu, monkeypatch, capfd):
    O = _O()
    monkeypatch.setenv("BKID_DEBUG_TIMING", "1")
    for i, (name, target, flagged, x, y) in enumerate(ladder.rungs):
        capfd.readouterr()
        _run_device(gpu, _pairs(ladder.buckets(only=name), seed=100 + i), 0)
        seen = flagged_witness(capfd.readouterr().err)
        n = len(O.remove_isolated(x, y, W))
        if n == 0:
            assert seen == [], name
            continue
        assert len(seen) == 1 and seen[0][2] == n and seen[0][3] == 1, (name, seen)
        pred = ladder.predicted_flagged_components(only=name)
        assert seen[0][1] == pred and (pred > 0) == flagged, (name, seen, pred)


@pytest.mark.gpu
def test_ladder_reaches_every_form_in_one_call(ladder, gpu, monkeypatch, capfd):
    from breakid_b200 import api
    monkeypatch.setenv("BKID_DEBUG_TIMING", "1")
    pairs = _pairs(ladder.buckets(), seed=0)
    capfd.readouterr()
    api.profile_kernels(True)
    try:
        api.profile_report()
        _run_device(gpu, pairs, 0)
        rep = api.profile_report()
    finally:
        api.profile_kernels(False)
    seen = flagged_witness(capfd.readouterr().err)
    assert len(seen) == 1
    pred = ladder.predicted_flagged_components()
    assert seen[0][1] == pred and pred > 0
    assert seen[0][3] == len(ladder.buckets()) > 256
    for k in ("is_big_part", "is_big_swap", "is_heap", "ahc_replay_rank", "ahc_replay_smem", "ahc_bucket_exact",
              "ahc_rg_prepare", "ahc_rg_sortkeys", "ahc_rg_rank_sorted", "ahc_rg_heads", "ahc_rg_ties", "ahc_rg_write"):
        assert rep.get(k, (0, 0.0))[0] > 0, k
