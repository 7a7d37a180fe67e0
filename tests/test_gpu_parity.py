"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs.  Bit-exact: everything on this path is integer / byte / index work, and the FP64 parts
(insert sd, AHC distances) are required to be bit-identical too."""
import os

import numpy as np
import pytest

from conftest import lattice_points

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx1():
    from breakid_b200 import api
    c = api.Context([1000000], ["chr1"], device=0)
    yield c
    c.close()


def test_sort_replay_matches_std_sort(ctx1):
    import oracle_py as O
    rng = np.random.RandomState(0)
    sizes = [0, 1, 2, 3, 15, 16, 17, 18, 31, 32, 33, 50, 100, 257, 1000, 5000, 40000]
    bad = []
    for trial in range(120):
        n = sizes[trial % len(sizes)] if trial % 2 else int(rng.randint(0, 600))
        kind = trial % 6
        if kind == 0: key = rng.randint(0, 5, n)
        elif kind == 1: key = rng.randint(0, max(1, n // 3 + 1), n)
        elif kind == 2: key = np.sort(rng.randint(0, n + 1, n))
        elif kind == 3: key = np.sort(rng.randint(0, n + 1, n))[::-1].copy()
        elif kind == 4: key = rng.randint(0, 2 ** 32, n)
        else: key = np.repeat(rng.randint(0, 1000, n // 4 + 1), 4)[:n]
        key = key.astype(np.uint32)
        a = O.sort_perm(key)
        b = ctx1.op_sort_perm(key)
        if not np.array_equal(a, b):
            bad.append((trial, n, kind))
    assert not bad, bad


def test_sort_replay_depth_limit(ctx1):
    """median-of-3 killer sequences exhaust the introsort depth budget -> heapsort fallback"""
    import oracle_py as O

    def killer(n):
        k = n // 2; a = np.zeros(n, np.uint32)
        for i in range(1, k + 1):
            if i % 2: a[i - 1] = i; a[i] = k + i
            a[k + i - 1] = 2 * i
        return a
    for n in (64, 1000, 4096, 20000):
        key = killer(n)
        assert np.array_equal(O.sort_perm(key), ctx1.op_sort_perm(key)), n


def test_sort_replay_big_segments(ctx1):
    """segments above 48 K elements are partitioned by several CTAs (is_big_part / is_big_swap): tile boundaries, heavy ties,
    sorted / reversed / merged-runs inputs, the depth-exhausted heapsort, against std::sort"""
    import oracle_py as O
    rng = np.random.RandomState(12)

    def killer(n):
        k = n // 2; a = np.zeros(n, np.uint32)
        for i in range(1, k + 1):
            if i % 2: a[i - 1] = i; a[i] = k + i
            a[k + i - 1] = 2 * i
        return a
    cases = []
    for n in (16385, 49152, 49153, 49154, 51201, 53249, 65536, 70001, 300000, 1 << 20):
        cases += [("ties5", rng.randint(0, 5, n)), ("ties", rng.randint(0, n // 3 + 1, n)), ("sorted", np.sort(rng.randint(0, n + 1, n))),
                  ("reversed", np.sort(rng.randint(0, n + 1, n))[::-1].copy()), ("random", rng.randint(0, 2 ** 32, n)),
                  ("runs", np.concatenate([np.sort(rng.randint(0, 2 ** 31, n - n // 2)), np.sort(rng.randint(0, 2 ** 31, n // 2))])),
                  ("const", np.full(n, 7))]
    cases += [("killer", killer(n)) for n in (30000, 60000, 100000)]
    bad = []
    for name, key in cases:
        key = key.astype(np.uint32)
        if not np.array_equal(O.sort_perm(key), ctx1.op_sort_perm(key)):
            bad.append((name, len(key)))
    assert not bad, bad


def test_sort_replay_depth_exhausted_segments(ctx1):
    """keys of a real near-sorted bucket (tests/golden/make_depth_exhausted_keys.py): introsort runs out of depth on segments
    of ~4 000 elements, which is_heap finishes with the literal heapsort out of shared memory"""
    import oracle_py as O
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "depth_exhausted_sort_keys.npz"))
    for name in ("sort2", "sort3"):
        key = g[name]
        assert np.array_equal(O.sort_perm(key), ctx1.op_sort_perm(key)), name
        rep = np.concatenate([key, key[::-1], key])          # the same with every key three times: ties inside the heapsort
        assert np.array_equal(O.sort_perm(rep), ctx1.op_sort_perm(rep)), name


def test_remove_isolated_big_buckets(ctx1):
    """the mask over buckets of 50 K .. 400 K pairs (three sort replays through the multi-CTA partition) against the oracle"""
    import oracle_py as O
    rng = np.random.RandomState(13)
    for n, span in ((50000, 3_000_000), (120000, 40_000_000), (400000, 100_000_000)):
        x = rng.randint(0, span, n).astype(np.uint32); y = rng.randint(0, span, n).astype(np.uint32)
        k = n // 10                                       # planted dense groups + exact duplicates
        x[:k] = (rng.randint(0, 50, k) * 1000 + rng.randint(0, 3, k) * 50).astype(np.uint32); y[:k] = (rng.randint(0, 50, k) * 1000 + rng.randint(0, 3, k) * 50).astype(np.uint32)
        p = rng.permutation(n); x = x[p]; y = y[p]
        a = O.remove_isolated(x, y, 1243.15); b = ctx1.op_remove_isolated(x, y, 1243.15)
        assert np.array_equal(a, b), (n, len(a), len(b))


def test_remove_isolated(ctx1):
    import oracle_py as O
    rng = np.random.RandomState(1)
    bad = []
    for trial in range(150):
        n = int(rng.randint(0, 400)); kind = trial % 4
        x, y = lattice_points(rng, n, kind)
        w = float(rng.choice([120.7, 260.2, 99.0, 1243.15]))
        a = O.remove_isolated(x, y, w); b = ctx1.op_remove_isolated(x, y, w)
        if not np.array_equal(a, b):
            bad.append((trial, n, kind, len(a), len(b)))
    assert not bad, bad


@pytest.mark.parametrize("mode", [0, 1])
def test_cluster_ops(ctx1, mode):
    import oracle_py as O
    rng = np.random.RandomState(2 + mode)
    bad = []
    for trial in range(200):
        n = int(rng.randint(2, 120)); kind = trial % 4
        x, y = lattice_points(rng, n, kind)
        w = float(rng.choice([120.7, 260.2, 99.0, 1243.15]))
        keep = O.remove_isolated(x, y, w)
        xs = np.ascontiguousarray(x[keep]); ys = np.ascontiguousarray(y[keep])
        if len(xs) < 2:
            continue
        ei, ec, er = O.cluster(mode, xs, ys, w)
        gi, gc, gr = ctx1.op_cluster(mode, xs, ys, w)
        if mode == 0:
            same = np.array_equal(ei, gi) and np.array_equal(ec, gc) and er == gr
        else:   # -fast: the oracle lists members in p1 order, the device groups them by cluster id
            o1 = np.lexsort((ei, ec)); o2 = np.lexsort((gi, gc))
            same = np.array_equal(ei[o1], gi[o2]) and np.array_equal(ec[o1], gc[o2]) and er == gr
        if not same:
            bad.append((trial, kind, len(xs), len(ei), len(gi), er, gr))
    assert not bad, bad


def test_ahc_unsorted_heavy_ties(ctx1):
    """util_cluster interface on arbitrary (unsorted) input with exact distance ties and duplicates"""
    import oracle_py as O
    rng = np.random.RandomState(9)
    bad = []
    for trial in range(150):
        n = int(rng.randint(2, 70)); kind = trial % 3
        if kind == 0:
            x = rng.randint(0, 5, n) * 50; y = rng.randint(0, 5, n) * 50
        elif kind == 1:
            k = max(1, n // 6); a = rng.randint(0, k, n); x = a * 1000 + rng.randint(0, 4, n) * 50; y = (a % 2) * 800 + rng.randint(0, 4, n) * 50
        else:
            k = max(1, n // 5); a = rng.randint(0, k, n); x = a * 500 + rng.randint(0, 3, n) * 50; y = rng.randint(0, 3, n) * 50 + (a % 3) * 400
        thr = float(rng.choice([60, 120, 200, 260]))
        x = x.astype(np.uint32); y = y.astype(np.uint32)
        ei, ec, er = O.cluster(0, x, y, thr)
        gi, gc, gr = ctx1.op_cluster(0, x, y, thr)
        if not (np.array_equal(ei, gi) and np.array_equal(ec, gc) and er == gr):
            bad.append((trial, kind, n, thr))
    assert not bad, bad


def _ctx_for(hb, **kw):
    from breakid_b200 import api
    c = api.Context(hb.target_len, hb.target_names, device=0, **kw)
    c.push(hb)
    return c


def test_insert_stats_and_classify(small_data):
    import oracle_py as O
    d, hb, nibs = small_data
    c = _ctx_for(hb)
    m, s = c.insert_stats()
    om, osd, S, n, T = O.insert_stats(hb)
    assert (m, s) == (om, osd)
    cls = c.fetch_class(hb.n)
    f = hb.cols["flag"].astype(np.int64); q = hb.cols["mapq"].astype(np.int64)
    ins = ((f & 1) != 0) & ((f & 2) != 0) & ((f & (0x4 | 0x100 | 0x200 | 0x400)) == 0)
    cand = (q >= 20) & ((f & 0x400) == 0) & ((f & 0x100) == 0) & ((f & 1) != 0) & ((f & 2) == 0)
    dep = (q > 0) & ((f & 0x400) == 0) & ((f & 1) != 0)
    assert np.array_equal((cls & 1) != 0, ins)
    assert np.array_equal((cls & 2) != 0, cand)
    assert np.array_equal((cls & 4) != 0, dep)
    c.close()


def test_insert_sd_adversarial():
    """the truncating accumulator: huge insert sizes push the running total through many binades"""
    import oracle_py as O
    from breakid_b200 import api
    rng = np.random.RandomState(3)
    for case in range(4):
        n = [5000, 70000, 300000, 20000][case]
        isz = rng.randint(-2000, 2000, n).astype(np.int32)
        if case == 1: isz = (rng.randint(0, 2, n) * rng.randint(0, 3000000, n)).astype(np.int32)
        if case == 3: isz = rng.randint(-20000000, 20000000, n).astype(np.int32)     # leaves the closed form (t >= 2^52) -> literal replay
        flag = np.where(rng.rand(n) < 0.9, 99, rng.choice([97, 1123, 355, 4], n)).astype(np.uint16)
        z = np.zeros(n, np.int32)
        hb = api.HostBatch({"flag": flag, "mapq": np.full(n, 60, np.uint8), "tid": z, "pos": np.arange(n, dtype=np.int32), "mtid": z, "mpos": z,
                            "isize": isz, "endpos": np.arange(n, dtype=np.int32) + 100}, np.arange(2 * n, dtype=np.uint64),
                           {"sa_rec": np.zeros(0, np.uint32), "cig_off": np.zeros(1, np.uint32), "cig_ops": np.zeros(0, np.uint32),
                            "sa_off": np.zeros(1, np.uint32), "sa_txt": np.zeros(0, np.uint8)}, [1000000000], ["chr1"])
        c = _ctx_for(hb)
        got = c.insert_stats()
        exp = O.insert_stats(hb)
        assert got == exp[:2], (case, got, exp)
        c.close()


def test_scan_pairs(small_data):
    import oracle_py as O
    d, hb, nibs = small_data
    c = _ctx_for(hb)
    m, s = c.insert_stats()
    w = O.dist(m, s)
    n = c.scan(w)
    got = c.fetch_pairs(0)
    exp = O.scan(hb, 20, w)
    assert n == len(exp)
    for k in exp.dtype.names:
        assert np.array_equal(got[k], exp[k]), k
    c.close()


@pytest.mark.parametrize("mode", [0, 1])
def test_whole_path(small_data, mode):
    import oracle_py as O
    d, hb, nibs = small_data
    c = _ctx_for(hb, fast=mode)
    for t, (p, l) in enumerate(nibs):
        c.set_nib(t, p, l)
    mean, sd, dist, ncall = c.run()
    got = c.fetch_clusters()
    om, osd, od, exp = O.run(hb, nibs, mode=mode)
    assert (mean, sd, dist) == (om, osd, od)
    assert len(got) == len(exp), (len(got), len(exp))
    for k in exp.dtype.names:
        assert np.array_equal(got[k], exp[k]), (k, got[k], exp[k])
    assert len(got) >= 5
    c.close()


@pytest.mark.parametrize("mode", [0, 1])
def test_whole_path_config1(config1_data, mode):
    import oracle_py as O
    d, hb, nibs = config1_data
    c = _ctx_for(hb, fast=mode)
    for t, (p, l) in enumerate(nibs):
        c.set_nib(t, p, l)
    mean, sd, dist, ncall = c.run()
    got = c.fetch_clusters()
    om, osd, od, exp = O.run(hb, nibs, mode=mode)
    assert (mean, sd, dist) == (om, osd, od)
    assert got.tobytes() == exp.tobytes()
    assert len(got) == 10          # every planted SV is called
    c.close()


def test_batched_push_equals_single_push(small_data):
    """records arriving in several batches (streaming decode) give the same result"""
    from breakid_b200 import api
    d, hb, nibs = small_data
    c1 = _ctx_for(hb)
    r1 = c1.run(); g1 = c1.fetch_clusters()
    c2 = api.Context(hb.target_len, hb.target_names, device=0)
    cuts = [0, hb.n // 3, hb.n // 2 + 7, hb.n]
    for a, b in zip(cuts[:-1], cuts[1:]):
        sa = hb.side["sa_rec"]; lo = np.searchsorted(sa, a); hi = np.searchsorted(sa, b)
        co, so, oo = hb.side["cig_off"], hb.side["sa_off"], hb.side["oc_off"]
        part = api.HostBatch({k: v[a:b] for k, v in hb.cols.items()}, hb.name_hash[2 * a:2 * b],
                             {"sa_rec": sa[lo:hi] - a, "cig_off": co[lo:hi + 1] - co[lo], "cig_ops": hb.side["cig_ops"][co[lo]:co[hi]],
                              "sa_off": so[lo:hi + 1] - so[lo], "sa_txt": hb.side["sa_txt"][so[lo]:so[hi]],
                              "oc_off": oo[lo:hi + 1] - oo[lo], "oc_txt": hb.side["oc_txt"][oo[lo]:oo[hi]]}, hb.target_len, hb.target_names)
        c2.push(part)
    r2 = c2.run(); g2 = c2.fetch_clusters()
    assert r1 == r2 and g1.tobytes() == g2.tobytes()
    c1.close(); c2.close()


@pytest.mark.parametrize("mode", ["ahc", "fast"])
def test_driver_call_files_match_reference_binary(tmp_path, mode):
    """drop-in check: the BreakID driver (GPU) and the reference CPU binary write byte-identical
    _fusion.txt / _fusion_all.txt / _params.txt on the same BAM + nib + refGene"""
    import os
    import subprocess
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio, synth
    ref = O.have_ref()
    cfg = synth.SynthConfig(chrom_lens=[300000, 200000, 150000], n_tra=3, n_inv=2, n_dup=2, n_del=2, seed=21, sv_jitter=1)
    d = synth.generate(cfg)
    paths = bamio.write_dataset(str(tmp_path), d, genes_per_mb=25.0)
    R.index(paths["bam"])
    flags = ["-all"] + (["-fast"] if mode == "fast" else [])
    if ref:
        O.ref_install_refgene(paths["refgene"])
        r = O.ref_run_binary(paths["bam"], str(tmp_path / "ref"), paths["nib"], fast=(mode == "fast"))
        assert r.returncode == 0, r.stderr[-500:]
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    g = subprocess.run([drv, "-i", paths["bam"], "-o", str(tmp_path / "gpu"), "-n", paths["nib"], "-r", paths["refgene"]] + flags,
                       timeout=600, capture_output=True, text=True)
    assert g.returncode == 0, g.stderr[-500:]
    if not ref:
        R.match_oracle(str(tmp_path / "gpu"), d, mode=int(mode == "fast"))
        assert len(R.fusion_all_rows(str(tmp_path / "gpu"))) >= 5
        return
    for suffix in ("_fusion.txt", "_fusion_all.txt"):
        a = open(str(tmp_path / "ref") + suffix).read()
        b = open(str(tmp_path / "gpu") + suffix).read()
        assert a == b, suffix
        assert len(a.splitlines()) >= (6 if suffix == "_fusion_all.txt" else 1)
    pa = open(str(tmp_path / "ref") + "_params.txt").read().replace(str(tmp_path / "ref"), "X")
    pb = open(str(tmp_path / "gpu") + "_params.txt").read().replace(str(tmp_path / "gpu"), "X")
    assert pa == pb


@pytest.mark.parametrize("mode", ["ahc", "fast"])
def test_driver_matches_stored_reference_call_files(tmp_path, mode):
    """the BreakID driver on the dataset of tests/golden/make_golden.py against the files the reference binary wrote on it
    (mini_ref_<mode>_fusion.txt, mini_ref_<mode>_fusion_all.txt, mini_ref_params.txt): byte for byte, gene annotation and
    the gene-fusion filter included, with no reference needed"""
    import os
    import subprocess
    import reference_calls as R
    from breakid_b200 import bamio, synth
    G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    cfg = synth.SynthConfig(chrom_lens=[120000, 90000], n_tra=2, n_inv=1, n_dup=1, n_del=1, seed=33, min_sv_sep=5000, sv_jitter=1,
                            chimeric_frac=0.02)                                   # make_golden.mini_cfg()
    d = synth.generate(cfg)
    z = np.load(os.path.join(G, "mini.npz"))                                     # the records the reference ran on
    assert all(np.array_equal(d.cols[k].numpy().view(z["col_" + k].dtype), z["col_" + k]) for k in ("flag", "mapq", "tid", "pos", "mtid", "mpos", "isize", "endpos"))
    assert np.array_equal(synth.name_hash_ids(d.cols["name_id"]).numpy().view(np.uint64).reshape(-1), z["name_hash"])
    paths = bamio.write_dataset(str(tmp_path), d, random_qual=False, genes_per_mb=40.0)
    assert open(paths["refgene"]).read() == open(os.path.join(G, "mini_refGene.txt")).read()
    R.index(paths["bam"])
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    out = str(tmp_path / mode)
    g = subprocess.run([drv, "-i", paths["bam"], "-o", out, "-n", paths["nib"], "-r", paths["refgene"], "-all"] + (["-fast"] if mode == "fast" else []),
                       timeout=600, capture_output=True, text=True)
    assert g.returncode == 0, g.stderr[-500:]
    for suffix in ("_fusion.txt", "_fusion_all.txt"):
        assert open(out + suffix).read() == open(os.path.join(G, "mini_ref_%s%s" % (mode, suffix))).read(), suffix
    exp = open(os.path.join(G, "mini_ref_params.txt")).read()                     # stored from the AHC run (out_file TMP/ahc)
    assert open(out + "_params.txt").read().replace(str(tmp_path), "TMP") == exp.replace("TMP/ahc", "TMP/" + mode)


@pytest.mark.parametrize("mode", [0, 1])
def test_shard_entry_points_single_rank(small_data, mode):
    """the multi-GPU orchestration (breakid_b200.dist.run_sharded) on one rank, through the bkid_shard_* ABI,
    equals the monolithic bkid_run and the oracle"""
    import torch
    import oracle_py as O
    from breakid_b200 import api
    from breakid_b200.dist import GpuEngine, run_sharded
    d, hb, nibs = small_data
    c = _ctx_for(hb, fast=mode)
    for t, (p, l) in enumerate(nibs):
        c.set_nib(t, p, l)
    mean, sd, dist_, out = run_sharded(GpuEngine(c, torch.device("cuda", 0)), hb.n, mode=mode)
    om, osd, od, exp = O.run(hb, nibs, mode=mode)
    assert (mean, sd, dist_) == (om, osd, od)
    assert out.tobytes() == exp.tobytes()
    c.close()


def test_sa_rows_match_oracle(small_data):
    """device split-read evidence rows (CIGAR / SA arithmetic) are byte-identical to the oracle's"""
    import ctypes as C
    import torch
    from breakid_b200.dist import GpuEngine
    from oracle_engine import OracleEngine
    d, hb, nibs = small_data
    c = _ctx_for(hb)
    got = GpuEngine(c, torch.device("cuda", 0)).sa_rows().cpu().numpy()
    exp = OracleEngine(hb).sa_rows().numpy()
    assert got.shape == exp.shape and got.shape[0] > 50
    assert np.array_equal(got, exp)
    c.close()


def test_ahc_large_bucket_rank_form(ctx1):
    """one bucket with > 4096 points (global-memory rank-form replay) incl. exact cross-component ties; the
    oracle side is the component model (proven equal to the literal O(N^3) restatement in the CPU suite)"""
    import oracle_py as O
    rng = np.random.RandomState(123)
    for n, spread in ((5000, 40), (9000, 6)):
        k = n // 12
        cx = np.sort(rng.choice(np.arange(0, 40_000_000, 5000), k, replace=False)); cy = rng.randint(0, 40_000_000, k)
        a = rng.randint(0, k, n)
        x = (cx[a] + rng.randint(0, spread, n) * 7).astype(np.uint32); y = (cy[a] + rng.randint(0, spread, n) * 7).astype(np.uint32)
        o = np.argsort(x, kind="stable"); x = np.ascontiguousarray(x[o]); y = np.ascontiguousarray(y[o])
        ei, ec, er = O.cluster(0, x, y, 1243.15, model=True)
        gi, gc, gr = ctx1.op_cluster(0, x, y, 1243.15)
        assert np.array_equal(ei, gi) and np.array_equal(ec, gc) and er == gr, n


def _adversarial_sa_batch(seed, n=4000):
    """records whose CIGAR / SA / OC fields exercise every branch of the split-read arithmetic: merged and
    =/X ops, H/I/D/N ops, all-clip cigars, OC tags, multi-entry SA tags, leading zeros, minus strands, odd
    chromosome names, duplicate / unpaired / secondary flags"""
    from breakid_b200 import api
    rng = np.random.RandomState(seed)
    ops = "MIDNSHP=X"

    def rand_cigar_text(simple):
        if simple:
            k = int(rng.randint(1, 149)); j = int(rng.randint(-12, 13))
            pats = ["%dM%dS" % (k, 150 - k), "%dS%dM" % (150 - k, k), "%dS%dM" % (max(1, k + j), max(1, 150 - k - j)), "%dM%dS" % (max(1, 150 - k - j), max(1, k + j)),
                    "0%dM%dS" % (k, 150 - k), "%dM%dM%dS" % (k // 2 + 1, k - k // 2, 150 - k), "%d=%dS" % (k, 150 - k), "%dX%dS" % (k, 150 - k), "%dS%dS" % (k, 150 - k)]
            return pats[rng.randint(0, len(pats))]
        return "".join("%d%s" % (rng.randint(0, 160), ops[rng.randint(0, len(ops))]) for _ in range(rng.randint(1, 5)))

    def text_to_bam(t):
        out, num = [], ""
        for ch in t:
            if ch.isdigit():
                num += ch
            else:
                out.append((int(num or 0) << 4) | ops.index(ch)); num = ""
        return out
    tid = np.sort(rng.randint(0, 3, n)).astype(np.int32)
    pos = np.zeros(n, np.int32)
    for t in range(3):
        m = tid == t
        pos[m] = np.sort(rng.randint(0, 5000, m.sum()))
    flag = rng.choice([99, 147, 355, 99 | 0x400, 98, 83, 163, 99 | 0x800, 355 | 0x10], n).astype(np.uint16)
    names = rng.randint(0, n // 3, n)                         # names repeat: primary / 0x100 partners
    nh = np.zeros(2 * n, np.uint64)
    from breakid_b200 import synth
    for i in range(n):
        nh[2 * i], nh[2 * i + 1] = synth.name_hash_py(synth.name_of(int(names[i])))
    sa_rec, cig_off, cig_ops, sa_off, sa_txt, oc_off, oc_txt = [], [0], [], [0], b"", [0], b""
    endpos = pos + 1
    chrs = ["chr1", "chr2", "chr3", "chrX", "chr07", "chrUn", "1"]
    for i in range(n):
        if rng.rand() < 0.6:
            own = text_to_bam(rand_cigar_text(rng.rand() < 0.7))[:6] or [(100 << 4)]
            sa_rec.append(i)
            cig_ops += own; cig_off.append(len(cig_ops))
            ref = sum(c >> 4 for c in own if (c & 15) in (0, 2, 3, 7, 8))
            endpos[i] = pos[i] + ref if not (flag[i] & 4) else pos[i] + 1
            ent = "%s,%s%d,%s,%s,60,0;" % (chrs[rng.randint(0, len(chrs))], "0" if rng.rand() < 0.05 else "", rng.randint(1, 6000), "+-"[rng.randint(0, 2)], rand_cigar_text(rng.rand() < 0.8))
            if rng.rand() < 0.15:
                ent += "chr2,77,+,50M100S,60,0;"
            if rng.rand() < 0.03:
                ent = "chr1,5"                                   # fewer than 4 fields: ignored
            sa_txt += ent.encode(); sa_off.append(len(sa_txt))
            if rng.rand() < 0.15:
                oc_txt += rand_cigar_text(rng.rand() < 0.8).encode()
            oc_off.append(len(oc_txt))
    z = np.zeros(n, np.int32)
    hb = api.HostBatch({"flag": flag, "mapq": np.full(n, 60, np.uint8), "tid": tid, "pos": pos, "mtid": tid, "mpos": pos, "isize": z, "endpos": endpos.astype(np.int32)}, nh,
                       {"sa_rec": np.array(sa_rec, np.uint32), "cig_off": np.array(cig_off, np.uint32), "cig_ops": np.array(cig_ops, np.uint32), "sa_off": np.array(sa_off, np.uint32),
                        "sa_txt": np.frombuffer(sa_txt, np.uint8), "oc_off": np.array(oc_off, np.uint32), "oc_txt": np.frombuffer(oc_txt or b"", np.uint8)},
                       [10000, 10000, 10000], ["chr1", "chr2", "chr3"])
    return hb


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_sa_rows_adversarial_cigars(seed):
    """CIGAR / SA-tag arithmetic on hostile inputs: device evidence rows == oracle rows, byte for byte"""
    import torch
    from breakid_b200.dist import GpuEngine
    from oracle_engine import OracleEngine
    hb = _adversarial_sa_batch(seed)
    c = _ctx_for(hb)
    got = GpuEngine(c, torch.device("cuda", 0)).sa_rows().cpu().numpy()
    exp = OracleEngine(hb).sa_rows().numpy()
    assert got.shape == exp.shape and got.shape[0] > 1000
    bad = np.nonzero((got != exp).any(axis=1))[0]
    assert len(bad) == 0, (len(bad), bad[:5], got[bad[:2]], exp[bad[:2]])
    ok = got[:, 84]
    assert ok.sum() > 50            # some rows are real evidence
    c.close()


def test_degenerate_inputs():
    """empty batch, no candidates, no SA records: every stage returns cleanly with nothing to call"""
    from breakid_b200 import api
    z32 = np.zeros(0, np.int32)
    empty = api.HostBatch({"flag": np.zeros(0, np.uint16), "mapq": np.zeros(0, np.uint8), "tid": z32, "pos": z32, "mtid": z32, "mpos": z32, "isize": z32, "endpos": z32},
                          np.zeros(0, np.uint64), {"sa_rec": np.zeros(0, np.uint32), "cig_off": np.zeros(1, np.uint32), "cig_ops": np.zeros(0, np.uint32),
                                                   "sa_off": np.zeros(1, np.uint32), "sa_txt": np.zeros(0, np.uint8)}, [1000, 2000], ["chr1", "chr2"])
    c = _ctx_for(empty)
    assert c.scan(100.0) == 0 and c.cluster(100.0, 0) == 0 and c.refine(100.0) == 0 and len(c.fetch_clusters()) == 0
    c.close()
    n = 5000
    rng = np.random.RandomState(0)
    pos = np.sort(rng.randint(0, 900, n)).astype(np.int32)
    z = np.zeros(n, np.int32)
    proper = api.HostBatch({"flag": np.full(n, 99, np.uint16), "mapq": np.full(n, 60, np.uint8), "tid": z, "pos": pos, "mtid": z, "mpos": pos + 200, "isize": np.full(n, 350, np.int32),
                            "endpos": pos + 150}, np.arange(2 * n, dtype=np.uint64), {"sa_rec": np.zeros(0, np.uint32), "cig_off": np.zeros(1, np.uint32), "cig_ops": np.zeros(0, np.uint32),
                                                                                    "sa_off": np.zeros(1, np.uint32), "sa_txt": np.zeros(0, np.uint8)}, [1000, 2000], ["chr1", "chr2"])
    c = _ctx_for(proper)
    mean, sd, dist, ncall = c.run()
    assert (mean, sd) == (350.0, 0.0) and ncall == 0 and len(c.fetch_pairs(0)) == 0
    c.close()


@pytest.mark.parametrize("split_per_sv,scale", [(40, 0.004), (700, 0.004), (4500, 0.002)])
def test_split_read_hotspots_config5(split_per_sv, scale):
    """BASELINE.json configs[4] shape (reduced): breakpoint hotspots with hundreds to thousands of split reads each,
    clip lengths U(20,130), breakpoints jittered +-3 bp.  40 -> per-entry vote, 700 -> shared-memory sort/unique vote,
    4500 (x2 sides > 8192 entries never happens, but > 256 uniques does not either: the global-memory sort is
    forced separately in test_vote_big_many_uniques)."""
    import oracle_py as O
    from breakid_b200 import api, synth
    cfg = synth.config5(scale=scale, split_per_sv=split_per_sv)
    d = synth.generate(cfg)
    hb = api.HostBatch.from_synth(d)
    c = _ctx_for(hb)
    mean, sd, dist, ncall = c.run()
    got = c.fetch_clusters()
    om, osd, od, exp = O.run(hb, None, mode=0)
    assert (mean, sd, dist) == (om, osd, od)
    assert got.tobytes() == exp.tobytes()
    assert len(got) >= 4 and int(got["n_split_read"].max()) > split_per_sv // 2
    c.close()


def test_vote_big_many_uniques():
    """one hotspot whose split reads are spread over +-60 bp: thousands of evidence entries with hundreds of
    distinct (bp1,bp2) keys -> exercises the windowed vote over unique keys and key-string tie breaking."""
    import oracle_py as O
    from breakid_b200 import api, synth
    cfg = synth.SynthConfig(chrom_lens=[400000, 300000], coverage=2.0, n_tra=1, n_inv=1, n_dup=0, n_del=1,
                            split_per_sv=9000, sv_jitter=60, split_k_min=20, split_k_max=131, seed=77)
    d = synth.generate(cfg)
    hb = api.HostBatch.from_synth(d)
    c = _ctx_for(hb)
    mean, sd, dist, ncall = c.run()
    got = c.fetch_clusters()
    om, osd, od, exp = O.run(hb, None, mode=0)
    assert got.tobytes() == exp.tobytes()
    assert len(got) == 3
    c.close()


@pytest.mark.parametrize("flags", [[], ["-q", "35"], ["-fast", "-q", "5"]])
def test_driver_config4_tumour_fusions(tmp_path, flags):
    """BASELINE.json configs[3] shape (reduced): tumour-like 100x BAM, translocations only, dense synthetic refGene so
    that most calls are gene fusions (annotation path: gene, strand, exon numbering columns); non-default -q (the
    reference's -t is declared without an argument, src/BreakID.cc:23, and crashes in atol(NULL): not testable).
    The driver (device decode + GPU path + host annotation) must write the reference binary's files byte for byte."""
    import os
    import subprocess
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio, synth
    ref = O.have_ref()
    cfg = synth.SynthConfig(chrom_lens=[260000, 220000, 180000, 140000], coverage=100.0, n_tra=10, n_inv=0, n_dup=0, n_del=0,
                            span_per_sv=40, split_per_sv=20, seed=44, sv_jitter=1)
    d = synth.generate(cfg)
    paths = bamio.write_dataset(str(tmp_path), d, genes_per_mb=30.0)
    R.index(paths["bam"])
    if ref:
        O.ref_install_refgene(paths["refgene"])
        r = O.ref_run_binary(paths["bam"], str(tmp_path / "ref"), paths["nib"], extra=flags)
        assert r.returncode == 0, r.stderr[-500:]
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    g = subprocess.run([drv, "-i", paths["bam"], "-o", str(tmp_path / "gpu"), "-n", paths["nib"], "-r", paths["refgene"], "-all"] + flags,
                       timeout=600, capture_output=True, text=True)
    assert g.returncode == 0, g.stderr[-500:]
    if ref:
        for suffix in ("_fusion.txt", "_fusion_all.txt"):
            a = open(str(tmp_path / "ref") + suffix).read()
            b = open(str(tmp_path / "gpu") + suffix).read()
            assert a == b, (suffix, flags)
    else:
        R.match_oracle(str(tmp_path / "gpu"), d, mode=int("-fast" in flags), qual=int(flags[flags.index("-q") + 1]) if "-q" in flags else None)
    rows = open(str(tmp_path / "gpu") + "_fusion_all.txt").read().splitlines()[1:]
    assert len(rows) >= 8 and all(x.split("\t")[0] == "Translocation" for x in rows)
    fused = [x for x in open(str(tmp_path / "gpu") + "_fusion.txt").read().splitlines()[1:]]
    assert len(fused) >= 1                      # at least one gene-gene fusion survives the filter
    # host decoder A/B: same files
    g2 = subprocess.run([drv, "-i", paths["bam"], "-o", str(tmp_path / "gpu_host"), "-n", paths["nib"], "-r", paths["refgene"], "-all"] + flags,
                        timeout=600, capture_output=True, text=True, env=dict(os.environ, BKID_HOST_DECODE="1"))
    assert g2.returncode == 0
    assert open(str(tmp_path / "gpu_host") + "_fusion_all.txt").read() == open(str(tmp_path / "gpu") + "_fusion_all.txt").read()


def _prefilter(hb, keep):
    """HostBatch with only the records keep[i] (what a pre-filtered BAM decodes to)"""
    from breakid_b200 import api
    idx = np.nonzero(keep)[0]
    cols = {k: v[idx] for k, v in hb.cols.items()}
    nh = hb.name_hash.reshape(-1, 2)[idx].reshape(-1)
    s = hb.side
    sa_keep = np.nonzero(keep[s["sa_rec"].astype(np.int64)])[0]
    new_index = np.cumsum(keep) - 1
    side = {"sa_rec": new_index[s["sa_rec"].astype(np.int64)[sa_keep]].astype(np.uint32)}
    for off, dat, dt in (("cig_off", "cig_ops", np.uint32), ("sa_off", "sa_txt", np.uint8), ("oc_off", "oc_txt", np.uint8)):
        o = s[off].astype(np.int64)
        parts = [s[dat][o[k]:o[k + 1]] for k in sa_keep]
        side[dat] = np.concatenate(parts).astype(dt) if parts else np.zeros(0, dt)
        side[off] = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.uint32)
    return api.HostBatch(cols, nh, side, hb.target_len, hb.target_names)


def _exclude_intervals(d, rng):
    """intervals that hit planted junctions, noise, chromosome starts/ends; overlapping, touching, empty and duplicate ones"""
    tr = {k: v.numpy() for k, v in d.truth.items()}
    iv = []
    for j in range(0, len(tr["A"]), 3):                       # knock out one side of every third SV
        iv.append((int(tr["A"][j]), int(tr["a"][j]) - 400, int(tr["a"][j]) + 300))
    for j in range(1, len(tr["A"]), 4):                       # and thin the other side of some (removes part of the split reads)
        iv.append((int(tr["B"][j]), int(tr["b"][j]) - 5, int(tr["b"][j]) + 40))
    L = d.cfg.chrom_lens
    for t, l in enumerate(L):
        iv += [(t, 0, 3000), (t, l - 2500, l + 100), (t, l // 2, l // 2 + 5000), (t, l // 2 + 4000, l // 2 + 9000), (t, l // 2 + 9000, l // 2 + 9500)]
        iv += [(t, int(x), int(x) + int(rng.randint(1, 2000))) for x in rng.randint(0, l, 6)]
    iv += [(0, 500, 500), (0, 700, 600), (1, -50, 10), (0, 100000, 100001), (0, 100000, 100001)]
    return np.array(iv, dtype=np.int64)


@pytest.mark.parametrize("mode", [0, 1])
def test_exclude_intervals_equal_prefiltered_input(config1_data, mode):
    """extension (BASELINE.json configs[2]: exclude-BED): device-side exclusion == the oracle on a pre-filtered batch"""
    import oracle_py as O
    d, hb, nibs = config1_data
    iv = _exclude_intervals(d, np.random.RandomState(8))
    tid, pos = hb.cols["tid"].astype(np.int64), hb.cols["pos"].astype(np.int64)
    keep = np.ones(hb.n, bool)
    for t, b, e in iv:
        keep &= ~((tid == t) & (pos >= max(b, 0)) & (pos < e))
    assert 0.02 < 1 - keep.mean() < 0.5
    hbf = _prefilter(hb, keep)
    om, osd, od, exp = O.run(hbf, nibs, mode=mode)
    c = _ctx_for(hb, fast=mode)
    c.set_exclude(iv[:, 0], iv[:, 1], iv[:, 2])
    for t, (p, l) in enumerate(nibs):
        c.set_nib(t, p, l)
    mean, sd, dist, ncall = c.run()
    got = c.fetch_clusters()
    assert (mean, sd, dist) == (om, osd, od)
    assert got.tobytes() == exp.tobytes()
    assert 3 <= len(got) < 10                                  # some planted SVs were knocked out, some survive
    # clearing the filter restores the unfiltered result
    c.set_exclude([], [], [])
    m2, s2, d2, _ = c.run()
    o2 = O.run(hb, nibs, mode=mode)
    assert (m2, s2, d2) == o2[:3] and c.fetch_clusters().tobytes() == o2[3].tobytes()
    c.close()


def test_driver_exclude_bed_matches_reference_on_prefiltered_bam(tmp_path):
    """driver -x regions.bed on the full BAM == the reference binary on a BAM written without the excluded records"""
    import os
    import subprocess
    import torch
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio, synth
    ref = O.have_ref()
    cfg = synth.SynthConfig(chrom_lens=[300000, 200000, 150000], n_tra=3, n_inv=2, n_dup=2, n_del=2, seed=21, sv_jitter=1)
    d = synth.generate(cfg)
    iv = _exclude_intervals(d, np.random.RandomState(4))
    full = bamio.write_dataset(str(tmp_path / "full"), d, genes_per_mb=25.0)
    with open(str(tmp_path / "ex.bed"), "w") as f:
        f.write("# exclude regions\ntrack name=x\n")
        for t, b, e in iv:
            f.write("%s\t%d\t%d\n" % (synth.chrom_name(int(t)), max(int(b), 0), int(e)))
        f.write("chrUn\t5\t10\n")
    tid, pos = d.cols["tid"].numpy().astype(np.int64), d.cols["pos"].numpy().astype(np.int64)
    keep = np.ones(d.n, bool)
    for t, b, e in iv:
        keep &= ~((tid == t) & (pos >= max(b, 0)) & (pos < e))
    kt = torch.from_numpy(keep)
    new_index = torch.cumsum(kt.to(torch.int64), 0) - 1
    sa_keep = kt[d.sa_rec]
    parts = lambda off, dat: torch.cat([dat[int(off[k]):int(off[k + 1])] for k in torch.nonzero(sa_keep).flatten().tolist()] or [dat[:0]])
    lens = lambda off: (off[1:] - off[:-1])[sa_keep]
    mkoff = lambda l: torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(l, 0)])
    d2 = synth.SynthData(cfg=cfg, cols={k: v[kt] for k, v in d.cols.items()}, sa_rec=new_index[d.sa_rec[sa_keep]],
                         cig_off=mkoff(lens(d.cig_off)), cig_ops=parts(d.cig_off, d.cig_ops), sa_off=mkoff(lens(d.sa_off)), sa_txt=parts(d.sa_off, d.sa_txt), truth=d.truth)
    filt = bamio.write_dataset(str(tmp_path / "filt"), d2, genes_per_mb=25.0)
    R.index(filt["bam"]); R.index(full["bam"])
    if ref:
        O.ref_install_refgene(full["refgene"])
        r = O.ref_run_binary(filt["bam"], str(tmp_path / "ref"), filt["nib"])
        assert r.returncode == 0, r.stderr[-500:]
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    g = subprocess.run([drv, "-i", full["bam"], "-o", str(tmp_path / "gpu"), "-n", full["nib"], "-r", full["refgene"], "-all", "-x", str(tmp_path / "ex.bed")],
                       timeout=600, capture_output=True, text=True)
    assert g.returncode == 0, g.stderr[-500:]
    if ref:
        for suffix in ("_fusion.txt", "_fusion_all.txt"):
            assert open(str(tmp_path / "ref") + suffix).read() == open(str(tmp_path / "gpu") + suffix).read(), suffix
    else:
        R.match_oracle(str(tmp_path / "gpu"), d2, check_w=False)
    assert len(open(str(tmp_path / "gpu") + "_fusion_all.txt").read().splitlines()) >= 4


def test_narrow_column_encodings(small_data):
    """isize16 / span16 / tid runs (include/breakid_b200.h) widen on the device to exactly the wide columns; a batch
    that does not fit falls back to the wide column for that field only"""
    from breakid_b200 import api
    d, hb, nibs = small_data
    assert set(hb.narrow()) == {"span16", "isize16", "tid_run_start", "tid_run_tid"}
    cn = _ctx_for(hb)                     # narrow (default)
    cw = api.Context(hb.target_len, hb.target_names, device=0)
    cw.push(hb, narrow=False)
    for k, dt in (("tid", np.int32), ("pos", np.int32), ("isize", np.int32), ("endpos", np.int32), ("flag", np.uint16), ("mapq", np.uint8)):
        a, b = cn.fetch_column(k, dt), cw.fetch_column(k, dt)
        if k == "isize":                  # only the values the path reads have to survive (they all do here)
            assert np.array_equal(a, np.clip(b, -32768, 32767))
        else:
            assert np.array_equal(a, b), k
    assert cn.run()[:3] == cw.run()[:3] and cn.fetch_clusters().tobytes() == cw.fetch_clusters().tobytes()
    cn.close(); cw.close()
    # a long-span record (RNA-style N skip) and a huge proper-pair insert: those two fields go wide, tid stays narrow
    cols = {k: v.copy() for k, v in hb.cols.items()}
    cols["endpos"][7] = cols["pos"][7] + 70000
    proper = np.nonzero((cols["flag"] & 3) == 3)[0]
    cols["isize"][proper[5]] = 40000
    hb2 = api.HostBatch(cols, hb.name_hash, hb.side, hb.target_len, hb.target_names)
    assert set(hb2.narrow()) == {"tid_run_start", "tid_run_tid"}
    c2 = _ctx_for(hb2)
    assert np.array_equal(c2.fetch_column("endpos", np.int32), cols["endpos"]) and np.array_equal(c2.fetch_column("isize", np.int32), cols["isize"])
    assert np.array_equal(c2.fetch_column("tid", np.int32), cols["tid"])
    import oracle_py as O
    om, osd, od, exp = O.run(hb2, None, mode=0)
    assert c2.run()[:3] == (om, osd, od) and c2.fetch_clusters().tobytes() == exp.tobytes()
    c2.close()


def _split_batches(api, hb, cuts):
    parts = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        sa = hb.side["sa_rec"]; lo = np.searchsorted(sa, a); hi = np.searchsorted(sa, b)
        co, so, oo = hb.side["cig_off"], hb.side["sa_off"], hb.side["oc_off"]
        parts.append(api.HostBatch({k: v[a:b] for k, v in hb.cols.items()}, hb.name_hash[2 * a:2 * b],
                                   {"sa_rec": sa[lo:hi] - a, "cig_off": co[lo:hi + 1] - co[lo], "cig_ops": hb.side["cig_ops"][co[lo]:co[hi]],
                                    "sa_off": so[lo:hi + 1] - so[lo], "sa_txt": hb.side["sa_txt"][so[lo]:so[hi]],
                                    "oc_off": oo[lo:hi + 1] - oo[lo], "oc_txt": hb.side["oc_txt"][oo[lo]:oo[hi]]}, hb.target_len, hb.target_names))
    return parts


@pytest.mark.parametrize("order", [(True, False, True), (False, True, True), (True, True, False)])
def test_mixed_narrow_and_wide_batches(small_data, order):
    """the context keeps isize / span narrow in HBM while every batch has them narrow; a wide batch arriving later
    widens what is already held, a narrow batch arriving at a wide context is widened on the way in"""
    from breakid_b200 import api
    d, hb, nibs = small_data
    c1 = _ctx_for(hb)
    r1 = c1.run(); g1 = c1.fetch_clusters()
    c2 = api.Context(hb.target_len, hb.target_names, device=0)
    for part, narrow in zip(_split_batches(api, hb, [0, hb.n // 3, hb.n // 2 + 7, hb.n]), order):
        c2.push(part, narrow=narrow)
    for k, dt in (("isize", np.int32), ("endpos", np.int32), ("tid", np.int32)):
        a, b = c2.fetch_column(k, dt), hb.cols[k]
        assert np.array_equal(np.clip(a, -32768, 32767), np.clip(b, -32768, 32767)) if k == "isize" else np.array_equal(a, b), k
    r2 = c2.run(); g2 = c2.fetch_clusters()
    assert r1 == r2 and g1.tobytes() == g2.tobytes()
    c1.close(); c2.close()


@pytest.mark.parametrize("variant", ["low32_small_groups", "low32_big_groups", "lo64_collisions"])
def test_join_name_hash_collisions(small_data, variant):
    """the join sorts on 32 bits of the 128-bit read-name hash and puts groups that hold several names in order in
    place; bigger mixed groups make it sort the other 32 bits too; names that share all 64 bits of the low word are told
    apart by the high word.  Forced here by degrading the hash: results must not change (the oracle compares 128 bits)."""
    import oracle_py as O
    from breakid_b200 import api
    d, hb, nibs = small_data
    nh = hb.name_hash.reshape(-1, 2).copy()
    lo, hi = nh[:, 0].copy(), nh[:, 1].copy()
    if variant == "low32_small_groups":
        lo = (lo & np.uint64(0xffffffff00000000)) | (lo & np.uint64(0x3ff))          # 1024 values of the sorted bits
    elif variant == "low32_big_groups":
        lo = (lo & np.uint64(0xffffffff00000000)) | (lo & np.uint64(0x3))            # 4 values: groups far beyond the in-place cap
    else:
        hi = hi ^ (lo * np.uint64(0x9E3779B97F4A7C15))                                # keep 128 bits distinct ...
        lo = lo & np.uint64(0x1f)                                                     # ... while only 32 values of name_lo remain
    nh2 = np.stack([lo, hi], 1).reshape(-1)
    # same names <=> same 128-bit value, before and after
    assert len(np.unique(nh.view([("a", "<u8"), ("b", "<u8")]))) == len(np.unique(np.stack([lo, hi], 1).copy().view([("a", "<u8"), ("b", "<u8")])))
    hb2 = api.HostBatch(hb.cols, nh2, hb.side, hb.target_len, hb.target_names)
    c = _ctx_for(hb2)
    m, s = c.insert_stats()
    w = O.dist(m, s)
    n = c.scan(w)
    got = c.fetch_pairs(0)
    exp = O.scan(hb2, 20, w)
    assert n == len(exp) and n > 50
    for k in exp.dtype.names:
        assert np.array_equal(got[k], exp[k]), k
    ref = O.scan(hb, 20, w)
    for k in ("p1_pos", "p2_pos", "p1_chr_pos", "p2_chr_pos", "bucket"):             # and the pairs are those of the undegraded hash
        assert np.array_equal(got[k], ref[k]), k
    c.close()


def test_sparse_table_is_validated(small_data):
    """a candidate missing from the sparse mate/name table, or a table that is not strictly ascending, is an argument
    error -- never a silently different result"""
    import ctypes as C
    from breakid_b200 import api
    d, hb, nibs = small_data
    cand = np.nonzero(((hb.cols["flag"] & 0x703) == 0x1) & (hb.cols["mapq"] >= 20))[0]
    for what in ("missing", "unsorted"):
        c = api.Context(hb.target_len, hb.target_names, device=0)
        b = hb.struct()
        x = {k: v.copy() for k, v in hb.x.items()}
        j = int(np.searchsorted(x["x_rec"], cand[len(cand) // 2]))
        if what == "missing":
            x = {"x_rec": np.delete(x["x_rec"], j), "x_mtid": np.delete(x["x_mtid"], j), "x_mpos": np.delete(x["x_mpos"], j),
                 "x_name_hash": np.delete(x["x_name_hash"].reshape(-1, 2), j, 0).reshape(-1).copy()}
        else:
            x["x_rec"][j], x["x_rec"][j + 1] = x["x_rec"][j + 1], x["x_rec"][j]
        b.n_x = int(x["x_rec"].shape[0])
        for k in x:
            setattr(b, k, x[k].ctypes.data)
        c._chk(c.lib.bkid_push_batch(c.ctx, C.byref(b)))
        with pytest.raises(api.BkidError) as e:
            c.run()
        assert "sparse mate/name table" in str(e.value), (what, str(e.value))
        c.close()


def test_sd_one_pass_form_equals_block_table_form(small_data, monkeypatch):
    """bkid_insert_stats takes the one-pass form (sum floor(a), exact when no record can need a rounding correction below
    the accumulator's final binade) and only otherwise the block tables + resolver: both must give the oracle's sd"""
    import oracle_py as O
    d, hb, nibs = small_data
    exp = O.insert_stats(hb)[:2]
    c = _ctx_for(hb)
    assert c.insert_stats() == exp
    c.close()
    monkeypatch.setenv("BKID_SD_GENERAL", "1")
    c = _ctx_for(hb)
    assert c.insert_stats() == exp
    c.close()


def test_sd_one_pass_form_detects_correctable_records():
    """insert sizes spread over [0, 30000]: the accumulator reaches binade 45, so every record whose squared deviation has a
    fraction >= 1 - 2^-8 may need a rounding correction: the one-pass form must notice them (E > 0, computed here the same
    way on the CPU) and the exact replay must then agree with the oracle's literal loop"""
    import oracle_py as O
    from breakid_b200 import api, dist as D
    rng = np.random.RandomState(8)
    n = 200000
    isz = (rng.randint(0, 30001, n) * rng.choice([-1, 1], n)).astype(np.int32)
    flag = np.full(n, 99, np.uint16)
    z = np.zeros(n, np.int32)
    x = np.abs(isz).astype(np.int64)
    S, N, SQ = int(x.sum()), n, int((x * x).sum())
    kub = D.sd_upper_binade(S, N, SQ, int(x.max()))
    a = (x.astype(np.float64) - float(S) / float(N)) ** 2
    assert 40 <= kub < 51 and int(((a - np.floor(a)) >= 1.0 - 2.0 ** (kub - 53)).sum()) > 100
    hb = api.HostBatch({"flag": flag, "mapq": np.full(n, 60, np.uint8), "tid": z, "pos": np.arange(n, dtype=np.int32), "mtid": z, "mpos": z,
                        "isize": isz, "endpos": np.arange(n, dtype=np.int32) + 100}, np.arange(2 * n, dtype=np.uint64),
                       {"sa_rec": np.zeros(0, np.uint32), "cig_off": np.zeros(1, np.uint32), "cig_ops": np.zeros(0, np.uint32),
                        "sa_off": np.zeros(1, np.uint32), "sa_txt": np.zeros(0, np.uint8)}, [1000000000], ["chr1"])
    assert "isize16" in hb.narrow()
    c = _ctx_for(hb)
    assert c.insert_stats() == O.insert_stats(hb)[:2]
    c.close()


@pytest.mark.parametrize("flags,sd_mult", [(["-s", "15"], 15), (["-q", "20", "-s", "15"], 15), (["-s", "1", "-fast"], 1)])
def test_driver_sd_multiplier_matches_patched_reference(tmp_path, flags, sd_mult):
    """-s (extension: the literal 3 of `times * sqrt(times) * (mean + 3 * sd)`, src/BreakID.cc:103; BASELINE.json configs[2] is quoted
    with `-q 20 -s 15`).  Oracle: the reference binary built with that ONE literal read from the environment (oracle/Makefile
    ref_s) -- the reference itself crashes on an unknown flag."""
    import os
    import subprocess
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio, synth
    ref = O.have_ref() and os.path.exists(O.REF_BIN + "_s")
    cfg = synth.SynthConfig(chrom_lens=[300000, 200000, 150000], n_tra=3, n_inv=2, n_dup=2, n_del=2, seed=29, sv_jitter=1)
    d = synth.generate(cfg)
    paths = bamio.write_dataset(str(tmp_path), d, genes_per_mb=25.0)
    R.index(paths["bam"])
    if ref:
        O.ref_install_refgene(paths["refgene"])
        r = O.ref_run_binary(paths["bam"], str(tmp_path / "ref"), paths["nib"], fast="-fast" in flags, qual=20 if "-q" in flags else None, sd_mult=sd_mult)
        assert r.returncode == 0, r.stderr[-500:]
        r3 = O.ref_run_binary(paths["bam"], str(tmp_path / "ref3"), paths["nib"], fast="-fast" in flags, qual=20 if "-q" in flags else None)
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    g = subprocess.run([drv, "-i", paths["bam"], "-o", str(tmp_path / "gpu"), "-n", paths["nib"], "-r", paths["refgene"], "-all"] + flags, timeout=600, capture_output=True, text=True)
    assert g.returncode == 0, g.stderr[-500:]
    if not ref:
        mean, sd, dist = R.match_oracle(str(tmp_path / "gpu"), d, mode=int("-fast" in flags), qual=20 if "-q" in flags else None, sd_mult=sd_mult)
        assert "%g" % dist != "%g" % O.dist(mean, sd)                  # the flag really changes w
        return
    for suffix in ("_fusion.txt", "_fusion_all.txt"):
        assert open(str(tmp_path / "ref") + suffix).read() == open(str(tmp_path / "gpu") + suffix).read(), suffix
    pa = open(str(tmp_path / "ref") + "_params.txt").read().replace(str(tmp_path / "ref"), "X")
    pb = open(str(tmp_path / "gpu") + "_params.txt").read().replace(str(tmp_path / "gpu"), "X")
    assert pa == pb
    assert pa != open(str(tmp_path / "ref3") + "_params.txt").read().replace(str(tmp_path / "ref3"), "X")     # the flag really changes w


@pytest.mark.parametrize("sd_mult", [15, 1])
def test_params_sd_mult_equals_oracle(small_data, sd_mult):
    """bkid_params.sd_mult through the C ABI against the oracle with the same multiplier"""
    import oracle_py as O
    d, hb, nibs = small_data
    c = _ctx_for(hb, sd_mult=sd_mult)
    mean, sd, dist, ncall = c.run()
    got = c.fetch_clusters()
    om, osd, od, exp = O.run(hb, None, mode=0, sd_mult=sd_mult)
    assert (mean, sd, dist) == (om, osd, od) and dist == O.dist(om, osd, sd_mult=sd_mult)
    assert got.tobytes() == exp.tobytes()
    c.close()


@pytest.mark.parametrize("mode", [0, 1])
def test_stage_by_stage_equals_whole_run(small_data, mode):
    """the reference's main() drives the stages bucket by bucket (src/BreakID.cc:119-167); the same walk through the C ABI --
    bkid_scan, then per bucket bkid_op_remove_isolated -> bkid_op_cluster -> bkid_op_summarize + bkid_refine -- must give
    the calls of bkid_run (and of the oracle), and bkid_set_params must re-classify when qual changes"""
    import oracle_py as O
    from breakid_b200 import api
    d, hb, nibs = small_data
    ctx = api.Context(hb.target_len, hb.target_names, device=0, qual=35)       # wrong threshold first
    ctx.push(hb)
    for t, (p, l) in enumerate(nibs):
        ctx.set_nib(t, p, l)
    mean, sd = ctx.insert_stats()
    ctx.set_params(qual=20, min_reads=2)
    om, osd, od, exp = O.run(hb, nibs, mode=mode)
    assert (mean, sd) == (om, osd)
    ctx.scan(od)
    pairs = ctx.fetch_pairs(0)
    pairs = pairs[np.argsort(pairs["orig"], kind="stable")]
    ranks = np.unique(pairs["bucket"])
    got = []
    for b in ranks:                                                            # dense bucket ids ascend in std::map<string> order
        q = pairs[pairs["bucket"] == b]
        keep = ctx.op_remove_isolated(q["p1_chr_pos"], q["p2_chr_pos"], od)
        q = q[keep]
        if len(q) < 2:
            continue
        idx, cl, roots = ctx.op_cluster(mode, q["p1_chr_pos"], q["p2_chr_pos"], od)
        q = q[idx].copy()
        q["cluster"] = cl
        q = q[np.argsort(q["cluster"], kind="stable")]
        if len(q) == 0:
            continue
        ctx.op_summarize(q, od)
        ctx.refine(od)
        got.append(ctx.fetch_clusters())
    got = np.concatenate(got) if got else np.zeros(0, api.CLUSTER_DTYPE)
    assert len(got) == len(exp) and len(exp) >= 4
    # the whole run numbers buckets densely; here every record carries the bucket of its own pairs: compare everything else
    a = got.copy(); b = exp.copy()
    a["bucket"] = 0; b["bucket"] = 0
    assert a.tobytes() == b.tobytes()
    ctx.close()


@pytest.mark.parametrize("mode", [0, 1])
def test_genome_longer_than_2_32_bases(mode):
    """targets of 2.1 + 2.1 + 0.4 Gb: genome-wide pair coordinates wrap in uint32 like combine_genome_chr_pos
    (src/util_bam.cc:57-68; the oracle's wrap is pinned to the reference in test_scan_wraps_genome_coordinates_like_the_reference);
    scan pairs and the whole path must equal the oracle"""
    import oracle_py as O
    from breakid_b200 import api, synth
    cfg = synth.SynthConfig(chrom_lens=[2_100_000_000, 2_100_000_000, 400_000_000], n_pairs=40000, n_tra=6, n_inv=3, n_dup=3, n_del=3, seed=7, sv_jitter=1)
    d = synth.generate(cfg)
    hb = api.HostBatch.from_synth(d)
    ctx = api.Context(hb.target_len, hb.target_names, device=0, fast=mode)
    ctx.push(hb)
    mean, sd, dist, n = ctx.run()
    om, osd, od, exp = O.run(hb, None, mode=mode)
    assert (mean, sd, dist) == (om, osd, od)
    got_pairs = ctx.fetch_pairs(0)
    ref_pairs = O.scan(hb, 20, od)
    assert np.array_equal(np.sort(got_pairs["p2_chr_pos"]), np.sort(ref_pairs["p2_chr_pos"])) and int((ref_pairs["p2_chr_pos"] < 400_000_000).sum()) >= 3
    assert ctx.fetch_clusters().tobytes() == exp.tobytes() and len(exp) >= 8
    ctx.close()
