"""The sharded hot path with the exchanges INSIDE the library (bkid_dist_run, breakid_b200/csrc/bkid_dist.cuh), ranks as
host threads of one process on one GPU (bkid_comm_local_create): every rank holds a contiguous slice of one
coordinate-sorted stream; every rank's result must be byte-identical to the CPU oracle on the unsplit input.  The same
pipeline code runs over NCCL on several GPUs (tests/dist_check.py, bench.py --gpus N)."""
import os

import numpy as np
import pytest

from test_multi_gloo import _slice

pytestmark = pytest.mark.gpu


def _contexts(api, hb, world, nibs=None, uneven=True, **kw):
    cuts = [0] + [hb.n * (i + 1) // world + ((13 * (i + 1)) % 29 if uneven and i + 1 < world else 0) for i in range(world)]
    ctxs = []
    for r in range(world):
        c = api.Context(hb.target_len, hb.target_names, device=0, **kw)
        c.push(_slice(hb, cuts[r], cuts[r + 1]))
        if nibs is not None:
            for t, (p, l) in enumerate(nibs):
                c.set_nib(t, p, l)
        ctxs.append(c)
    return ctxs


@pytest.mark.parametrize("world,mode", [(2, 0), (3, 1), (5, 0), (8, 0)])
def test_ranks_as_threads_equal_oracle(small_data, world, mode):
    import oracle_py as O
    from breakid_b200 import api
    d, hb, nibs = small_data
    ctxs = _contexts(api, hb, world, nibs, fast=mode)
    res = api.dist_run_local(ctxs, mode)
    m, s, dd, exp = O.run(hb, nibs, mode=mode)
    assert len(exp) >= 5
    for r, c in enumerate(ctxs):
        assert res[r][:3] == (m, s, dd), r
        assert c.fetch_clusters().tobytes() == exp.tobytes(), r
        c.close()


def test_ranks_as_threads_config2_shape(config1_data):
    """BASELINE.json configs[2]: exclude intervals + -q 20 -s 15, sharded"""
    import oracle_py as O
    from breakid_b200 import api
    from test_gpu_parity import _exclude_intervals, _prefilter
    d, hb, nibs = config1_data
    iv = _exclude_intervals(d, np.random.RandomState(8))
    ctxs = _contexts(api, hb, 4, nibs, qual=20, sd_mult=15)
    for c in ctxs:
        c.set_exclude(iv[:, 0], iv[:, 1], iv[:, 2])
    res = api.dist_run_local(ctxs, 0)
    tid, pos = hb.cols["tid"].astype(np.int64), hb.cols["pos"].astype(np.int64)
    keep = np.ones(hb.n, bool)
    for t, b, e in iv:
        keep &= ~((tid == t) & (pos >= max(b, 0)) & (pos < e))
    m, s, dd, exp = O.run(_prefilter(hb, keep), nibs, qual=20, mode=0, sd_mult=15)
    assert len(exp) >= 3
    for r, c in enumerate(ctxs):
        assert res[r][:3] == (m, s, dd), r
        assert c.fetch_clusters().tobytes() == exp.tobytes(), r
        c.close()


def test_ranks_as_threads_sd_replay_chain():
    """insert sizes spread so wide that records can need rounding corrections: the one-pass sd form reports E > 0 and the
    exact order-dependent replay is chained rank to rank"""
    import oracle_py as O
    from breakid_b200 import api
    rng = np.random.RandomState(8)
    n = 120000
    isz = (rng.randint(0, 30001, n) * rng.choice([-1, 1], n)).astype(np.int32)
    z = np.zeros(n, np.int32)
    hb = api.HostBatch({"flag": np.full(n, 99, np.uint16), "mapq": np.full(n, 60, np.uint8), "tid": z, "pos": np.arange(n, dtype=np.int32), "mtid": z, "mpos": z,
                        "isize": isz, "endpos": np.arange(n, dtype=np.int32) + 100}, np.arange(2 * n, dtype=np.uint64),
                       {"sa_rec": np.zeros(0, np.uint32), "cig_off": np.zeros(1, np.uint32), "cig_ops": np.zeros(0, np.uint32),
                        "sa_off": np.zeros(1, np.uint32), "sa_txt": np.zeros(0, np.uint8)}, [1000000000], ["chr1"])
    ctxs = _contexts(api, hb, 3)
    res = api.dist_run_local(ctxs, 0)
    exp = O.insert_stats(hb)[:2]
    for r, c in enumerate(ctxs):
        assert res[r][:2] == exp, (r, res[r], exp)
        c.close()


def test_ranks_as_threads_sharded_decode(tmp_path, small_data):
    """ingest sharded too: every rank inflates and decodes its own BGZF block range of one BAM file"""
    import oracle_py as O
    from breakid_b200 import api, bamio
    d, hb, nibs = small_data
    bam = str(tmp_path / "reads.bam")
    bamio.write_bam(bam, d)
    f = api.BgzfFile(bam)
    world = 4
    cuts = [f.n_blocks * i // world for i in range(world + 1)]
    ctxs, marks = [], []
    for r in range(world):
        c = api.Context(f.target_len, f.target_names, device=0)
        n, a, b = c.push_bgzf_range(f, cuts[r], cuts[r + 1])
        marks.append((a, b, n))
        for t, (p, l) in enumerate(nibs):
            c.set_nib(t, p, l)
        ctxs.append(c)
    assert all(marks[i][1] == marks[i + 1][0] for i in range(world - 1)) and sum(m[2] for m in marks) == hb.n
    res = api.dist_run_local(ctxs, 0)
    m, s, dd, exp = O.run(hb, nibs, mode=0)
    for r, c in enumerate(ctxs):
        assert res[r][:3] == (m, s, dd), r
        assert c.fetch_clusters().tobytes() == exp.tobytes(), r
        c.close()
    f.close()


@pytest.mark.parametrize("gpus,flags", [("0,0,0", []), ("0,0", ["-fast"]), ("0,0,0,0", ["-q", "20", "-s", "15"])])
def test_multi_gpu_driver_matches_reference_binary(tmp_path, gpus, flags):
    """`BreakID -gpu a,b,...`: one rank (host thread + context) per entry, sharded BGZF ingest, exchanges inside the library.
    Naming one device several times makes the ranks share it (device-copy communicator) -- the same driver code that runs
    over NCCL on distinct devices.  Call files must be byte-identical to the reference CPU binary (for -s: the reference
    built with the literal 3 of src/BreakID.cc:103 read from the environment, oracle/Makefile ref_s)."""
    import subprocess
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio, synth
    sd_mult = 15 if "-s" in flags else None
    ref = O.have_ref() and (sd_mult is None or os.path.exists(O.REF_BIN + "_s"))
    cfg = synth.SynthConfig(chrom_lens=[300000, 200000, 150000], n_tra=3, n_inv=2, n_dup=2, n_del=2, seed=23, sv_jitter=1)
    d = synth.generate(cfg)
    paths = bamio.write_dataset(str(tmp_path), d, genes_per_mb=25.0)
    R.index(paths["bam"])
    if ref:
        O.ref_install_refgene(paths["refgene"])
        r = O.ref_run_binary(paths["bam"], str(tmp_path / "ref"), paths["nib"], fast="-fast" in flags, qual=20 if "-q" in flags else None, sd_mult=sd_mult)
        assert r.returncode == 0, r.stderr[-500:]
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    g = subprocess.run([drv, "-i", paths["bam"], "-o", str(tmp_path / "gpu"), "-n", paths["nib"], "-r", paths["refgene"], "-all", "-gpu", gpus] + flags,
                       timeout=600, capture_output=True, text=True)
    assert g.returncode == 0, (g.stdout[-300:], g.stderr[-500:])
    if not ref:
        R.match_oracle(str(tmp_path / "gpu"), d, mode=int("-fast" in flags), qual=20 if "-q" in flags else None, sd_mult=sd_mult or 3)
        assert len(R.fusion_all_rows(str(tmp_path / "gpu"))) >= 5
        assert "communicator\tlocal" in open(str(tmp_path / "gpu") + "_b200_timings.txt").read()
        return
    for suffix in ("_fusion.txt", "_fusion_all.txt"):
        a = open(str(tmp_path / "ref") + suffix).read()
        b = open(str(tmp_path / "gpu") + suffix).read()
        assert a == b, suffix
        assert len(a.splitlines()) >= (5 if suffix == "_fusion_all.txt" else 1)
    pa = open(str(tmp_path / "ref") + "_params.txt").read().replace(str(tmp_path / "ref"), "X")
    pb = open(str(tmp_path / "gpu") + "_params.txt").read().replace(str(tmp_path / "gpu"), "X")
    assert pa == pb
    assert "communicator\tlocal" in open(str(tmp_path / "gpu") + "_b200_timings.txt").read()
