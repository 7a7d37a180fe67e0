"""The insert-size mean and sd (src/BreakID.cc:1909-1954) through every entry point that computes them: bkid_insert_stats,
bkid_run, the sharded run with the exchanges inside the library (1, 2 and 3 ranks as threads) and the shard entry points
driven by breakid_b200.dist.run_sharded.  Every one must give the oracle's (mean, sd) bit for bit, with the one-pass form
alone where it is exact and with the exact replay where a record may need a rounding correction (E > 0, or a binade
bound of 51 from an |isize| above 65535).  BKID_SD_GENERAL=1 forces the replay after the one pass."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BATCHES = ["adversarial0", "adversarial1", "adversarial2", "adversarial3", "correctable", "binade51", "small_data"]
PATHS = ["insert_stats", "run", "insert_stats_general", "run_general", "dist1", "dist2", "dist3", "sharded"]


def _isize_batch(isz, flag):
    from breakid_b200 import api
    n = len(isz)
    z = np.zeros(n, np.int32)
    return api.HostBatch({"flag": flag, "mapq": np.full(n, 60, np.uint8), "tid": z, "pos": np.arange(n, dtype=np.int32), "mtid": z, "mpos": z,
                          "isize": isz, "endpos": np.arange(n, dtype=np.int32) + 100}, np.arange(2 * n, dtype=np.uint64),
                         {"sa_rec": np.zeros(0, np.uint32), "cig_off": np.zeros(1, np.uint32), "cig_ops": np.zeros(0, np.uint32),
                          "sa_off": np.zeros(1, np.uint32), "sa_txt": np.zeros(0, np.uint8)}, [1000000000], ["chr1"])


def _batch(name, request):
    if name == "small_data":
        return request.getfixturevalue("small_data")[1]
    if name.startswith("adversarial"):                 # the cases of test_gpu_parity.test_insert_sd_adversarial, same generator
        rng = np.random.RandomState(3)
        for case in range(int(name[-1]) + 1):
            n = [5000, 70000, 300000, 20000][case]
            isz = rng.randint(-2000, 2000, n).astype(np.int32)
            if case == 1: isz = (rng.randint(0, 2, n) * rng.randint(0, 3000000, n)).astype(np.int32)
            if case == 3: isz = rng.randint(-20000000, 20000000, n).astype(np.int32)
            flag = np.where(rng.rand(n) < 0.9, 99, rng.choice([97, 1123, 355, 4], n)).astype(np.uint16)
        return _isize_batch(isz, flag)
    if name == "correctable":                          # the E > 0 batch of test_sd_one_pass_form_detects_correctable_records
        rng = np.random.RandomState(8)
        n = 200000
        isz = (rng.randint(0, 30001, n) * rng.choice([-1, 1], n)).astype(np.int32)
        return _isize_batch(isz, np.full(n, 99, np.uint16))
    rng = np.random.RandomState(21)                    # binade51: narrow insert sizes but one proper pair beyond 65535
    n = 50000
    isz = rng.randint(-600, 600, n).astype(np.int32)
    isz[1234] = -70001
    return _isize_batch(isz, np.full(n, 99, np.uint16))


def _needs_replay(hb):
    """the one-pass form cannot be exact: a binade bound of 51, or a record whose squared deviation has a fraction at least
    1 - 2^(kub-53) (the same test as the kernel's, on the CPU)"""
    from breakid_b200 import dist as D
    f = hb.cols["flag"].astype(np.int64)
    ins = ((f & 1) != 0) & ((f & 2) != 0) & ((f & (0x4 | 0x100 | 0x200 | 0x400)) == 0)
    x = np.abs(hb.cols["isize"][ins].astype(np.int64))
    S, N, SQ = int(x.sum()), len(x), int((x * x).sum())
    kub = D.sd_upper_binade(S, N, SQ, int(x.max()))
    a = (x.astype(np.float64) - float(S) / float(N)) ** 2
    return kub >= 51 or bool(((a - np.floor(a)) >= 1.0 - 2.0 ** (kub - 53)).any())


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("batch", BATCHES)
def test_insert_stats_every_path_equals_oracle(batch, path, request, monkeypatch, capfd):
    import torch
    import oracle_py as O
    from breakid_b200 import api
    from breakid_b200.dist import GpuEngine, run_sharded
    from test_dist_local import _contexts
    hb = _batch(batch, request)
    exp = O.insert_stats(hb)[:2]
    monkeypatch.setenv("BKID_DEBUG_TIMING", "1")
    if path.endswith("_general"):
        monkeypatch.setenv("BKID_SD_GENERAL", "1")
    if path.startswith("dist"):
        ctxs = _contexts(api, hb, int(path[-1]))
        got = [r[:2] for r in api.dist_run_local(ctxs, 0)]
    else:
        ctxs = _contexts(api, hb, 1)
        c = ctxs[0]
        if path.startswith("insert_stats"):
            got = [c.insert_stats()]
        elif path.startswith("run"):
            got = [c.run()[:2]]
        else:
            got = [run_sharded(GpuEngine(c, torch.device("cuda", 0)), hb.n)[:2]]
    for c in ctxs:
        c.close()
    for r, g in enumerate(got):
        assert g == exp, (batch, path, r, g, exp)
    if path.endswith("_general") or _needs_replay(hb):
        assert "sd: resolve" in capfd.readouterr().err, (batch, path, "the exact replay did not run")
