"""Multi-GPU parity on real devices: runs tests/dist_check.py under torchrun with every visible GPU (>= 2), NCCL
backend.  Skipped on single-GPU boxes; the host-side logic of the same path is covered on CPU by test_multi_gloo.py."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu


def test_sharded_path_matches_oracle_on_all_gpus():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
                        "--master-port", "29531", os.path.join(here, "dist_check.py")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-2000:])
    assert r.stdout.count("identical to oracle: True") == 3 and r.stdout.count("pre-filtered input: True") == 2, r.stdout[-2000:]
    assert r.stdout.count("identical on every rank: True") == 2, r.stdout[-2000:]
    assert "ranges stitch: True" in r.stdout


@pytest.mark.parametrize("flags", [[], ["-fast"]])
def test_multi_gpu_driver_over_nccl_matches_reference_binary(tmp_path, flags):
    """`BreakID -gpu 0-<n-1>` on distinct devices: one rank per GPU in ONE process, NCCL (ncclCommInitAll) between them;
    the call files must be byte-identical to the reference CPU binary."""
    import torch
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio, synth
    n = min(torch.cuda.device_count(), 8)
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    ref = O.have_ref()
    cfg = synth.SynthConfig(chrom_lens=[300000, 200000, 150000], n_tra=3, n_inv=2, n_dup=2, n_del=2, seed=29, sv_jitter=1)
    d = synth.generate(cfg)
    paths = bamio.write_dataset(str(tmp_path), d, genes_per_mb=25.0)
    R.index(paths["bam"])
    if ref:
        O.ref_install_refgene(paths["refgene"])
        r = O.ref_run_binary(paths["bam"], str(tmp_path / "ref"), paths["nib"], fast="-fast" in flags)
        assert r.returncode == 0, r.stderr[-2000:]
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    g = subprocess.run([drv, "-i", paths["bam"], "-o", str(tmp_path / "gpu"), "-n", paths["nib"], "-r", paths["refgene"], "-all", "-gpu", "0-%d" % (n - 1)] + flags,
                       timeout=600, capture_output=True, text=True)
    assert g.returncode == 0, (g.stdout[-2000:], g.stderr[-2000:])
    assert "communicator\tnccl" in open(str(tmp_path / "gpu") + "_b200_timings.txt").read()
    if not ref:
        R.match_oracle(str(tmp_path / "gpu"), d, mode=int("-fast" in flags))
        assert len(R.fusion_all_rows(str(tmp_path / "gpu"))) >= 5
        return
    for suffix in ("_fusion.txt", "_fusion_all.txt"):
        a = open(str(tmp_path / "ref") + suffix).read()
        assert a == open(str(tmp_path / "gpu") + suffix).read(), suffix
        assert len(a.splitlines()) >= (5 if suffix == "_fusion_all.txt" else 1)
    pa = open(str(tmp_path / "ref") + "_params.txt").read().replace(str(tmp_path / "ref"), "X")
    assert pa == open(str(tmp_path / "gpu") + "_params.txt").read().replace(str(tmp_path / "gpu"), "X")
