"""What the driver-vs-reference tests check where the reference binary is not built (oracle/_ref needs the reference
sources, which are not part of this repository).

There, the driver's _fusion_all.txt rows (type, breakpoints, N_DRP, N_SR, depths, AFs, 41-mers) and the w line of its
_params.txt are compared with the CPU oracle on the same records.  The oracle is pinned to the reference by
tests/test_golden.py (stored output of the reference binary and functions) and, where the reference is built, by
tests/test_oracle_vs_ref.py.  The gene annotation columns and the filtered _fusion.txt are compared with the reference
only where it is built, and on the mini dataset of tests/golden (test_driver_matches_stored_reference_call_files).
"""
import oracle_py as O


def index(bam):
    """the .bai next to a BAM: built by the reference's htslib where it is built; elsewhere an empty file, since the
    driver only checks that an index exists"""
    if O.have_ref():
        O.ref_index(bam)
    else:
        open(bam + ".bai", "wb").close()


def fusion_all_rows(prefix):
    """the compared columns of every row of <prefix>_fusion_all.txt"""
    rows = set()
    for ln in open(prefix + "_fusion_all.txt").read().splitlines()[1:]:
        f = ln.split("\t")
        rows.add((f[0], f[1], f[2], f[7], f[8], f[9], f[10], f[11], f[12], f[13], f[14]))
    return rows


def match_oracle(prefix, d, mode=0, qual=None, sd_mult=3, check_w=True, target_names=None):
    """assert the driver's files under `prefix` hold the oracle's calls on SynthData `d` (and its w); returns the oracle's
    (mean, sd, dist).  target_names: the header names the files were written with (default synth.chrom_name)"""
    from breakid_b200 import api, synth
    from test_golden import _format_calls
    hb = api.HostBatch.from_synth(d, target_names)
    nibs = [(synth.random_nib_bytes(l, d.cfg.seed * 1000 + t).numpy(), l) for t, l in enumerate(d.cfg.chrom_lens)]
    mean, sd, dist, cl = O.run(hb, nibs, mode=mode, sd_mult=sd_mult, **({"qual": qual} if qual is not None else {}))
    assert fusion_all_rows(prefix) == _format_calls(cl, hb.target_names)
    if check_w:
        w_line = [ln for ln in open(prefix + "_params.txt").read().splitlines() if ln.startswith("w\t")][0]
        assert w_line == "w\t%g" % dist
    return mean, sd, dist
