"""Headers outside the chr1..chrY convention through every name-dependent stage, against the CPU oracle.

The reference names a chromosome three ways, and they need not agree (SURVEY.md:350-357): the own side of a split read by
chromID2ChrName(tid) ("chr1".."chr22", "chrX", "chrY", "" from tid 24 on), the SA side by the SA tag's text, and a
cluster's p1 side by the header name (src/BreakID.cc:618-619,647).  Buckets are keys "<p1 name>_<p2 name>" of a
std::map<string> (src/BreakID.cc:1500-1512).  The device replaces these strings with codes (chr_code, canon[], the
host-built bucket rank table), so it must be run on headers where the three differ.  Every other suite names target t
chromID2ChrName(t), where they cannot differ.

`build_names_batch` plants the same junctions and split reads under every header profile; only the @SQ names and the
names inside the SA texts change.  Each junction's SA texts follow one convention: the header names (what an aligner
writes), chromID2ChrName names, one of each on the two records, or zero-padded names ("chr01").  The profiles are:

  * canonical: chromID2ChrName names (the control);
  * ucsc_hg19: chrM at tid 0, so every chrN sits one tid later, then _random, _hap and chrUn_ contigs;
  * b37: 1..22, X, Y, MT, GL000192.1, NC_007605, hs37d5, ...;
  * hg38_like: chr1..chrY, then chr1_KI270706v1_random, HLA-A*01:01:01:01, chrUn_GL000220v1, chrEBV, ...: junctions
    on tids 24 and 25, whose own name is "";
  * permuted: the chrN names in a scrambled order (chr2 at tid 0, chr1 at tid 1), so chromID2ChrName(t) is the header
    name of another tid;
  * punct: names starting with ! # $ % & (they sort before "*"), names with . - : = | ~ (around "_"), and names that
    are prefixes of others (chr1_, chr1, chr10);
  * collide: scaf, scaf_1, 1_2 and 2 at tids 4..7: the target pairs (scaf, 1_2) and (scaf_1, 2) both give the
    bucket string "scaf_1_2", one bucket of the reference's map.

The CPU tests prove with the oracle alone that each rung is reached; the GPU tests require the device to equal the
oracle byte for byte through the library, the sharded path, the decoders and the BreakID driver."""
import os
import subprocess
import time

import numpy as np
import pytest
import torch

L = 150
NT = 30
JT = (0, 1, 2, 3, 4, 5, 6, 7, 24, 25)                      # the tids that hold records
LENS = [200000 if t in JT else 30000 + 1000 * t for t in range(NT)]
SEED = 53

PAIRED, PROPER, UNMAP, MUNMAP, REVERSE, MREVERSE, READ1, READ2, SECONDARY, DUP = (
    0x1, 0x2, 0x4, 0x8, 0x10, 0x20, 0x40, 0x80, 0x100, 0x400)
CONVS = ("header", "chrom", "mixed", "padded")
N_SPLIT = 4


def cid_name(t):
    """chromID2ChrName (src/util_bam.cc:128-142)"""
    if t == 23:
        return "chrY"
    if t == 22:
        return "chrX"
    return "chr%d" % (t + 1) if 0 <= t < 22 else ""


def _canonical():
    from breakid_b200 import synth
    return [synth.chrom_name(t) for t in range(NT)]


HG38_EXTRA = ["chr1_KI270706v1_random", "HLA-A*01:01:01:01", "chrUn_GL000220v1", "chrEBV", "chrM", "chr22_KI270731v1_random"]


def _permuted():
    rng = np.random.RandomState(7)
    while True:
        p = rng.permutation(np.arange(2, 24))
        if np.all(p != np.arange(2, 24)):
            break
    return ["chr2", "chr1"] + [cid_name(int(t)) for t in p] + HG38_EXTRA


PROFILES = {
    "canonical": _canonical(),
    "ucsc_hg19": ["chrM"] + [cid_name(t) for t in range(24)] + ["chr1_gl000191_random", "chr4_ctg9_hap1", "chr17_gl000205_random",
                                                                 "chrUn_gl000211", "chrUn_gl000249"],
    "b37": [str(i) for i in range(1, 23)] + ["X", "Y", "MT", "GL000192.1", "NC_007605", "hs37d5", "GL000207.1", "GL000226.1"],
    "hg38_like": [cid_name(t) for t in range(24)] + HG38_EXTRA,
    "permuted": _permuted(),
    "punct": ["chr1_", "chr1", "chr10", "!chr", "#1", "$scaf", "%2", "&x", "chr1.1", "chr1-1", "chr1:1", "chr1|1", "chr1~1",
              "chr1_a", "chr2", "chr3", "chr4", "chr5", "chr6", "chr7", "chr8", "chr9", "chrX", "chrY", "chr1=1", "a=b",
              "z|z", "~end", "chr1.", "chr1-"],
    "collide": _canonical()[:4] + ["scaf", "scaf_1", "1_2", "2"] + _canonical()[8:],
}
NO_COLLIDE = PROFILES["collide"][:6] + ["1_3"] + PROFILES["collide"][7:]


def hg38_names(n=3366):
    """a header of hg38 analysis-set size: chr1..chrY, chrM, chrEBV, then _random, chrUn_ and _alt contigs and HLA alleles"""
    out = [cid_name(t) for t in range(24)] + ["chrM", "chrEBV"]
    k = 0
    while len(out) < n:
        kind = k % 4
        if kind == 0:
            out.append("chr%d_KI27%04dv1_random" % (k % 22 + 1, k))
        elif kind == 1:
            out.append("chrUn_GL00%04dv1" % k)
        elif kind == 2:
            out.append("chr%d_KI27%04dv1_alt" % (k % 22 + 1, k))
        else:
            out.append("HLA-%s*%02d:%02d:%02d" % ("ABC"[k % 3], k % 97, k % 89, k % 83))
        k += 1
    return out


# ------------------------------------------------------------------------------------------------------------ batch
def _sa(name, pos1, cig):
    return ("%s,%d,+,%s,60,0;" % (name, pos1, cig)).encode()


def _sa_name(names, t, conv, on_a):
    """the name the SA text of the record on side A (on_a) or B gives to target t"""
    if conv == "header" or (conv == "mixed" and on_a):
        return names[t]
    if conv == "padded" and t < 9:
        return "chr0%d" % (t + 1)
    return cid_name(t) if t < 24 else names[t]


def junctions():
    """(name, A, B, SA convention, flip): flip puts the primary record on B and the 0x100 record on A (side 1)"""
    out = []
    for conv in CONVS:
        for flip in (False, True):
            out.append(("ab_%s_%s" % (conv, "flip" if flip else "plain"), 0, 1, conv, flip))
    for conv in ("header", "chrom", "mixed"):
        out.append(("same_%s" % conv, 2, 2, conv, False))
        out.append(("a24_%s" % conv, 3, 24, conv, False))
        out.append(("hi_%s" % conv, 24, 25, conv, False))
    out.append(("col_a", 4, 6, "chrom", False))
    out.append(("col_b", 5, 7, "chrom", False))
    out.append(("col_c", 4, 6, "header", True))
    return out


def build_names_batch(names, seed=SEED):
    """the batch as synth.SynthData and the junction table.  The records are the same for every list of names: the
    SA texts alone name targets"""
    from breakid_b200 import synth
    from test_chrom_edges import _cigar_ops
    rng = np.random.RandomState(seed)
    recs, meta = [], {}
    nid = [0]

    def name():
        nid[0] += 1
        return nid[0] - 1

    def add(flag, mapq, tid, pos, mtid, mpos, isize, endpos, n, sa=None):
        recs.append((flag, mapq, tid, pos, mtid, mpos, isize, endpos, n, sa))

    for t in (0, 1, 2, 3):                                   # proper pairs: the insert-size statistics
        npairs = LENS[t] * 3 // (2 * L)
        starts = rng.randint(0, LENS[t] - 1000, npairs)
        ins = np.clip(np.round(rng.randn(npairs) * 30 + 350), L + 1, 800).astype(np.int64)
        for p1, i in zip(starts.tolist(), ins.tolist()):
            p2 = p1 + i - L
            n = name()
            add(PAIRED | PROPER | MREVERSE | READ1, 60, t, p1, t, p2, i, p1 + L, n)
            add(PAIRED | PROPER | REVERSE | READ2, 60, t, p2, t, p1, -i, p2 + L, n)
    nxt = {t: 20000 for t in JT}
    for jn, A, B, conv, flip in junctions():
        a = nxt[A]; nxt[A] += 15000
        if A == B:
            b = a + 6000; nxt[A] += 15000
        else:
            b = nxt[B]; nxt[B] += 15000
        assert a < LENS[A] - 20000 and b < LENS[B] - 20000
        p1s, p2s = [], []
        for _ in range(12):                                  # spanning pairs: the A reads end before a, the B reads start after b
            r1 = a - L - 1 - int(rng.randint(0, 250))
            r2 = b - 1 + int(rng.randint(0, 250)) + (200 if A == B else 0)
            k = name()
            add(PAIRED | MREVERSE | READ1, 60, A, r1, B, r2, 0, r1 + L, k)
            add(PAIRED | REVERSE | READ2, 60, B, r2, A, r1, 0, r2 + L, k)
            p1s.append(r1 + 1); p2s.append(r2 + 1)
        for _ in range(N_SPLIT):                             # split reads: left part ends at A:a on +, right part starts at B:b
            k = int(rng.randint(L // 2 + 1, L - 20))
            n = name()
            left, right = "%dM%dS" % (k, L - k), "%dS%dM" % (k, L - k)
            fa = PAIRED | PROPER | MREVERSE | READ1 | (SECONDARY if flip else 0)
            fb = PAIRED | PROPER | MREVERSE | READ1 | (0 if flip else SECONDARY)
            add(fa, 60, A, a - k, A, a - k + 200, 0 if flip else 200 + L, a, n, (left, _sa(_sa_name(names, B, conv, True), b, right)))
            add(fb, 60, B, b - 1, A, a - k + 200, 200 + L if flip else 0, b - 1 + L - k, n,
                (right, _sa(_sa_name(names, A, conv, False), a - k + 1, left)))
        meta[jn] = dict(A=A, a=a, B=B, b=b, conv=conv, flip=flip, p1_mean=int(sum(p1s) / len(p1s)), p2_mean=int(sum(p2s) / len(p2s)))
    tid = np.array([r[2] for r in recs], np.int64)
    pos = np.array([r[3] for r in recs], np.int64)
    order = np.lexsort((pos, tid.astype(np.uint32)))
    recs = [recs[i] for i in order]
    cols = {}
    for c, (k, dt) in enumerate((("flag", torch.int16), ("mapq", torch.uint8), ("tid", torch.int32), ("pos", torch.int32),
                                 ("mtid", torch.int32), ("mpos", torch.int32), ("isize", torch.int32), ("endpos", torch.int32),
                                 ("name_id", torch.int64))):
        v = np.array([r[c] for r in recs], np.int64)
        cols[k] = torch.from_numpy(v.astype(np.uint16).view(np.int16) if k == "flag" else v).to(dt)
    sa_rec = [i for i, r in enumerate(recs) if r[9] is not None]
    cig, cig_off, txt, sa_off = [], [0], b"", [0]
    for i in sa_rec:
        cig += _cigar_ops(recs[i][9][0]); cig_off.append(len(cig))
        txt += recs[i][9][1]; sa_off.append(len(txt))
    cfg = synth.SynthConfig(chrom_lens=list(LENS), read_len=L, n_tra=0, n_inv=0, n_dup=0, n_del=0, seed=seed)
    i64 = lambda x: torch.tensor(x, dtype=torch.int64)
    d = synth.SynthData(cfg=cfg, cols=cols, sa_rec=i64(sa_rec), cig_off=i64(cig_off), cig_ops=i64(cig), sa_off=i64(sa_off),
                        sa_txt=torch.tensor(list(txt), dtype=torch.uint8), truth={})
    return d, meta


def nibs_for(d):
    from breakid_b200 import synth
    return [(synth.random_nib_bytes(l, d.cfg.seed * 1000 + t).numpy(), l) for t, l in enumerate(d.cfg.chrom_lens)]


_CACHE = {}


def profile_data(profile, names=None):
    """(SynthData, HostBatch, nibs, junction table, oracle run per mode) of a profile, built once per session"""
    import oracle_py as O
    from breakid_b200 import api
    key = profile if names is None else (profile, tuple(names))
    if key not in _CACHE:
        names = PROFILES[profile] if names is None else names
        d, meta = build_names_batch(names)
        hb = api.HostBatch.from_synth(d, names)
        nibs = nibs_for(d)
        runs = {mode: O.run(hb, nibs, mode=mode) for mode in (0, 1)}
        _CACHE[key] = (d, hb, nibs, meta, runs)
    return _CACHE[key]


def _find(cl, j):
    """the call of junction j: its chromosomes, and its breakpoints within 40 bp of (a, b) or of (b, a)"""
    hit = [c for c in cl if (int(c["p1_tid"]), int(c["p2_tid"])) == (j["A"], j["B"]) and
           ((abs(int(c["p1_exact_pos"]) - j["a"]) <= 40 and abs(int(c["p2_exact_pos"]) - j["b"]) <= 40) or
            (abs(int(c["p1_exact_pos"]) - j["b"]) <= 40 and abs(int(c["p2_exact_pos"]) - j["a"]) <= 40))]
    assert len(hit) <= 1
    return hit[0] if hit else None


def _side1_rows(hb, j, w):
    import oracle_py as O
    from test_chrom_edges import _region
    return O.find_sa_reads(hb, j["A"], *_region(j["p1_mean"], w))


# ------------------------------------------------------------------------------------------------ CPU: rungs are reached
def test_profiles_shape():
    for p, names in PROFILES.items():
        assert len(names) == NT and len(set(names)) == NT, p
        assert all(n and not set(n) & set(",; \t\n") for n in names), p
    assert [cid_name(t) for t in range(NT)][:24] == PROFILES["canonical"][:24] and cid_name(24) == ""
    assert sum(PROFILES["ucsc_hg19"][t] == cid_name(t - 1) for t in range(1, 25)) == 24
    assert not any(PROFILES["b37"][t] == cid_name(t) for t in range(NT))
    perm = PROFILES["permuted"]
    assert all(perm[t] != cid_name(t) and cid_name(t) in perm for t in range(24))
    pu = PROFILES["punct"]
    assert sum(n.encode() < b"*" for n in pu) == 5 and sum(n.startswith("chr1") and n[4:5] in ".-:=|~" for n in pu) >= 6
    assert {"chr1", "chr1_", "chr10"} <= set(pu)
    col = PROFILES["collide"]
    assert col[4] + "_" + col[6] == col[5] + "_" + col[7] == "scaf_1_2"
    assert len({a + "_" + b for a in NO_COLLIDE for b in NO_COLLIDE}) == NT * NT
    h = hg38_names()
    assert len(h) == len(set(h)) == 3366 and any("*" in n and ":" in n for n in h)


def test_writers_name_every_target(tmp_path):
    """write_dataset names the @SQ lines of the BAM and the SAM, RNAME / RNEXT, ref_names.txt, the nib files and the
    refGene rows by the profile; the host decoders read the names back"""
    from breakid_b200 import api, bamio
    names = PROFILES["hg38_like"]
    d, hb, nibs, meta, runs = profile_data("hg38_like")
    paths = bamio.write_dataset(str(tmp_path), d, sam=True, target_names=names)
    got = api.HostBatch.from_bam(paths["bam"])
    assert got.target_names == names and list(got.target_len) == LENS
    for k in ("flag", "tid", "pos", "mtid", "mpos", "isize", "endpos"):
        assert np.array_equal(got.cols[k], hb.cols[k]), k
    assert bytes(got.side["sa_txt"]) == bytes(hb.side["sa_txt"])
    assert open(os.path.join(paths["nib"], "ref_names.txt")).read().split("\n")[:-1] == names
    assert all(os.path.exists(os.path.join(paths["nib"], "hg19_%s.nib" % n)) for n in names)
    assert {ln.split("\t")[2] for ln in open(paths["refgene"]).read().splitlines()} == set(names)
    sf = api.SamFile(paths["sam"])
    assert sf.target_names == names and sf.target_len == LENS
    sf.close()
    sam = open(paths["sam"]).read().splitlines()
    assert [ln.split("\t")[1][3:] for ln in sam if ln.startswith("@SQ")] == names
    body = [ln.split("\t") for ln in sam if not ln.startswith("@")]
    assert {f[2] for f in body} == {names[t] for t in JT} and "HLA-A*01:01:01:01" in {f[6] for f in body}
    assert {f[6] for f in body} - {"="} <= set(names)


def test_sa_conventions_reach_every_rung():
    """which SA naming yields split-read evidence depends on the header: the oracle's calls per profile"""
    for p in PROFILES:
        d, hb, nibs, meta, runs = profile_data(p)
        names = PROFILES[p]
        for mode in (0, 1):
            m, s, dist, cl = runs[mode]
            called = {jn for jn, j in meta.items() if _find(cl, j) is not None}
            for jn in called:
                assert int(_find(cl, meta[jn])["n_split_read"]) == N_SPLIT, (p, jn)
            # tid 24 and up: the own name is "", no SA text can match it
            assert not any(jn.startswith(("a24_", "hi_")) for jn in called), (p, called)
            if p == "canonical":
                assert {"ab_header_plain", "ab_chrom_flip", "same_header", "col_a", "col_b"} <= called
                assert not {"ab_padded_plain", "ab_padded_flip"} & called        # "chr01" is not chromID2ChrName(0)
            if p == "b37":                                    # header-named SA texts: no evidence at all
                assert not any(meta[jn]["conv"] in ("header", "mixed") for jn in called) and "ab_chrom_plain" in called
            if p == "ucsc_hg19":                              # the own name is the next tid's header name
                assert "ab_header_plain" not in called and "ab_chrom_plain" in called
            if p == "hg38_like":
                assert "ab_header_plain" in called
        assert all(names[t] == cid_name(t) for t in (0, 1)) == (p in ("canonical", "hg38_like", "collide"))


def test_primary_rows_oriented_from_p2():
    """b37 header, chromID2ChrName SA texts: the side-1 rows are primaries whose primary chromosome (chromID2ChrName(0))
    is not p1's header name "1", so the reference takes x from the p2 side: the call is (b, a)"""
    d, hb, nibs, meta, runs = profile_data("b37")
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        j = meta["ab_chrom_plain"]
        rows = _side1_rows(hb, j, int(dist))
        assert len(rows) == N_SPLIT and np.all(rows["secondary"] == 0) and np.all(rows["primary_chr"] == 0)
        c = _find(cl, j)
        assert (int(c["p1_tid"]), int(c["p1_exact_pos"]), int(c["p2_exact_pos"])) == (0, j["b"], j["a"])
    c = _find(profile_data("canonical")[4][0][3], profile_data("canonical")[3]["ab_chrom_plain"])
    assert (int(c["p1_exact_pos"]), int(c["p2_exact_pos"])) == (meta["ab_chrom_plain"]["a"], meta["ab_chrom_plain"]["b"])


def test_secondary_row_oriented_from_p1():
    """permuted header (chr2 at tid 0), chromID2ChrName SA texts, primary on B: the side-1 rows are 0x100 records whose
    primary chromosome (the SA's "chr2") is p1's header name, so x is their primary breakpoint, which lies on B: the
    call is (b, a).  Under the canonical header the same records give (a, b)"""
    d, hb, nibs, meta, runs = profile_data("permuted")
    j = meta["ab_chrom_flip"]
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        rows = _side1_rows(hb, j, int(dist))
        assert len(rows) == N_SPLIT and np.all(rows["secondary"] == 1) and np.all(rows["primary_chr"] == 1)
        c = _find(cl, j)
        assert (int(c["p1_exact_pos"]), int(c["p2_exact_pos"])) == (j["b"], j["a"])
        cc = _find(profile_data("canonical")[4][mode][3], j)
        assert (int(cc["p1_exact_pos"]), int(cc["p2_exact_pos"])) == (j["a"], j["b"])


def _rank_model(names):
    """dense rank of every "A_B" string (index 0 = "*") in byte order, the std::map<string> order"""
    m = len(names) + 1
    nm = [b"*"] + [n.encode() for n in names]
    keys = np.array([a + b"_" + b for a in nm for b in nm], dtype=object)
    uniq = sorted(set(keys.tolist()))
    pos = {k: i for i, k in enumerate(uniq)}
    return np.array([pos[k] for k in keys.tolist()], np.int32).reshape(m, m)


def _rank_table(names):
    import oracle_py as O
    import types
    rank = np.zeros((len(names) + 1) ** 2, np.int32)
    O.olib().orc_bucket_rank_table(len(names), O._names(types.SimpleNamespace(target_names=names)), rank)
    return rank.reshape(len(names) + 1, len(names) + 1)


@pytest.mark.parametrize("profile", sorted(PROFILES) + ["no_collide"])
def test_bucket_rank_table_is_dense_byte_order(profile):
    names = NO_COLLIDE if profile == "no_collide" else PROFILES[profile]
    got = _rank_table(names)
    assert np.array_equal(got, _rank_model(names))
    ties = (NT + 1) ** 2 - len(np.unique(got))
    assert ties == (1 if profile == "collide" else 0)         # "scaf" + "_" + "1_2" == "scaf_1" + "_" + "2"
    if profile == "collide":
        assert got[5, 7] == got[6, 8]


def test_bucket_rank_table_hg38_size():
    names = hg38_names()
    got = _rank_table(names)
    m = len(names) + 1
    nm = np.array([b"*"] + [n.encode() for n in names], dtype=object)
    keys = (nm[:, None] + b"_" + nm[None, :]).reshape(-1)
    order = np.argsort(keys, kind="stable")
    sk = keys[order]
    dense = np.concatenate([[0], np.cumsum(sk[1:] != sk[:-1])]).astype(np.int32)
    exp = np.empty(m * m, np.int32)
    exp[order] = dense
    assert np.array_equal(got.reshape(-1), exp)


def test_colliding_names_merge_buckets():
    """orc_scan on collide: the pairs of (scaf, 1_2) and (scaf_1, 2) are one bucket, so the calls differ from the same
    records under names that do not collide"""
    import oracle_py as O
    d, hb, nibs, meta, runs = profile_data("collide")
    m, s, dist, cl = runs[0]
    pairs = O.scan(hb, 20, dist)
    tp = {(int(a), int(b)) for a, b in zip(pairs["p1_tid"], pairs["p2_tid"])}
    assert len(np.unique(pairs["bucket"])) < len(tp)
    b46 = set(pairs["bucket"][(pairs["p1_tid"] == 4) & (pairs["p2_tid"] == 6)].tolist())
    b57 = set(pairs["bucket"][(pairs["p1_tid"] == 5) & (pairs["p2_tid"] == 7)].tolist())
    assert len(b46) == 1 and b46 == b57
    merged = pairs[pairs["bucket"] == b46.pop()]
    assert np.all(np.diff(merged["orig"].astype(np.int64)) > 0)                      # emission order inside the bucket
    for mode in (0, 1):
        other = profile_data("no_collide", NO_COLLIDE)[4][mode][3]
        assert runs[mode][3].tobytes() != other.tobytes()
        assert _find(runs[mode][3], meta["col_a"]) is not None and _find(runs[mode][3], meta["col_b"]) is not None


def test_create_refuses_headers_above_the_limit():
    """50 000 targets: bkid_create returns NULL with the reason at once, before it looks for a device"""
    from breakid_b200 import api
    n = 50000
    t0 = time.time()
    with pytest.raises(api.BkidError, match="header has 50000 targets; at most 46339"):
        api.Context([1000] * n, ["c%d" % i for i in range(n)])
    assert time.time() - t0 < 5
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "breakid_b200.h")).read()
    assert "#define BKID_MAX_TARGETS 46339" in hdr and (46339 + 1) ** 2 < 2 ** 31 <= (46340 + 1) ** 2


# ------------------------------------------------------------------------------------------------ GPU: device == oracle
def _device_run(hb, nibs, mode, narrow=True):
    from breakid_b200 import api
    c = api.Context(hb.target_len, hb.target_names, device=0, fast=mode)
    c.push(hb, narrow=narrow)
    for t, (p, l) in enumerate(nibs):
        c.set_nib(t, p, l)
    res = c.run()
    got = c.fetch_clusters()
    c.close()
    return res, got


def _assert_equal(res, got, exp_run):
    m, s, dist, exp = exp_run
    assert res[:3] == (m, s, dist)
    assert len(got) == len(exp), (len(got), len(exp))
    for k in exp.dtype.names:
        assert np.array_equal(got[k], exp[k]), (k, got[k], exp[k])
    assert got.tobytes() == exp.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("narrow", [True, False])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("profile", sorted(PROFILES))
def test_library_equals_oracle(profile, mode, narrow):
    d, hb, nibs, meta, runs = profile_data(profile)
    res, got = _device_run(hb, nibs, mode, narrow=narrow)
    _assert_equal(res, got, runs[mode])
    assert len(got) >= 3


@pytest.mark.gpu
@pytest.mark.parametrize("profile", sorted(PROFILES))
def test_stage0_pairs_grouped_as_the_scan(profile):
    """fetch_pairs(0): the pairs grouped into buckets and ordered as orc_scan's std::map does, colliding names merged"""
    import oracle_py as O
    from breakid_b200 import api
    d, hb, nibs, meta, runs = profile_data(profile)
    c = api.Context(hb.target_len, hb.target_names, device=0)
    c.push(hb)
    dist = runs[0][2]
    n = c.scan(dist)
    got = c.fetch_pairs(0)
    exp = O.scan(hb, 20, dist)
    assert n == len(exp) > 100
    for k in exp.dtype.names:
        assert np.array_equal(got[k], exp[k]), k
    c.close()


def _cuts(hb, meta, world):
    """cuts inside the side-1 region of ab_chrom_plain (between its spanning reads) and, for 3 ranks, inside the tid-24
    region of hi_header"""
    tid, pos = hb.cols["tid"], hb.cols["pos"]
    first = lambda m: int(np.nonzero(m)[0][0])
    j1, j2 = meta["ab_chrom_plain"], meta["hi_header"]
    c1 = first((tid == 0) & (pos >= j1["a"] - 300))
    c2 = first((tid == 24) & (pos >= j2["a"] - 300))
    return [0, c1, hb.n] if world == 2 else [0, c1, c2, hb.n]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("profile", ["b37", "collide", "hg38_like", "permuted", "punct"])
def test_sharded_equals_oracle(profile, mode, world):
    from breakid_b200 import api
    from test_multi_gloo import _slice
    d, hb, nibs, meta, runs = profile_data(profile)
    cuts = _cuts(hb, meta, world)
    assert all(a < b for a, b in zip(cuts[:-1], cuts[1:]))
    ctxs = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        c = api.Context(hb.target_len, hb.target_names, device=0, fast=mode)
        c.push(_slice(hb, a, b))
        for t, (p, l) in enumerate(nibs):
            c.set_nib(t, p, l)
        ctxs.append(c)
    res = api.dist_run_local(ctxs, mode)
    m, s, dist, exp = runs[mode]
    for r, c in enumerate(ctxs):
        assert res[r][:3] == (m, s, dist), r
        assert c.fetch_clusters().tobytes() == exp.tobytes(), r
        c.close()


@pytest.mark.gpu
def test_decoders_on_a_3366_target_header(tmp_path):
    """a BAM and a SAM whose header has 3366 @SQ lines of hg38 analysis-set names (*, :, = inside names): push_bgzf and
    push_sam give the host decoder's columns, RNAME / RNEXT / SA text included, and bkid_create succeeds"""
    from breakid_b200 import api, bamio, synth
    from test_sam_input import ALL, DENSE
    names = hg38_names()
    names[24:30] = ["HLA-A*01:01:01:01", "chr1=x*y:z", "chr1_KI270706v1_random", "chrUn_GL000220v1", "chrEBV", "chrM"]
    d, meta = build_names_batch(names)
    lens = LENS + [1000 + t for t in range(NT, len(names))]
    d = synth.SynthData(cfg=synth.SynthConfig(**dict(d.cfg.__dict__, chrom_lens=lens)), cols=d.cols, sa_rec=d.sa_rec,
                        cig_off=d.cig_off, cig_ops=d.cig_ops, sa_off=d.sa_off, sa_txt=d.sa_txt, truth={})
    bam, sam = str(tmp_path / "r.bam"), str(tmp_path / "r.sam")
    bamio.write_bam(bam, d, target_names=names)
    bamio.write_sam(sam, d, target_names=names)
    hb = api.HostBatch.from_bam(bam)
    assert hb.target_names == names
    t0 = time.time()
    ref = api.Context(hb.target_len, hb.target_names, device=0)
    t_create = time.time() - t0
    f = api.BgzfFile(bam)
    ref.push_bgzf(f)
    exp = {k: ref.fetch_column(k, dt) for k, dt in ALL}
    for k, dt in DENSE:
        assert np.array_equal(exp[k], hb.cols[k].astype(dt)), k
    assert bytes(exp["sa_txt"]) == bytes(hb.side["sa_txt"])
    sf = api.SamFile(sam)
    assert sf.target_names == names
    c = api.Context(hb.target_len, hb.target_names, device=0)
    assert c.push_sam(sf.text()) == hb.n
    sf.close()
    for k, _ in ALL:
        assert np.array_equal(c.fetch_column(k, dict(ALL)[k]), exp[k]), k
    print("bkid_create with %d targets: %.3f s" % (len(names), t_create))
    c.close(); ref.close(); f.close()


def _driver(tmp_path, inp, paths, tag, flags):
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    return subprocess.run([drv, "-i", inp, "-o", str(tmp_path / tag), "-n", paths["nib"], "-r", paths["refgene"]] + flags,
                          timeout=600, capture_output=True, text=True)


@pytest.mark.gpu
@pytest.mark.parametrize("profile", sorted(PROFILES))
def test_driver_on_named_bam_and_sam(tmp_path, profile):
    """BreakID -all on the BAM and on the SAM written with the profile's names (nib files and refGene rows named alike):
    the oracle's calls; with -x on a region named by the profile, the oracle's calls without that region's records;
    the reference binary's files where it is built"""
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio
    from test_golden import _format_calls
    from test_gpu_parity import _prefilter
    names = PROFILES[profile]
    d, hb, nibs, meta, runs = profile_data(profile)
    paths = bamio.write_dataset(str(tmp_path), d, sam=True, target_names=names)
    R.index(paths["bam"])
    for tag, inp in (("bam", paths["bam"]), ("sam", paths["sam"])):
        for mode in (0, 1):
            g = _driver(tmp_path, inp, paths, "%s%d" % (tag, mode), ["-all"] + (["-fast"] if mode else []))
            assert g.returncode == 0, (tag, g.stderr[-500:])
            R.match_oracle(str(tmp_path / ("%s%d" % (tag, mode))), d, mode=mode, target_names=names)
    # -x: drop the side-2 region of ab_chrom_plain and of same_header
    iv = [(meta["ab_chrom_plain"]["B"], meta["ab_chrom_plain"]["b"] - 3000, meta["ab_chrom_plain"]["b"] + 3000),
          (meta["same_header"]["B"], meta["same_header"]["b"] - 3000, meta["same_header"]["b"] + 3000)]
    bed = tmp_path / "x.bed"
    bed.write_text("".join("%s\t%d\t%d\n" % (names[t], b, e) for t, b, e in iv))
    tid, pos = hb.cols["tid"].astype(np.int64), hb.cols["pos"].astype(np.int64)
    keep = np.ones(hb.n, bool)
    for t, b, e in iv:
        keep &= ~((tid == t) & (pos >= b) & (pos < e))
    exp = O.run(_prefilter(hb, keep), nibs, mode=0)[3]
    g = _driver(tmp_path, paths["bam"], paths, "x", ["-all", "-x", str(bed)])
    assert g.returncode == 0, g.stderr[-500:]
    assert R.fusion_all_rows(str(tmp_path / "x")) == _format_calls(exp, names)
    assert len(exp) < len(runs[0][3]) or len(runs[0][3]) == 0
    if O.have_ref():
        O.ref_install_refgene(paths["refgene"])
        r = O.ref_run_binary(paths["bam"], str(tmp_path / "ref"), paths["nib"])
        assert r.returncode == 0, r.stderr[-500:]
        for suffix in ("_fusion.txt", "_fusion_all.txt"):
            assert open(str(tmp_path / "ref") + suffix).read() == open(str(tmp_path / "bam0") + suffix).read(), suffix


@pytest.mark.gpu
def test_create_at_hg38_size_and_refusal_on_device(tmp_path):
    """3366 targets: bkid_create succeeds; 50 000: it fails at once with the reason, and so does the driver (exit 1)"""
    from breakid_b200 import api, bamio, synth
    names = hg38_names()
    c = api.Context([100000] * len(names), names, device=0)
    c.close()
    n = 50000
    with pytest.raises(api.BkidError, match="at most 46339"):
        api.Context([1000] * n, ["c%d" % i for i in range(n)], device=0)
    d, meta = build_names_batch(PROFILES["canonical"])
    lens = [1000] * n
    lens[:NT] = LENS
    d = synth.SynthData(cfg=synth.SynthConfig(**dict(d.cfg.__dict__, chrom_lens=lens)), cols=d.cols, sa_rec=d.sa_rec,
                        cig_off=d.cig_off, cig_ops=d.cig_ops, sa_off=d.sa_off, sa_txt=d.sa_txt, truth={})
    os.makedirs(str(tmp_path / "nib"))
    names = PROFILES["canonical"] + ["c%d" % i for i in range(NT, n)]
    bamio.write_bam(str(tmp_path / "r.bam"), d, target_names=names)
    synth.write_ref_names(str(tmp_path / "nib" / "ref_names.txt"), n, target_names=names)
    t0 = time.time()
    g = _driver(tmp_path, str(tmp_path / "r.bam"), {"nib": str(tmp_path / "nib"), "refgene": str(tmp_path / "none.txt")}, "o", [])
    assert g.returncode == 1 and "header has 50000 targets; at most 46339" in g.stderr, (g.returncode, g.stderr[-500:])
    assert time.time() - t0 < 60
