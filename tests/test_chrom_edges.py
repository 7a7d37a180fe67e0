"""Every stage at the ends of chromosomes, on contigs shorter than a read or than the scan distance w, and with the
unmapped tail of a BAM, against the CPU oracle.

synth.generate keeps every read and breakpoint 2 kb away from both ends of its chromosome, so none of the device
branches that exist only for coordinates near 0 or near a chromosome's length is reached by the other tests.  Those
branches reproduce quirks of the reference: the +-2 breakpoint vote compares uint32 keys, so a key at x = 1 wraps and
gets no votes (src/BreakID.cc:820-821); a region start `mean - w` wraps and is clamped to 0; the depth window
[pos-1, pos) is clamped; a 41-mer base outside the nib repeats the previous base, starting from 'N'
(src/nibtools.cc:45-46); and a region past a chromosome's end must not pick up records of the next tid.

`edge_data` builds a small batch (about 18 000 records) that reaches all of them.  The CPU tests prove each edge is
actually reached with the oracle alone; the GPU tests require the device to equal the oracle byte for byte through the
library, the sharded path and the BreakID driver, in AHC and -fast mode."""
import os
import subprocess

import numpy as np
import pytest
import torch

L = 150
# chr1 and chr6 (the first and last tid) hold edge junctions; chr2 is shorter than a read, chr3 shorter than w; chr4 has
# records and split-read rows at its start, right after the short contigs (the "next tid" of a region past chr3's end);
# chr5 holds no record at all
LENS = [30000, 100, 600, 20000, 15000, 30000]
EMPTY = 4
SEED = 29

PAIRED, PROPER, UNMAP, MUNMAP, REVERSE, MREVERSE, READ1, READ2, SECONDARY, DUP = (
    0x1, 0x2, 0x4, 0x8, 0x10, 0x20, 0x40, 0x80, 0x100, 0x400)

# planted junctions: the left part ends at A:a on +, the right part starts at B:b (1-based).  `bs` lists the b of the
# split reads when they differ from b (keys at 1 and 3 only: see test_position_one_votes_differ_from_wrap_free_vote).
JUNCTIONS = {
    "x1_small": dict(A=5, a=10000, B=0, b=1, bs=(1, 3), n_span=14, n_split=40),       # p1 = chr1:1, k8_vote
    "x1_big": dict(A=5, a=20000, B=3, b=1, bs=(1, 3), n_span=14, n_split=300),        # p1 = chr4:1, k8_vote_big
    "y1_small": dict(A=0, a=15000, B=5, b=1, bs=(1, 3), n_span=14, n_split=30),       # p2 = chr6:1
    "chr1_end": dict(A=0, a=LENS[0] - 5, B=5, b=5000, n_span=14, n_split=20),         # 41-mer runs past chr1's end
    "chr6_end": dict(A=3, a=12000, B=5, b=LENS[5] - 15, n_span=14, n_split=20),       # 41-mer 5 bases past chr6's end
    "chr2_short": dict(A=1, a=95, B=5, b=25000, n_span=10, n_split=12, kmin=20),      # on a 100 bp contig
    "chr3_short": dict(A=2, a=592, B=0, b=22000, n_span=12, n_split=16),              # on a 600 bp contig, next tid chr4
}


def _sa_text(tid, pos1, cig):
    from breakid_b200 import synth
    return ("%s,%d,+,%s,60,0;" % (synth.chrom_name(tid), pos1, cig)).encode()


def _cigar_ops(txt):
    """'30M120S' -> BAM cigar ops (the encoder of test_gpu_parity._adversarial_sa_batch)"""
    ops, out, num = "MIDNSHP=X", [], ""
    for ch in txt:
        if ch.isdigit():
            num += ch
        else:
            out.append((int(num) << 4) | ops.index(ch)); num = ""
    return out


def build_edge_batch(seed=SEED):
    """the edge batch as synth.SynthData (so that it goes through HostBatch.from_synth and bamio.write_dataset alike);
    deterministic from `seed`"""
    from breakid_b200 import synth
    rng = np.random.RandomState(seed)
    recs = []                    # (flag, mapq, tid, pos, mtid, mpos, isize, endpos, name_id, sa or None)
    nid = [0]

    def name():
        nid[0] += 1
        return nid[0] - 1

    def proper(t, p1, ins):
        ln = LENS[t]
        p2 = p1 + ins - L
        if p2 >= ln:                                       # mate would start past the end: both at p1
            p2, ins = p1, L
        n = name()
        recs.append((PAIRED | PROPER | MREVERSE | READ1, 60, t, p1, t, p2, ins, p1 + L, n, None))
        recs.append((PAIRED | PROPER | REVERSE | READ2, 60, t, p2, t, p1, -ins, p2 + L, n, None))

    # background: proper pairs tile every populated chromosome, from pos 0 to the last base (reads overhang the end)
    for t, ln in enumerate(LENS):
        if t == EMPTY:
            continue
        npairs = max(10, ln * 30 // (2 * L))
        starts = np.concatenate([[0, ln - 1], rng.randint(0, ln, npairs - 2)])
        ins = np.clip(np.round(rng.randn(npairs) * 30 + 350), L + 1, 800).astype(np.int64)
        for p, i in zip(starts, ins):
            proper(t, int(p), int(i))
    # placed-unmapped mates, as aligners write them: at the mate's position, mapq 0, bam_endpos = pos + 1
    for t, p in [(0, 0), (0, 3), (0, LENS[0] - 1), (1, 0), (1, 99), (2, 0), (2, 599), (3, 1), (5, LENS[5] - 1)] + \
            [(0, int(x)) for x in rng.randint(0, 400, 6)] + [(5, int(x)) for x in rng.randint(LENS[5] - 400, LENS[5], 6)]:
        n = name()
        recs.append((PAIRED | MUNMAP | READ1, 60, t, p, t, p, 0, p + L, n, None))
        recs.append((PAIRED | UNMAP | READ2, 0, t, p, t, p, 0, p + 1, n, None))

    for j in JUNCTIONS.values():
        A, a, B, b = j["A"], j["a"], j["B"], j["b"]
        for _ in range(j["n_span"]):                      # discordant spanning pairs (flags 97 / 145)
            r1 = int(np.clip(a - L - rng.randint(0, 250), 0, LENS[A] - 1))
            r2 = int(np.clip(b - 1 + rng.randint(0, 250), 0, LENS[B] - 1))
            n = name()
            recs.append((PAIRED | MREVERSE | READ1, 60, A, r1, B, r2, 0, r1 + L, n, None))
            recs.append((PAIRED | REVERSE | READ2, 60, B, r2, A, r1, 0, r2 + L, n, None))
        bs = j.get("bs", (b,))
        for s in range(j["n_split"]):                      # split reads: kM(L-k)S primary + kS(L-k)M 0x100 record
            k = int(rng.randint(j.get("kmin", L // 2 + 1), min(L - 20, a + 1)))
            bb = bs[s % len(bs)]
            ppos = a - k                                   # 0-based start of the primary
            mate = min(ppos + 200, LENS[A] - 1)
            n = name()
            recs.append((PAIRED | PROPER | MREVERSE | READ1, 60, A, ppos, A, mate, 200 + L, ppos + k, n,
                         ("%dM%dS" % (k, L - k), _sa_text(B, bb, "%dS%dM" % (k, L - k)))))
            recs.append((PAIRED | PROPER | REVERSE | READ2, 60, A, mate, A, ppos, -(200 + L), mate + L, n, None))
            recs.append((PAIRED | PROPER | MREVERSE | READ1 | SECONDARY, 60, B, bb - 1, A, mate, 0, bb - 1 + L - k, n,
                         ("%dS%dM" % (k, L - k), _sa_text(A, a - k + 1, "%dM%dS" % (k, L - k)))))
    # the unmapped tail: tid = -1, pos = -1, mtid = -1
    for _ in range(40):
        n = name()
        recs.append((PAIRED | UNMAP | MUNMAP | READ1, 0, -1, -1, -1, -1, 0, 0, n, None))
        recs.append((PAIRED | UNMAP | MUNMAP | READ2, 0, -1, -1, -1, -1, 0, 0, n, None))

    # coordinate sort, tid < 0 last (samtools order), stable
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
    return synth.SynthData(cfg=cfg, cols=cols, sa_rec=i64(sa_rec), cig_off=i64(cig_off), cig_ops=i64(cig), sa_off=i64(sa_off),
                           sa_txt=torch.tensor(list(txt), dtype=torch.uint8), truth={})


def nibs_for(d):
    from breakid_b200 import synth
    return [(synth.random_nib_bytes(l, d.cfg.seed * 1000 + t).numpy(), l) for t, l in enumerate(d.cfg.chrom_lens)]


@pytest.fixture(scope="module")
def edge_data():
    import oracle_py as O
    from breakid_b200 import api
    d = build_edge_batch()
    hb = api.HostBatch.from_synth(d)
    nibs = nibs_for(d)
    runs = {mode: O.run(hb, nibs, mode=mode) for mode in (0, 1)}
    return d, hb, nibs, runs


def _call(cl, name):
    """the call of junction `name` (its chromosomes and breakpoints within 5 bp, either side first)"""
    j = JUNCTIONS[name]
    x = {(j["A"], j["B"]): (j["a"], j["b"]), (j["B"], j["A"]): (j["b"], j["a"])}
    hit = [c for c in cl if (int(c["p1_tid"]), int(c["p2_tid"])) in x and
           abs(int(c["p1_exact_pos"]) - x[(int(c["p1_tid"]), int(c["p2_tid"]))][0]) <= 5 and
           abs(int(c["p2_exact_pos"]) - x[(int(c["p1_tid"]), int(c["p2_tid"]))][1]) <= 5]
    assert len(hit) == 1, (name, len(hit))
    return hit[0]


def _region(mean, w):
    return (int(mean) - w) & 0xFFFFFFFF, (int(mean) + w) & 0xFFFFFFFF


def _entries(hb, c, w):
    """the (x, y) evidence entries the oracle's vote of call c counts: side-1 rows matched by name and fields with side-2
    rows (src/BreakID.cc:627-637), oriented by p1's chromosome"""
    import oracle_py as O
    e1 = O.find_sa_reads(hb, int(c["p1_tid"]), *_region(c["p1_mean_pos"], w))
    e2 = O.find_sa_reads(hb, int(c["p2_tid"]), *_region(c["p2_mean_pos"], w))
    fields = ("name_lo", "name_hi", "primary_chr", "secondary_chr", "primary_start", "secondary_start", "primary_end",
              "secondary_end", "primary_cigar_h", "secondary_cigar_h", "primary_bp", "secondary_bp")
    side2 = {}
    for r in e2:
        side2.setdefault((tuple(int(r[f]) for f in fields), int(r["secondary"])), []).append(r)
    out = []
    for a in e1:
        key = tuple(int(a[f]) for f in fields)
        for _ in side2.get((key, 1 - int(a["secondary"])), []):
            if int(a["primary_chr"]) == int(c["p1_tid"]):
                out.append((int(a["primary_bp"]), int(a["secondary_bp"])))
            else:
                out.append((int(a["secondary_bp"]), int(a["primary_bp"])))
    return np.array(out, np.int64).reshape(-1, 2)


def _wrap_free_vote(ent, err=2):
    """the +-2 vote with signed 64-bit windows: first strict maximum in key-string order"""
    keys = sorted({(int(x), int(y)) for x, y in ent}, key=lambda k: "%d,%d" % k)
    best, call = 0, None
    for kx, ky in keys:
        n = int(((np.abs(ent[:, 0] - kx) <= err) & (np.abs(ent[:, 1] - ky) <= err)).sum())
        if n > best:
            best, call = n, (kx, ky)
    return call, best


def _longest_run(s):
    best, i = 0, 0
    while i < len(s):
        j = i
        while j < len(s) and s[j] == s[i]:
            j += 1
        best, i = max(best, j - i), j
    return best


# ------------------------------------------------------------------------------------------------ CPU: edges are reached
def test_batch_shape(edge_data):
    d, hb, nibs, runs = edge_data
    tid, pos = hb.cols["tid"].astype(np.int64), hb.cols["pos"].astype(np.int64)
    assert np.array_equal(np.lexsort((pos, tid.astype(np.uint32))), np.arange(hb.n))   # coordinate sorted, tid < 0 last
    tail = np.nonzero(tid < 0)[0]
    assert len(tail) == 80 and tail[0] == hb.n - 80 and np.all(pos[tail] == -1) and np.all(hb.cols["mtid"][tail] == -1)
    assert (tid == EMPTY).sum() == 0 and (tid == EMPTY - 1).sum() > 0 and (tid == EMPTY + 1).sum() > 0
    assert 10000 < hb.n < 60000
    ln = np.asarray(LENS, np.int64)[np.maximum(tid, 0)]
    mapped = (hb.cols["flag"] & UNMAP) == 0
    assert np.any((pos == 0) & mapped & (tid == 0)) and np.any((hb.cols["endpos"] > ln) & mapped & (tid >= 0))
    unm = (hb.cols["flag"] & UNMAP) != 0
    placed = unm & (tid >= 0)
    assert placed.sum() >= 20 and np.all(hb.cols["endpos"][placed] == pos[placed] + 1) and np.all(hb.cols["mapq"][unm] == 0)
    assert set(hb.narrow()) == {"span16", "isize16", "tid_run_start", "tid_run_tid"}


@pytest.mark.parametrize("name,size", [("x1_small", "small"), ("x1_big", "big"), ("y1_small", "small")])
def test_position_one_votes_differ_from_wrap_free_vote(edge_data, name, size):
    """keys only at 1 and 3 on the wrapping side: both windows hold every entry, so a wrap-free vote ties and calls 1
    (key string "1,..." first); the reference's uint32 window gives key 1 no votes and calls 3"""
    import oracle_py as O
    d, hb, nibs, runs = edge_data
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        w = int(dist)
        c = _call(cl, name)
        ent = _entries(hb, c, w)
        assert (len(ent) <= 256) if size == "small" else (len(ent) > 256), len(ent)
        assert int(c["n_split_read"]) == len(ent)
        side = 0 if name.startswith("x") else 1
        assert set(ent[:, side].tolist()) == {1, 3} and len(set(ent[:, 1 - side].tolist())) == 1
        free, nfree = _wrap_free_vote(ent)
        got = (int(c["p1_exact_pos"]), int(c["p2_exact_pos"]))
        assert free[side] == 1 and got[side] == 3 and free[1 - side] == got[1 - side] and nfree == len(ent)
        fb = O.find_bp(hb, int(c["p1_tid"]), *_region(c["p1_mean_pos"], w), int(c["p2_tid"]), *_region(c["p2_mean_pos"], w))
        assert fb == (len(ent),) + got


def test_region_start_wraps(edge_data):
    d, hb, nibs, runs = edge_data
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        w = int(dist)
        low = [c for c in cl if int(c["p1_mean_pos"]) < w or int(c["p2_mean_pos"]) < w]
        assert len(low) >= 4, len(low)
        assert int(_call(cl, "x1_small")["p1_mean_pos"]) < w and int(_call(cl, "y1_small")["p2_mean_pos"]) < w


def test_end_of_chromosome_trap_is_armed(edge_data):
    """the chr3 call (600 bp contig) has its coverage region and depth window on chr3 only; chr4 right after it has
    records under both, so a bound that crossed into the next tid would count them"""
    import oracle_py as O
    d, hb, nibs, runs = edge_data
    tid, pos, end = hb.cols["tid"], hb.cols["pos"].astype(np.int64), hb.cols["endpos"].astype(np.int64)
    f, q = hb.cols["flag"], hb.cols["mapq"]
    m, s, dist, cl = runs[0]
    w = int(dist)
    for name, t in (("chr3_short", 2), ("chr2_short", 1)):
        c = _call(cl, name)
        side = 1 if int(c["p1_tid"]) == t else 2
        mean = int(c["p%d_mean_pos" % side])
        beg, stop = max(mean - w, 0), mean + w
        assert stop > LENS[t]                                            # the region runs past the contig's end
        over = (pos < stop) & (end > beg)
        assert over[tid == t].sum() >= 5 and over[tid == t + 1].sum() > 0    # tid-aware coverage != tid-blind count
        bp = int(c["p%d_exact_pos" % side])
        dep = O.single_base_depth(hb, t, bp)
        ok = (q > 0) & ((f & DUP) == 0) & ((f & PAIRED) != 0) & (pos < bp) & (end > bp - 1)
        assert dep == ok[tid == t].sum() == float(c["p%d_bp_depth" % side])
        assert ok[tid >= 0].sum() > dep                                  # a tid-blind depth picks up the next tid


def test_41mers_padded_at_both_ends(edge_data):
    import oracle_py as O
    d, hb, nibs, runs = edge_data
    for mode in (0, 1):
        cl = runs[mode][3]
        lead, trail = 0, 0
        for c in cl:
            for side in (1, 2):
                s = bytes(c["p%d_rpt" % side])
                t, bp = int(c["p%d_tid" % side]), int(np.int64(c["p%d_exact_pos" % side]))
                assert s == O.neighbor_41(nibs[t][0], LENS[t], bp) and len(s) == 41
                if bp <= 10:
                    assert s[:21 - bp] == b"N" * (21 - bp) and c["is_rpt"] == 1
                    lead += 1
                if bp >= LENS[t] - 9:
                    pad = bp + 20 - LENS[t]
                    assert len(set(s[-pad - 1:])) == 1 and c["is_rpt"] == 1
                    trail += 1
        assert lead >= 3 and trail >= 3, (lead, trail)
        c = _call(cl, "chr6_end")                                        # 5 padded bases: shorter than a run
        assert int(c["p2_exact_pos"]) == LENS[5] - 15
        s = bytes(c["p2_rpt"])
        assert len(set(s[-6:])) == 1 and _longest_run(s) <= 10 and _longest_run(bytes(c["p1_rpt"])) <= 10 and c["is_rpt"] == 0


def test_calls_on_short_contigs(edge_data):
    d, hb, nibs, runs = edge_data
    for mode in (0, 1):
        cl = runs[mode][3]
        for name, t in (("chr2_short", 1), ("chr3_short", 2)):
            c = _call(cl, name)
            assert t in (int(c["p1_tid"]), int(c["p2_tid"]))
        assert not any(EMPTY in (int(c["p1_tid"]), int(c["p2_tid"])) for c in cl)
        assert len(cl) == len(JUNCTIONS)


# ------------------------------------------------------------------------------------------------ GPU: device == oracle
def _device_run(hb, nibs, mode, narrow=True, exclude=None):
    from breakid_b200 import api
    c = api.Context(hb.target_len, hb.target_names, device=0, fast=mode)
    c.push(hb, narrow=narrow)
    if exclude is not None:
        c.set_exclude(exclude[:, 0], exclude[:, 1], exclude[:, 2])
    for t, (p, l) in enumerate(nibs):
        if p is not None:
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
def test_library_path_equals_oracle(edge_data, mode, narrow):
    d, hb, nibs, runs = edge_data
    res, got = _device_run(hb, nibs, mode, narrow=narrow)
    _assert_equal(res, got, runs[mode])
    assert len(got) == len(JUNCTIONS)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_nib_shorter_than_target_and_missing_nib(edge_data, mode):
    """chr6's nib ends 30 bases before its target length (the chr6_end 41-mer then runs into the padding) and chr2 has
    no nib (its 41-mers stay empty)"""
    import oracle_py as O
    d, hb, nibs, runs = edge_data
    var = list(nibs)
    short = LENS[5] - 30
    var[5] = (nibs[5][0][:(short + 1) // 2].copy(), short)
    var[1] = (None, 0)
    exp = O.run(hb, var, mode=mode)
    res, got = _device_run(hb, var, mode)
    _assert_equal(res, got, exp)
    c, full = _call(exp[3], "chr6_end"), _call(runs[mode][3], "chr6_end")
    assert c["is_rpt"] == 1 and full["is_rpt"] == 0 and bytes(c["p2_rpt"]).endswith(bytes(c["p2_rpt"])[-36:-35] * 36)
    c = _call(exp[3], "chr2_short")
    assert bytes(c["p1_rpt"]) == b"" and len(bytes(c["p2_rpt"])) == 41


def _edge_intervals():
    """[0, k) and [len - k, len) on the edge chromosomes and the whole of the 100 bp contig"""
    return np.array([(0, 0, 2), (0, LENS[0] - 40, LENS[0]), (5, 0, 1), (5, LENS[5] - 12, LENS[5]), (3, 0, 2),
                     (1, 0, LENS[1]), (2, 0, 300)], np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_exclude_intervals_at_chromosome_ends(edge_data, mode):
    """device-side exclusion == the oracle on the pre-filtered batch (test_gpu_parity pattern).  [0, 2) on chr1 and chr4
    drops the split reads whose right part starts at 1, so the position-1 votes change; chr2 disappears"""
    import oracle_py as O
    from test_gpu_parity import _prefilter
    d, hb, nibs, runs = edge_data
    iv = _edge_intervals()
    tid, pos = hb.cols["tid"].astype(np.int64), hb.cols["pos"].astype(np.int64)
    keep = np.ones(hb.n, bool)
    for t, b, e in iv:
        keep &= ~((tid == t) & (pos >= max(b, 0)) & (pos < e))
    exp = O.run(_prefilter(hb, keep), nibs, mode=mode)
    res, got = _device_run(hb, nibs, mode, exclude=iv)
    _assert_equal(res, got, exp)
    assert not any(1 in (int(c["p1_tid"]), int(c["p2_tid"])) for c in got)
    before = {(int(c["p1_tid"]), int(c["p2_tid"]), int(c["p1_exact_pos"]), int(c["p2_exact_pos"]), int(c["n_split_read"])) for c in runs[mode][3]}
    after = {(int(c["p1_tid"]), int(c["p2_tid"]), int(c["p1_exact_pos"]), int(c["p2_exact_pos"]), int(c["n_split_read"])) for c in got}
    assert len(after) >= 4 and len(before - after) >= 3


def _cut_points(hb, kind):
    tid, pos = hb.cols["tid"], hb.cols["pos"]
    first = lambda m: int(np.nonzero(m)[0][0])
    tail = first(tid < 0)
    if kind == "chr1_head":                       # inside the first w bases of chr1 (x1_small): coverage / depth split
        return [0, first((tid == 0) & (pos >= 2)), hb.n]
    if kind == "boundary_tail":                   # at the chr3 / chr4 boundary; the last rank holds little more than the tail
        return [0, first(tid == 3), tail - 5, hb.n]
    return [0, first((tid == 3) & (pos >= 2)), first(tid == 5), hb.n]    # inside chr4's head (x1_big), at the chr6 boundary


@pytest.mark.gpu
@pytest.mark.parametrize("kind,mode", [("chr1_head", 0), ("chr1_head", 1), ("boundary_tail", 0), ("boundary_tail", 1), ("chr4_head", 0)])
def test_sharded_cuts_at_edges_equal_oracle(edge_data, kind, mode):
    """ranks as threads (api.dist_run_local), the record stream cut at chromosome boundaries, inside the first w bases of
    a chromosome with a position-1 cluster, and just before the unmapped tail: every rank equals the oracle"""
    from breakid_b200 import api
    from test_multi_gloo import _slice
    d, hb, nibs, runs = edge_data
    cuts = _cut_points(hb, kind)
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
    assert len(exp) == len(JUNCTIONS)
    for r, c in enumerate(ctxs):
        assert res[r][:3] == (m, s, dist), r
        assert c.fetch_clusters().tobytes() == exp.tobytes(), r
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["ahc", "fast"])
def test_driver_on_edge_bam(tmp_path, edge_data, mode):
    """the batch written as a BAM (placed-unmapped mates, the unmapped tail, an empty chromosome, contigs shorter than a
    read): BreakID -all with device decode and with the host decoder writes the oracle's calls, and the reference
    binary's files where it is built"""
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio
    d, hb, nibs, runs = edge_data
    paths = bamio.write_dataset(str(tmp_path), d)
    R.index(paths["bam"])
    flags = ["-all"] + (["-fast"] if mode == "fast" else [])
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    for tag, env in (("gpu", None), ("gpu_host", dict(os.environ, BKID_HOST_DECODE="1"))):
        g = subprocess.run([drv, "-i", paths["bam"], "-o", str(tmp_path / tag), "-n", paths["nib"], "-r", paths["refgene"]] + flags,
                           timeout=600, capture_output=True, text=True, env=env)
        assert g.returncode == 0, (tag, g.stderr[-500:])
        R.match_oracle(str(tmp_path / tag), d, mode=int(mode == "fast"))
        assert len(R.fusion_all_rows(str(tmp_path / tag))) == len(JUNCTIONS)
    assert open(str(tmp_path / "gpu") + "_fusion_all.txt").read() == open(str(tmp_path / "gpu_host") + "_fusion_all.txt").read()
    if O.have_ref():
        O.ref_install_refgene(paths["refgene"])
        r = O.ref_run_binary(paths["bam"], str(tmp_path / "ref"), paths["nib"], fast=(mode == "fast"))
        assert r.returncode == 0, r.stderr[-500:]
        for suffix in ("_fusion.txt", "_fusion_all.txt"):
            assert open(str(tmp_path / "ref") + suffix).read() == open(str(tmp_path / "gpu") + suffix).read(), suffix
