"""Split-read refinement (k7_collect, k8_vote, k8_vote_big, k9_depth, k10_finish) through every gate, pairing rule and
vote form, against the CPU oracle.

The other suites compare whole runs, and synth plants breakpoints well inside a chromosome with a few bases of jitter, so
most of the branches of the refinement stage are reached by chance or not at all.  `build_refine_batch` plants one
junction per rung on four chromosomes: two with a background of proper pairs, and two quiet ones that hold nothing but
the records of the gate rungs, so their coverage can be counted exactly.  The rungs are:

  * vote forms: clusters of m = 1, 2, 255, 256, 257 (k8_vote up to 256 entries, k8_vote_big above), 8192, 8193
    (k8_vote_big sorts in shared memory up to 8192 keys, in global memory beyond) and about 20 000 entries, and a read
    name with three rows on side 1 and two on side 2 (the reference pairs them as a full product);
  * ties: keys whose votes tie at the top across a digit-count boundary in x (9999 / 10000) and in y, and with the same
    digit count (first and last maximum differ).  The reference keeps the first strict maximum in the order of the key
    strings "x,y" (std::map<std::string,int>, src/BreakID.cc:806-855), which differs from numeric order there;
  * gates: total coverage 4 and 5 with 2 evidence rows, 1 and 2 evidence rows at coverage >= 5, on side 1 and on side 2
    behind a side 1 that passes (src/BreakID.cc:1032-1035); the coverage is made of MAPQ-0, duplicate, secondary,
    placed-unmapped and long-span (large N) records, the last reaching the region only through the maxspan look-back;
    best votes of exactly 1 and 2 (src/BreakID.cc:446);
  * the fatal "error cigar" record (src/BreakID.cc:954-968) outside every region, behind a side 1 that fails its gate
    and in a cluster dropped as close (all silent), and inside a collected region on side 1 or side 2 (BKID_ERR_CIGAR);
  * a call whose breakpoint depth is 0 (its reads have MAPQ 0), so its allele frequency is inf;
  * a rung whose SA cigars are complementary only within 3, 5 or 20 bases (mismatch_num).

`pairing_batch` is a library-only variant whose read-name hashes and OC tags are set in the HostBatch: rows that agree in
everything but the high word of name_lo, name_hi, the secondary flag, a chromosome, a cigar text or a breakpoint.  The
start and end fields cannot differ alone (see _plant_pairing).

The CPU tests prove with the oracle alone that each rung is reached and sits at its threshold; the GPU tests require the
device to equal the oracle byte for byte through the library, the sharded path and the BreakID driver."""
import os
import subprocess

import numpy as np
import pytest
import torch

from test_chrom_edges import _cigar_ops, _entries, _region, _wrap_free_vote

L = 150
Q1, BG1, BG2, Q2 = 0, 1, 2, 3          # quiet, background, background, quiet
LENS = [220000, 420000, 420000, 160000]
SEED = 41

PAIRED, PROPER, UNMAP, MUNMAP, REVERSE, MREVERSE, READ1, READ2, SECONDARY, DUP = (
    0x1, 0x2, 0x4, 0x8, 0x10, 0x20, 0x40, 0x80, 0x100, 0x400)

VOTE_SIZES = {"m1": 1, "m2": 2, "m255": 255, "m256": 256, "m257": 257, "m8192": 8192, "m8193": 8193, "m20k": 19997}
EXTRA_KINDS = ("mapq0", "dup", "secondary", "unmapped", "longspan")
SMALL_RUNGS = ("m1", "m2", "tie_y", "tie_first", "g1_cov4", "g1_cov5_longspan", "g2_ev1", "vote1", "vote2", "product")
PAIR_FIELDS = ("name_lo_hi32", "name_hi", "secondary", "pcig", "scig", "pchr", "schr", "pbp", "sbp")


def _err_code(name):
    """a status code of the C ABI, read from include/breakid_b200.h"""
    import re
    hdr = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "breakid_b200.h")
    return int(re.search(r"\b%s\s*=\s*(-?\d+)" % name, open(hdr).read()).group(1))


BKID_ERR_CIGAR = _err_code("BKID_ERR_CIGAR")


def _sa(tid, pos1, cig):
    from breakid_b200 import synth
    return ("%s,%d,+,%s,60,0;" % (synth.chrom_name(tid), pos1, cig)).encode()


class _Builder:
    """records as (flag, mapq, tid, pos, mtid, mpos, isize, endpos, name_id, (cigar, SA text[, OC text]) or None,
    hash tweak)"""

    def __init__(self, seed):
        self.rng = np.random.RandomState(seed)
        self.recs, self.nid, self.meta = [], 0, {}

    def name(self):
        self.nid += 1
        return self.nid - 1

    def add(self, flag, mapq, tid, pos, mtid, mpos, isize, endpos, n, sa=None, tweak=None):
        self.recs.append((flag, mapq, tid, pos, mtid, mpos, isize, endpos, n, sa, tweak))

    def background(self, t, cov=10):
        ln = LENS[t]
        npairs = ln * cov // (2 * L)
        starts = self.rng.randint(0, ln - 1000, npairs)
        ins = np.clip(np.round(self.rng.randn(npairs) * 30 + 350), L + 1, 800).astype(np.int64)
        for p1, i in zip(starts.tolist(), ins.tolist()):
            p2 = p1 + i - L
            n = self.name()
            self.add(PAIRED | PROPER | MREVERSE | READ1, 60, t, p1, t, p2, i, p1 + L, n)
            self.add(PAIRED | PROPER | REVERSE | READ2, 60, t, p2, t, p1, -i, p2 + L, n)

    def span(self, A, a, B, b, n):
        """n discordant pairs (flags 97 / 145) around the junction; the A reads end at a-1 or before, so they never
        cover the breakpoint base a"""
        p1s, p2s = [], []
        for _ in range(n):
            r1 = a - L - 1 - int(self.rng.randint(0, 250))
            r2 = b - 1 + int(self.rng.randint(0, 250))
            if A == B:
                r2 = b + 200 + int(self.rng.randint(0, 250))
            k = self.name()
            self.add(PAIRED | MREVERSE | READ1, 60, A, r1, B, r2, 0, r1 + L, k)
            self.add(PAIRED | REVERSE | READ2, 60, B, r2, A, r1, 0, r2 + L, k)
            p1s.append(r1 + 1); p2s.append(r2 + 1)
        return p1s, p2s

    def split(self, A, x, B, y, mapq=60, d=0, flip=False, n_prim=1, n_sec=1, k=None, n=None,
              prim_sa=None, sec_sa=None, prim_tweak=None, sec_tweak=None, sec_primary=False):
        """one split read: the left part ends at A:x on +, the right part starts at B:y (1-based), entry (x, y).
        Normally the primary record (kM(L-k)S) lies on A and the 0x100 record (kS(L-k)M) on B; flip swaps which of the
        two parts is the primary.  d shifts the clip of the right part's cigar (complementary within |d| bases).
        n_prim / n_sec: copies of the two records under the same name.  prim_sa / sec_sa replace the SA text of the
        record on A / on B (a decoy that differs in one row field); *_tweak change the name hash of that record in the
        library-only batch; sec_primary drops the 0x100 flag of the B record (two primaries)."""
        if k is None:
            k = int(self.rng.randint(L // 2 + 1, L - 20))
        if n is None:
            n = self.name()
        left, right = "%dM%dS" % (k, L - k), "%dS%dM" % (k + d, L - k - d)
        fa = PAIRED | PROPER | MREVERSE | READ1 | (SECONDARY if flip else 0)
        fb = PAIRED | PROPER | MREVERSE | READ1 | (0 if (flip or sec_primary) else SECONDARY)
        for _ in range(n_prim if not flip else n_sec):
            self.add(fa, mapq, A, x - k, A, x - k + 200, 0 if flip else 200 + L, x, n,
                     (left, prim_sa if prim_sa is not None else _sa(B, y, right)), prim_tweak)
        for _ in range(n_sec if not flip else n_prim):
            self.add(fb, mapq, B, y - 1, A, x - k + 200, 200 + L if flip else 0, y - 1 + L - k - d, n,
                     (right, sec_sa if sec_sa is not None else _sa(A, x - k + 1, left)), sec_tweak)
        return n

    def extra(self, kind, t, p):
        """one record that counts toward the coverage of a region holding p, and is no evidence row"""
        n = self.name()
        if kind == "mapq0":
            self.add(PAIRED | PROPER | MREVERSE | READ1, 0, t, p, t, p + 200, 200 + L, p + L, n)
        elif kind == "dup":
            self.add(PAIRED | PROPER | MREVERSE | READ1 | DUP, 60, t, p, t, p + 200, 200 + L, p + L, n)
        elif kind == "secondary":
            self.add(PAIRED | PROPER | MREVERSE | READ1 | SECONDARY, 60, t, p, t, p + 200, 0, p + L, n)
        elif kind == "unmapped":              # placed at its mate's position, as aligners write it
            self.add(PAIRED | UNMAP | READ2, 0, t, p, t, p, 0, p + 1, n)
        elif kind == "longspan":              # starts 4 kb before the breakpoint, ends 400 b before it
            self.add(PAIRED | PROPER | MREVERSE | READ1, 60, t, p - 4000, t, p + 200, 200 + L, p - 400, n,
                     ("50M3450N100M", _sa(t, p + 5000, "50S100M")))
        else:
            raise ValueError(kind)

    def fatal(self, t, p):
        """a complementary split alignment whose SA cigar has no clip after merging (own 5M145S, SA 75M75M)"""
        n = self.name()
        self.add(PAIRED | PROPER | MREVERSE | READ1, 60, t, p, t, p + 200, 200 + L, p + 5, n, ("5M145S", _sa(t, p + 3000, "75M75M")))

    def junction(self, name, A, a, B, b, n_span):
        p1s, p2s = self.span(A, a, B, b, n_span)
        self.meta[name] = dict(A=A, a=a, B=B, b=b, p1_mean=int(sum(p1s) / len(p1s)), p2_mean=int(sum(p2s) / len(p2s)))


class _Slots:
    """junction positions 15 kb apart on every chromosome, around the reserved ones"""

    def __init__(self, reserved):
        self.next = {t: 25000 for t in range(len(LENS))}
        self.reserved = reserved

    def __call__(self, t):
        p = self.next[t]
        while any(abs(p - r) < 12000 for r in self.reserved.get(t, ())):
            p += 15000
        self.next[t] = p + 15000
        assert p < LENS[t] - 15000, (t, p)
        return p


def _plant(B, rungs):
    """the rungs of the main batch (all of them, or the names in `rungs`)"""
    rng = B.rng
    want = lambda r: rungs is None or r in rungs
    slot = _Slots({BG1: (10000, 100000), BG2: (100000,)})

    # ---- vote forms: m entries with keys jittered by up to 15 bases in x and y
    for r, m in VOTE_SIZES.items():
        if not want(r):
            continue
        a, b = slot(BG1), slot(BG2)
        B.junction(r, BG1, a, BG2, b, 12)
        if m <= 2:
            for _ in range(m):
                B.split(BG1, a, BG2, b)
            if m == 1:                     # one more evidence row on each side that pairs with nothing
                B.split(BG1, a, BG2, b + 9000, n_sec=0)
                B.split(BG1, a - 9000, BG2, b, n_prim=0)
        else:
            jx, jy = rng.randint(-15, 16, m), rng.randint(-15, 16, m)
            for i in range(m):
                B.split(BG1, a + int(jx[i]), BG2, b + int(jy[i]), flip=bool(i % 5 == 0))
    if want("product"):                    # 3 rows on side 1 x 2 rows on side 2 of one name, + 2 plain split reads
        a, b = slot(BG1), slot(BG2)
        B.junction("product", BG1, a, BG2, b, 12)
        B.split(BG1, a + 4, BG2, b, n_prim=3, n_sec=2)
        B.split(BG1, a, BG2, b)
        B.split(BG1, a, BG2, b)

    # ---- ties: every key's window holds every entry, so all keys tie; the key that wins in string order occurs once
    if want("tie_x"):                      # "10000,y" < "9999,y"; 256 entries: every k8_vote thread holds two
        b = slot(BG2)
        B.junction("tie_x", BG1, 10000, BG2, b, 12)
        B.split(BG1, 10000, BG2, b)
        for i in range(255):
            B.split(BG1, 9999, BG2, b, flip=bool(i % 3 == 0))
    if want("tie_y"):                      # "x,100000" < "x,99999"; 100 entries over all four warps
        a = slot(BG1)
        B.junction("tie_y", BG1, a, BG2, 100000, 12)
        B.split(BG1, a, BG2, 100000)
        for i in range(99):
            B.split(BG1, a, BG2, 99999, flip=bool(i % 4 == 0))
    if want("tie_first"):                  # same digit counts: the first maximum (x = a) differs from the last (a + 1)
        a, b = slot(BG1), slot(BG2)
        B.junction("tie_first", BG1, a, BG2, b, 12)
        B.split(BG1, a, BG2, b)
        for _ in range(39):
            B.split(BG1, a + 1, BG2, b)
    if want("tie_big"):                    # k8_vote_big: "100000,y" < "99999,y"
        b = slot(BG2)
        B.junction("tie_big", BG1, 100000, BG2, b, 12)
        B.split(BG1, 100000, BG2, b)
        for i in range(299):
            B.split(BG1, 99999, BG2, b, flip=bool(i % 2 == 0))

    # ---- gates on side 1 (quiet chr1 is p1): coverage = 2 spanning reads + evidence rows + extra records
    def gate1(r, n_ev, extras, product=False):
        a, b = slot(Q1), slot(BG2)
        B.junction(r, Q1, a, BG2, b, 2)
        if product:                        # one row on side 1 that pairs with two rows on side 2
            B.split(Q1, a, BG2, b, n_sec=2)
        else:
            for _ in range(n_ev):
                B.split(Q1, a, BG2, b)
        for i, kind in enumerate(extras):
            B.extra(kind, Q1, a - 200 - 37 * i)
        return a, b
    if want("g1_cov4"):
        a, b = gate1("g1_cov4", 2, ())
        B.fatal(BG2, b + 100)              # side 2 of a cluster whose side 1 fails: never read
    for kind in EXTRA_KINDS:
        if want("g1_cov5_" + kind):
            gate1("g1_cov5_" + kind, 2, (kind,))
    if want("g1_ev1"):
        gate1("g1_ev1", 1, ("mapq0", "dup"), product=True)
    if want("g1_ev2"):
        gate1("g1_ev2", 2, ("mapq0", "dup", "unmapped"))

    # ---- gates on side 2 (quiet chr4 is p2) behind a side 1 on background
    def gate2(r, n_ev, extras, product=False):
        a, b = slot(BG1), slot(Q2)
        B.junction(r, BG1, a, Q2, b, 2)
        if product:                        # two rows on side 1 that pair with one row on side 2
            B.split(BG1, a, Q2, b, n_prim=2)
        else:
            for _ in range(n_ev):
                B.split(BG1, a, Q2, b)
        for i, kind in enumerate(extras):
            B.extra(kind, Q2, b + 300 + 41 * i)
    if want("g2_cov4"):
        gate2("g2_cov4", 2, ())
    if want("g2_cov5"):
        gate2("g2_cov5", 2, ("longspan",))
    if want("g2_ev1"):
        gate2("g2_ev1", 1, ("secondary", "unmapped"), product=True)
    if want("g2_ev2"):
        gate2("g2_ev2", 2, ("mapq0", "secondary", "unmapped"))

    # ---- votes of exactly 1 (two keys 10 apart) and exactly 2
    if want("vote1"):
        a, b = slot(BG1), slot(BG2)
        B.junction("vote1", BG1, a, BG2, b, 12)
        B.split(BG1, a, BG2, b)
        B.split(BG1, a + 10, BG2, b + 10)
    if want("vote2"):
        a, b = slot(BG1), slot(BG2)
        B.junction("vote2", BG1, a, BG2, b, 12)
        B.split(BG1, a, BG2, b)
        B.split(BG1, a + 2, BG2, b - 2, flip=True)
        B.split(BG1, a + 7, BG2, b)

    # ---- cigars complementary within 0, 3, 5 and 20 bases, at keys 10 and 20 bases apart
    if want("mismatch"):
        a, b = slot(BG1), slot(BG2)
        B.junction("mismatch", BG1, a, BG2, b, 12)
        for dd, cnt, off in ((0, 2, 0), (3, 3, 10), (5, 1, 10), (20, 5, 20)):
            for _ in range(cnt):
                B.split(BG1, a + off, BG2, b, d=dd, k=int(rng.randint(90, 110)))

    # ---- depth 0 at p1's breakpoint: the split reads have MAPQ 0 and the spanning reads end before it
    if want("zero_depth"):
        a, b = slot(Q1), slot(BG2)
        B.junction("zero_depth", Q1, a, BG2, b, 2)
        for _ in range(3):
            B.split(Q1, a, BG2, b, mapq=0)

    # ---- the fatal record where it is never read: outside every region, and in a cluster dropped as close
    if want("fatal_outside"):
        B.fatal(BG1, slot(BG1))
    if want("close"):
        a = slot(BG1)
        slot(BG1)
        B.junction("close", BG1, a, BG1, a + 1500, 12)
        B.fatal(BG1, a - 100)


def _guards(B):
    """the isolated-pair mask drops the first and the last pair of every bucket in p1 order and again in p2 order
    (src/BreakID.cc:1830-1870), and -fast leaves the last clusters of a bucket open: groups of four spanning pairs
    below and above every junction of each bucket take those losses"""
    for A, Bt in sorted({(j["A"], j["B"]) for j in B.meta.values()}):
        B.span(A, 4000, Bt, 3000 if A != Bt else 7000, 4)
        for off in (9000, 4000):
            B.span(A, LENS[A] - off, Bt, LENS[Bt] - off + 1000 if A != Bt else LENS[A] - off + 3000, 4)


def build_refine_batch(seed=SEED, rungs=None, fatal_at=None, fatal_side=2, pairing=False):
    """the batch as synth.SynthData, the library-only parts (per-record name-hash tweaks and OC texts, for
    pairing_batch) and the junction table.  rungs: the rung names to plant (None: all).  fatal_at: also plant the fatal
    record in the side-`fatal_side` region of that rung (a region that is read).  pairing: plant the pairing rungs
    instead"""
    from breakid_b200 import synth
    B = _Builder(seed)
    for t in (BG1, BG2):
        B.background(t)
    if pairing:
        _plant_pairing(B)
    else:
        _plant(B, rungs)
    _guards(B)
    if fatal_at is not None:
        j = B.meta[fatal_at]
        if fatal_side == 1:
            B.fatal(j["A"], j["a"] - 60)
        else:
            B.fatal(j["B"], j["b"] + 60)
    recs = B.recs
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
    lib = {"tweaks": [(i, r[10]) for i, r in enumerate(recs) if r[10] is not None],
           "oc": [recs[i][9][2] if len(recs[i][9]) > 2 else b"" for i in sa_rec]}
    return d, lib, B.meta


# ------------------------------------------------------------------------------------------------------------ pairing
def _plant_pairing(B):
    """per field and orientation: 2 split reads at key (a, b) and 3 decoys near (a + 60, b + 60) that pair only if that
    one field is ignored.  The orientation is the kind of the side-1 row: the primary record (its own chromosome is p1's)
    or the 0x100 record (its primary chromosome is the SA's, not p1's).  The start and end fields cannot differ alone:
    on both kinds of row, end = start + M - 1 of the cigar whose text is compared, so a row pair that differs in start
    or end differs in the other, or in the cigar text, too"""
    slot = _Slots({})
    other = {"pchr": Q1, "schr": Q2}
    for field in PAIR_FIELDS:
        for flip in (False, True):
            r = "%s_%s" % (field, "flip" if flip else "plain")
            if field == "secondary":
                _secondary_rung(B, r, slot, flip)
                continue
            a, b = slot(BG1), slot(BG2)
            B.junction(r, BG1, a, BG2, b, 10)
            B.split(BG1, a, BG2, b, flip=flip)
            B.split(BG1, a, BG2, b, flip=flip)
            x, y = a + 60, b + 60
            for _ in range(3):
                if field in ("pbp", "sbp"):
                    _bp_decoy(B, field, x, y, flip)
                    continue
                k = int(B.rng.randint(80, 120))
                left, right = "%dM%dS" % (k, L - k), "%dS%dM" % (k, L - k)
                kw = {}
                # the record whose SA text carries the primary part's fields (p*) is the 0x100 one
                prim_side_b = flip                 # flip: the primary record is the one on B
                if field == "name_lo_hi32":
                    kw["sec_tweak" if not flip else "prim_tweak"] = "lo_hi32"
                elif field == "name_hi":
                    kw["sec_tweak" if not flip else "prim_tweak"] = "hi"
                elif field in ("pcig", "pchr"):    # the SA text of the 0x100 record names the primary part
                    txt = _sa(other["pchr"] if field == "pchr" else (BG2 if prim_side_b else BG1),
                              (y if prim_side_b else x - k + 1), ("0" if field == "pcig" else "") + (right if prim_side_b else left))
                    kw["prim_sa" if prim_side_b else "sec_sa"] = txt
                elif field in ("scig", "schr"):    # the SA text of the primary names the secondary part
                    txt = _sa(other["schr"] if field == "schr" else (BG1 if prim_side_b else BG2),
                              (x - k + 1 if prim_side_b else y), ("0" if field == "scig" else "") + (left if prim_side_b else right))
                    kw["sec_sa" if prim_side_b else "prim_sa"] = txt
                B.split(BG1, x, BG2, y, k=k, flip=flip, **kw)


def _bp_decoy(B, field, x, y, flip):
    """a primary record P and its 0x100 record S whose rows differ in primary_bp (pbp) or secondary_bp (sbp) alone.
    With an OC tag, a row's own end comes from the OC cigar but its own breakpoint, when that cigar ends in a clip, is the
    end of the BAM cigar (src/BreakID.cc:933-1016): the OC cigar is the one the partner's SA text names, the BAM cigar
    reaches one base further.  plain: P on BG1 (side 1), S on BG2; flip: P on BG2, S on BG1 (side 1)"""
    cp, xp, cs, ys = (BG1, x, BG2, y) if not flip else (BG2, y + 100, BG1, x)
    n = B.name()
    fp = PAIRED | PROPER | MREVERSE | READ1
    if field == "pbp":                     # P's own part is the left one: OC kM(L-k)S, BAM (k+1)M(L-k-1)S
        k = int(B.rng.randint(80, 120))
        p = xp - k
        oc, right = "%dM%dS" % (k, L - k), "%dS%dM" % (k, L - k)
        B.add(fp, 60, cp, p, cp, p + 200, 200 + L, p + k + 1, n, ("%dM%dS" % (k + 1, L - k - 1), _sa(cs, ys, right), oc.encode()))
        B.add(fp | SECONDARY, 60, cs, ys - 1, cp, p + 200, 0, ys - 1 + L - k, n, (right, _sa(cp, p + 1, oc)))
    else:                                  # S's own part ends in the clip: OC (L-k)MkS, BAM (L-k+1)M(k-1)S
        k = int(B.rng.randint(72, 79))
        p = xp - 1
        own, oc = "%dS%dM" % (k, L - k), "%dM%dS" % (L - k, k)
        B.add(fp, 60, cp, p, cp, p + 200, 200 + L, p + L - k, n, (own, _sa(cs, ys, oc)))
        B.add(fp | SECONDARY, 60, cs, ys - 1, cp, p + 200, 0, ys - 1 + L - k + 1, n,
              ("%dM%dS" % (L - k + 1, k - 1), _sa(cp, p + 1, own), oc.encode()))


def _secondary_rung(B, r, slot, flip):
    """a junction inside BG1 whose two regions lie 6 kb apart, 2 split reads, and 3 decoy records that are evidence
    rows in both regions: OC kM(L-k)S over a BAM cigar with a 5.6 kb N.  Each decoy's row meets itself on side 2 with
    every field equal and the same secondary flag, so it pairs only if secondary != secondary is dropped
    (src/BreakID.cc:627-637).  plain: the decoys are primaries (primary chromosome = p1's); flip: 0x100 records whose SA
    text names another chromosome"""
    a = slot(BG1)
    b = a + 6000
    slot(BG1)
    B.junction(r, BG1, a, BG1, b, 10)
    B.split(BG1, a, BG1, b)
    B.split(BG1, a, BG1, b)
    for _ in range(3):
        k = int(B.rng.randint(80, 120))
        p, gap = a + 60 - k, 5600
        oc, right = "%dM%dS" % (k, L - k), "%dS%dM" % (k, L - k)
        sa = _sa(BG1, b + 60, right) if not flip else _sa(Q2, 5000, right)
        B.add(PAIRED | PROPER | MREVERSE | READ1 | (SECONDARY if flip else 0), 60, BG1, p, BG1, p + 200, 0 if flip else 200 + L,
              p + k + gap, B.name(), ("%dM%dN%dS" % (k, gap, L - k), sa, oc.encode()))


def pairing_batch(seed=SEED + 1):
    """the pairing rungs as a HostBatch, with the name hashes of the decoy records changed: high word of name_lo
    (the low 32 bits, which the device's name index sorts on, stay equal) or name_hi, and the OC tags of the
    breakpoint and secondary decoys"""
    from breakid_b200 import api, synth
    d, lib, meta = build_refine_batch(seed, pairing=True)
    hb = api.HostBatch.from_synth(d)
    nh = synth.name_hash_ids(d.cols["name_id"]).cpu().numpy().view(np.uint64).reshape(-1, 2).copy()
    for i, tw in lib["tweaks"]:
        if tw == "lo_hi32":
            nh[i, 0] ^= np.uint64(1 << 40)
        elif tw == "hi":
            nh[i, 1] ^= np.uint64(1)
    cols = {k: d.cols[k].cpu().numpy() for k in ("mapq", "tid", "pos", "mtid", "mpos", "isize", "endpos")}
    cols["flag"] = d.cols["flag"].cpu().numpy().view(np.uint16)
    side = {k: hb.side[k] for k in ("sa_rec", "cig_off", "cig_ops", "sa_off", "sa_txt")}
    side["oc_off"] = np.concatenate([[0], np.cumsum([len(o) for o in lib["oc"]])]).astype(np.uint32)
    side["oc_txt"] = np.frombuffer(b"".join(lib["oc"]), np.uint8)
    return api.HostBatch(cols, nh.reshape(-1), side, hb.target_len, hb.target_names), meta, lib


# ------------------------------------------------------------------------------------------------------------ models
FIELDS = ("name_lo", "name_hi", "primary_chr", "secondary_chr", "primary_start", "secondary_start", "primary_end",
          "secondary_end", "primary_cigar_h", "secondary_cigar_h", "primary_bp", "secondary_bp")


def _cl(j):
    """the cluster record fields _entries reads, from the junction table"""
    return {"p1_tid": j["A"], "p2_tid": j["B"], "p1_mean_pos": j["p1_mean"], "p2_mean_pos": j["p2_mean"]}


def _entries_ignoring(hb, c, w, ignore):
    """_entries with one field of the match left out ("secondary": rows of equal flags pair too; "name_lo_hi32": only
    the low 32 bits of name_lo are compared)"""
    import oracle_py as O
    e1 = O.find_sa_reads(hb, int(c["p1_tid"]), *_region(c["p1_mean_pos"], w))
    e2 = O.find_sa_reads(hb, int(c["p2_tid"]), *_region(c["p2_mean_pos"], w))
    fmap = {"pcig": "primary_cigar_h", "scig": "secondary_cigar_h", "pchr": "primary_chr", "schr": "secondary_chr",
            "name_hi": "name_hi", "pbp": "primary_bp", "sbp": "secondary_bp"}

    def key(r):
        out = []
        for f in FIELDS:
            v = int(r[f])
            if f == fmap.get(ignore):
                v = 0
            if f == "name_lo" and ignore == "name_lo_hi32":
                v &= 0xFFFFFFFF
            out.append(v)
        return tuple(out)
    n = 0
    for a in e1:
        for b in e2:
            if key(a) == key(b) and (ignore == "secondary" or int(a["secondary"]) != int(b["secondary"])):
                n += 1
    return n


def _vote(ent, err=2, order="string", last=False):
    """the vote with the reference's uint32 windows, the winner chosen over the keys in string or numeric order"""
    u = ent.astype(np.uint32)
    keys = sorted({(int(x), int(y)) for x, y in ent}, key=(lambda k: "%d,%d" % k) if order == "string" else None)
    best, call = 0, None
    for kx, ky in keys:
        kx32, ky32 = np.uint32(kx), np.uint32(ky)
        lo_x, hi_x = kx32 - np.uint32(err), kx32 + np.uint32(err)
        lo_y, hi_y = ky32 - np.uint32(err), ky32 + np.uint32(err)
        n = int(((u[:, 0] <= hi_x) & (u[:, 0] >= lo_x) & (u[:, 1] <= hi_y) & (u[:, 1] >= lo_y)).sum())
        if n > best or (last and n == best and n > 0):
            best, call = n, (kx, ky)
    return call, best


def _coverage(hb, t, mean, w):
    """total coverage of the region of `mean`: every record the index iterator returns (src/BreakID.cc:894)"""
    beg, end = _region(mean, w)
    beg = max(int(np.int32(np.uint32(beg))), 0)
    c = hb.cols
    return int(((c["tid"] == t) & (c["pos"] < int(np.int32(np.uint32(end)))) & (c["endpos"] > beg)).sum())


def nibs_for(d):
    from breakid_b200 import synth
    return [(synth.random_nib_bytes(l, d.cfg.seed * 1000 + t).numpy(), l) for t, l in enumerate(d.cfg.chrom_lens)]


@pytest.fixture(scope="module")
def refine_data():
    import oracle_py as O
    from breakid_b200 import api
    d, _, meta = build_refine_batch()
    hb = api.HostBatch.from_synth(d)
    nibs = nibs_for(d)
    runs = {mode: O.run(hb, nibs, mode=mode) for mode in (0, 1)}
    return d, hb, nibs, meta, runs


def _find(cl, j):
    """the call of junction j (chromosomes, and breakpoints within 40 bp), or None"""
    hit = [c for c in cl if (int(c["p1_tid"]), int(c["p2_tid"])) == (j["A"], j["B"]) and
           abs(int(c["p1_exact_pos"]) - j["a"]) <= 40 and abs(int(c["p2_exact_pos"]) - j["b"]) <= 40]
    assert len(hit) <= 1
    return hit[0] if hit else None


def _model_m(hb, meta, w, skip=("close",)):
    return {r: len(_entries(hb, _cl(j), w)) for r, j in meta.items() if r not in skip}


# ------------------------------------------------------------------------------------------------ CPU: rungs are reached
def test_batch_shape(refine_data):
    d, hb, nibs, meta, runs = refine_data
    tid, pos = hb.cols["tid"].astype(np.int64), hb.cols["pos"].astype(np.int64)
    assert np.array_equal(np.lexsort((pos, tid.astype(np.uint32))), np.arange(hb.n))
    assert 100000 < hb.n < 200000
    assert set(hb.narrow()) == {"span16", "isize16", "tid_run_start", "tid_run_tid"}
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        # one cluster per junction: its means are those of the junction's spanning reads
        assert len(cl) >= 20


def test_vote_form_sizes(refine_data):
    """each vote-form rung has its designed number of entries, and the n_split_read the oracle reports is the vote"""
    d, hb, nibs, meta, runs = refine_data
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        w = int(dist)
        mm = _model_m(hb, meta, w)
        for r, size in VOTE_SIZES.items():
            assert mm[r] == size, (r, mm[r])
            c = _find(cl, meta[r])
            assert (c is None) == (size == 1), r
            if c is not None:
                ent = _entries(hb, c, w)
                call, best = _vote(ent)
                assert (int(c["p1_exact_pos"]), int(c["p2_exact_pos"]), int(c["n_split_read"])) == call + (best,)
        assert mm["product"] == 3 * 2 + 2 and int(_find(cl, meta["product"])["n_split_read"]) >= 6
        assert mm["m8192"] <= 8192 < mm["m8193"] and mm["m256"] <= 256 < mm["m257"]


def test_tie_rungs_order_matters(refine_data):
    """every tie rung: all keys get the same vote; the numeric-order winner differs from the string-order one (the
    oracle's); on the same-digit rung the last maximum differs from the first"""
    d, hb, nibs, meta, runs = refine_data
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        w = int(dist)
        for r, small in (("tie_x", True), ("tie_y", True), ("tie_big", False), ("tie_first", True)):
            c = _find(cl, meta[r])
            ent = _entries(hb, c, w)
            assert (len(ent) <= 256) == small, (r, len(ent))
            got = (int(c["p1_exact_pos"]), int(c["p2_exact_pos"]))
            sv, nv = _vote(ent, order="string")
            num, _ = _vote(ent, order="numeric")
            last, _ = _vote(ent, order="string", last=True)
            assert sv == got and nv == len(ent) == int(c["n_split_read"])
            assert _wrap_free_vote(ent) == (sv, nv)            # no window wraps here
            assert len({tuple(e) for e in ent.tolist()}) == 2
            if r == "tie_first":
                assert num == sv and last != sv
            else:
                assert num != sv, r
        assert _find(cl, meta["tie_x"])["p1_exact_pos"] == 10000
        assert _find(cl, meta["tie_big"])["p1_exact_pos"] == 100000
        assert _find(cl, meta["tie_y"])["p2_exact_pos"] == 100000


def test_gate_rungs_at_threshold(refine_data):
    """coverage and evidence rows of each gate rung sit at the threshold, and only the rungs that pass are called"""
    import oracle_py as O
    d, hb, nibs, meta, runs = refine_data
    want = {"g1_cov4": (1, 4, 2, False), "g1_ev1": (1, 5, 1, False), "g1_ev2": (1, 7, 2, True),
            "g2_cov4": (2, 4, 2, False), "g2_cov5": (2, 5, 2, True), "g2_ev1": (2, 5, 1, False), "g2_ev2": (2, 7, 2, True)}
    for kind in EXTRA_KINDS:
        want["g1_cov5_" + kind] = (1, 5, 2, True)
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        w = int(dist)
        for r, (side, cov, nev, called) in want.items():
            j = meta[r]
            t, mean = (j["A"], j["p1_mean"]) if side == 1 else (j["B"], j["p2_mean"])
            assert _coverage(hb, t, mean, w) == cov, (r, _coverage(hb, t, mean, w))
            beg, end = _region(mean, w)
            ev = O.find_sa_reads(hb, t, beg, end, mismatch=10)
            assert len(ev) == (nev if cov >= 5 and nev >= 2 else 0), r
            assert (_find(cl, j) is not None) == called, r
        # the long-span record reaches its region only from maxspan bases to the left
        j = meta["g1_cov5_longspan"]
        beg = _region(j["p1_mean"], w)[0]
        ls = (hb.cols["tid"] == Q1) & (hb.cols["pos"] < beg) & (hb.cols["endpos"] > beg)
        assert ls.sum() == 1 and int(hb.cols["endpos"][ls][0] - hb.cols["pos"][ls][0]) == 3600


def test_vote_rungs(refine_data):
    """best votes of exactly 1 (no call) and 2 (a call)"""
    d, hb, nibs, meta, runs = refine_data
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        w = int(dist)
        ent = _entries(hb, _cl(meta["vote1"]), w)
        assert len(ent) == 2 and _vote(ent)[1] == 1 and _find(cl, meta["vote1"]) is None
        c = _find(cl, meta["vote2"])
        assert int(c["n_split_read"]) == 2 and len(_entries(hb, c, w)) == 3
        assert _find(cl, meta["m1"]) is None and int(_find(cl, meta["m2"])["n_split_read"]) == 2


def test_zero_depth_call_has_inf_allele_frequency(refine_data):
    import oracle_py as O
    d, hb, nibs, meta, runs = refine_data
    for mode in (0, 1):
        c = _find(runs[mode][3], meta["zero_depth"])
        assert float(c["p1_bp_depth"]) == 0 and np.isinf(c["p1_alle_freq"]) and float(c["p2_bp_depth"]) > 0
        assert O.single_base_depth(hb, Q1, int(c["p1_exact_pos"])) == 0


def test_fatal_rung_reaches_the_oracle_only_when_read(refine_data):
    """the clip-free record makes the oracle fail inside a region that is read; outside every region, behind a side 1
    that fails its gate, and in a cluster dropped as close, it changes nothing"""
    import oracle_py as O
    from breakid_b200 import api
    d, hb, nibs, meta, runs = refine_data
    for mode in (0, 1):
        m, s, dist, cl = runs[mode]
        assert _find(cl, meta["close"]) is None and _find(cl, meta["vote2"]) is not None
        j = meta["close"]
        assert abs(j["p1_mean"] - j["p2_mean"]) <= 2 * dist                 # the close rule (src/BreakID.cc:348)
    assert fatal_count(hb) == 3
    for side in (1, 2):
        fd, _, _ = build_refine_batch(fatal_at="vote2", fatal_side=side)
        fhb = api.HostBatch.from_synth(fd)
        assert fatal_count(fhb) == 4
        with pytest.raises(RuntimeError, match="error cigar"):
            O.run(fhb, nibs, mode=0)


def fatal_count(hb):
    s = hb.side
    n = 0
    for k in range(hb.n_sa):
        if bytes(s["sa_txt"][s["sa_off"][k]:s["sa_off"][k + 1]]).endswith(b"75M75M,60,0;"):
            n += 1
    return n


def test_pairing_rungs_change_when_field_ignored():
    """each pairing rung: 2 entries; ignoring its one differing field would add the 3 decoys"""
    import oracle_py as O
    hb, meta, lib = pairing_batch()
    assert len(lib["tweaks"]) == 2 * 2 * 3 and sum(len(o) > 0 for o in lib["oc"]) == 3 * 2 * 3
    assert set(r.rsplit("_", 1)[0] for r in meta) == set(PAIR_FIELDS)
    m, s, dist, cl = O.run(hb, mode=0)
    w = int(dist)
    for r, j in meta.items():
        field = r.rsplit("_", 1)[0]
        ent = _entries(hb, _cl(j), w)
        assert len(ent) == 2, (r, len(ent))
        c = _find(cl, j)
        assert c is not None and int(c["n_split_read"]) == 2 and int(c["p1_exact_pos"]) == j["a"], r
        assert _entries_ignoring(hb, _cl(j), w, field) == 5, r


def test_refine_consts_defaults_change_nothing(refine_data):
    import oracle_py as O
    d, hb, nibs, meta, runs = refine_data
    got = O.run(hb, nibs, mode=1, bp_err=2, mismatch=10)
    assert got[:3] == runs[1][:3] and got[3].tobytes() == runs[1][3].tobytes()
    with O.refine_consts(2, 10):
        again = O.run(hb, nibs, mode=1)
    assert again[3].tobytes() == runs[1][3].tobytes()


def test_refine_consts_nest_and_restore(refine_data):
    """a block's constants reach run() and find_sa_reads() called without them, an inner block overrides one of them,
    and each block restores what was in force before it"""
    import oracle_py as O
    d, hb, nibs, meta, runs = refine_data
    wide = O.run(hb, nibs, mode=1, bp_err=40)[3]
    assert wide.tobytes() != runs[1][3].tobytes()
    j = meta["mismatch"]
    w = int(runs[1][2])
    n_ev = lambda: len(O.find_sa_reads(hb, j["A"], *_region(j["p1_mean"], w)))
    with O.refine_consts(40, 10):
        assert O.run(hb, nibs, mode=1)[3].tobytes() == wide.tobytes()
        full = n_ev()
        with O.refine_consts(mismatch=0):
            assert O._refine == [40, 0]
            assert n_ev() == full - 4 == 2                   # without the 3 + 1 rows whose cigars are off by 3 and 5
        assert O._refine == [40, 10] and O.run(hb, nibs, mode=1)[3].tobytes() == wide.tobytes()
    assert O._refine == [2, 10] and O.run(hb, nibs, mode=1)[3].tobytes() == runs[1][3].tobytes()


def test_refine_consts_reach_the_oracle(refine_data):
    """the mismatch rung and the big rungs change with the two constants, and the defaults are restored afterwards"""
    import oracle_py as O
    d, hb, nibs, meta, runs = refine_data
    base = runs[1][3]
    calls = {}
    for kw in ({"mismatch": 0}, {"mismatch": 3}, {"mismatch": 25}, {"bp_err": 0}, {"bp_err": 40}):
        cl = O.run(hb, nibs, mode=1, **kw)[3]
        calls[tuple(kw.items())] = cl
        assert cl.tobytes() != base.tobytes(), kw
    mm = lambda cl: (int(_find(cl, meta["mismatch"])["p1_exact_pos"]) - meta["mismatch"]["a"], int(_find(cl, meta["mismatch"])["n_split_read"]))
    assert mm(base) == (10, 4)
    assert mm(calls[(("mismatch", 0),)]) == (0, 2) and mm(calls[(("mismatch", 25),)]) == (20, 5)
    assert mm(calls[(("mismatch", 3),)]) == (10, 3)
    assert O.run(hb, nibs, mode=1)[3].tobytes() == base.tobytes()
    # at 40 every key of a big rung sees every entry of it
    c = _find(calls[(("bp_err", 40),)], meta["m8193"])
    assert int(c["n_split_read"]) == 8193


def test_small_batch_stays_below_vote_big():
    """the small batch's entry total is at most 256, so k8_vote_big is never launched on it"""
    import oracle_py as O
    from breakid_b200 import api
    d, _, meta = build_refine_batch(rungs=SMALL_RUNGS)
    hb = api.HostBatch.from_synth(d)
    w = int(O.run(hb, mode=0)[2])
    mm = _model_m(hb, meta, w)
    assert 100 < sum(mm.values()) <= 256 and mm["tie_y"] == 100


# ------------------------------------------------------------------------------------------------ GPU: device == oracle
def _device_run(hb, nibs, mode, narrow=True, **params):
    from breakid_b200 import api
    c = api.Context(hb.target_len, hb.target_names, device=0, fast=mode)
    if params:
        c.set_params(**params)
    c.push(hb, narrow=narrow)
    for t, (p, l) in enumerate(nibs or []):
        c.set_nib(t, p, l)
    res = c.run()
    got = c.fetch_clusters()
    tm = c.timings()
    c.close()
    return res, got, tm


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
def test_library_equals_oracle(refine_data, mode, narrow):
    """byte for byte, and the device's entry count is the model's sum over the clusters (which picks the vote forms)"""
    d, hb, nibs, meta, runs = refine_data
    res, got, tm = _device_run(hb, nibs, mode, narrow=narrow)
    _assert_equal(res, got, runs[mode])
    w = int(runs[mode][2])
    assert tm["n_evidence"] == sum(_model_m(hb, meta, w).values())


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_small_batch_without_vote_big(mode):
    """at most 256 entries in the whole step: k8_vote_big is never launched"""
    import oracle_py as O
    from breakid_b200 import api
    d, _, meta = build_refine_batch(rungs=SMALL_RUNGS)
    hb = api.HostBatch.from_synth(d)
    nibs = nibs_for(d)
    exp = O.run(hb, nibs, mode=mode)
    res, got, tm = _device_run(hb, nibs, mode)
    _assert_equal(res, got, exp)
    assert 0 < tm["n_evidence"] <= 256 and len(got) >= 5


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_pairing_variant_equals_oracle(mode):
    import oracle_py as O
    hb, meta, _ = pairing_batch()
    exp = O.run(hb, mode=mode)
    res, got, tm = _device_run(hb, None, mode)
    _assert_equal(res, got, exp)
    assert len(got) == len(meta)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [{"bp_pos_error": 0}, {"bp_pos_error": 1}, {"bp_pos_error": 5}, {"bp_pos_error": 40},
                                {"mismatch_num": 0}, {"mismatch_num": 3}, {"mismatch_num": 25}])
def test_refine_params_equal_oracle(refine_data, kw):
    import oracle_py as O
    d, hb, nibs, meta, runs = refine_data
    exp = O.run(hb, nibs, mode=1, bp_err=kw.get("bp_pos_error", 2), mismatch=kw.get("mismatch_num", 10))
    res, got, tm = _device_run(hb, nibs, 1, **kw)
    _assert_equal(res, got, exp)


@pytest.mark.gpu
@pytest.mark.parametrize("side", [1, 2])
@pytest.mark.parametrize("mode", [0, 1])
def test_fatal_cigar_library(refine_data, mode, side):
    """BKID_ERR_CIGAR through bkid_run when the record is read, on side 1 or side 2; the three silent copies of the
    main batch equal the oracle (test_library_equals_oracle)"""
    from breakid_b200 import api
    d, hb, nibs, meta, runs = refine_data
    fd, _, _ = build_refine_batch(fatal_at="vote2", fatal_side=side)
    fhb = api.HostBatch.from_synth(fd)
    c = api.Context(fhb.target_len, fhb.target_names, device=0, fast=mode)
    c.push(fhb)
    with pytest.raises(api.BkidError, match="error %d: error cigar" % BKID_ERR_CIGAR):
        c.run()
    c.close()




def _ranks(hb, cuts, nibs, mode):
    from breakid_b200 import api
    from test_multi_gloo import _slice
    ctxs = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        c = api.Context(hb.target_len, hb.target_names, device=0, fast=mode)
        c.push(_slice(hb, a, b))
        for t, (p, l) in enumerate(nibs):
            c.set_nib(t, p, l)
        ctxs.append(c)
    return ctxs


def _gate_cuts(hb, meta, world):
    """cuts inside the side-1 region of g1_cov5_mapq0 (between its records) and, for 3 ranks, inside the side-2 region
    of g2_cov5: the gate then sees coverage 5 only as the sum of partial counts"""
    tid, pos = hb.cols["tid"], hb.cols["pos"]
    first = lambda m: int(np.nonzero(m)[0][0])
    j1, j2 = meta["g1_cov5_mapq0"], meta["g2_cov5"]
    c1 = first((tid == Q1) & (pos >= j1["a"] - 150))
    c2 = first((tid == Q2) & (pos >= j2["b"] - 1))
    return [0, c1, hb.n] if world == 2 else [0, c1, c2, hb.n]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("mode", [0, 1])
def test_sharded_gate_cuts_equal_oracle(refine_data, world, mode):
    from breakid_b200 import api
    d, hb, nibs, meta, runs = refine_data
    cuts = _gate_cuts(hb, meta, world)
    assert all(a < b for a, b in zip(cuts[:-1], cuts[1:]))
    ctxs = _ranks(hb, cuts, nibs, mode)
    res = api.dist_run_local(ctxs, mode)
    m, s, dist, exp = runs[mode]
    for r, c in enumerate(ctxs):
        assert res[r][:3] == (m, s, dist), r
        assert c.fetch_clusters().tobytes() == exp.tobytes(), r
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("side", [1, 2])
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_fatal_cigar(refine_data, world, side):
    """every rank returns BKID_ERR_CIGAR, and none waits for the others"""
    from breakid_b200 import api
    d, hb, nibs, meta, runs = refine_data
    fd, _, fmeta = build_refine_batch(fatal_at="vote2", fatal_side=side)
    fhb = api.HostBatch.from_synth(fd)
    ctxs = _ranks(fhb, _gate_cuts(fhb, fmeta, world), nibs, 0)
    with pytest.raises(api.BkidError, match="error %d" % BKID_ERR_CIGAR):
        api.dist_run_local(ctxs, 0)
    L_ = api.cuda_lib()
    for c in ctxs:
        assert b"error cigar" in (L_.bkid_last_error(c.ctx) or b"")
        c.close()


def _driver(tmp_path, paths, tag, flags, env=None):
    drv = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "breakid_b200", "host", "BreakID")
    return subprocess.run([drv, "-i", paths["bam"], "-o", str(tmp_path / tag), "-n", paths["nib"], "-r", paths["refgene"]] + flags,
                          timeout=600, capture_output=True, text=True, env=env)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["ahc", "fast"])
def test_driver_on_refine_bam(tmp_path, refine_data, mode):
    """the batch as a BAM: BreakID -all with device and host decode writes the oracle's calls (inf allele frequency
    included), and the reference binary's files where it is built"""
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio
    d, hb, nibs, meta, runs = refine_data
    paths = bamio.write_dataset(str(tmp_path), d)
    R.index(paths["bam"])
    flags = ["-all"] + (["-fast"] if mode == "fast" else [])
    for tag, env in (("gpu", None), ("gpu_host", dict(os.environ, BKID_HOST_DECODE="1"))):
        g = _driver(tmp_path, paths, tag, flags, env)
        assert g.returncode == 0, (tag, g.stderr[-500:])
        R.match_oracle(str(tmp_path / tag), d, mode=int(mode == "fast"))
    txt = open(str(tmp_path / "gpu") + "_fusion_all.txt").read()
    assert "\tinf\t" in txt
    assert txt == open(str(tmp_path / "gpu_host") + "_fusion_all.txt").read()
    if O.have_ref():
        O.ref_install_refgene(paths["refgene"])
        r = O.ref_run_binary(paths["bam"], str(tmp_path / "ref"), paths["nib"], fast=(mode == "fast"))
        assert r.returncode == 0, r.stderr[-500:]
        for suffix in ("_fusion.txt", "_fusion_all.txt"):
            assert open(str(tmp_path / "ref") + suffix).read() == open(str(tmp_path / "gpu") + suffix).read(), suffix


@pytest.mark.gpu
def test_driver_fatal_cigar(tmp_path):
    """the reference exits with status 255 (exit(-1)) on the error cigar and writes no call file: so does the driver.
    The message is the driver's own, on stderr (INTEGRATION.md): only the status and the missing files are compared"""
    import oracle_py as O
    import reference_calls as R
    from breakid_b200 import bamio
    fd, _, _ = build_refine_batch(fatal_at="vote2")
    paths = bamio.write_dataset(str(tmp_path), fd)
    R.index(paths["bam"])
    g = _driver(tmp_path, paths, "gpu", ["-all"])
    assert g.returncode == 255 and "error cigar" in g.stderr, (g.returncode, g.stderr[-500:])
    assert not os.path.exists(str(tmp_path / "gpu") + "_fusion_all.txt")
    assert not os.path.exists(str(tmp_path / "gpu") + "_fusion.txt")
    if O.have_ref():
        O.ref_install_refgene(paths["refgene"])
        r = O.ref_run_binary(paths["bam"], str(tmp_path / "ref"), paths["nib"])
        assert r.returncode == g.returncode
        assert not os.path.exists(str(tmp_path / "ref") + "_fusion_all.txt")
        assert not os.path.exists(str(tmp_path / "ref") + "_fusion.txt")
