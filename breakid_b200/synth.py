"""Deterministic synthetic workloads for the BreakID hot path (SURVEY.md §8d).

hg19 .nib files and real BAMs are not available offline, so every config of BASELINE.json is a
generated genome + a simulated coordinate-sorted, duplicate-marked alignment set with planted
translocations / inversions / tandem duplications / deletions, produced directly as the
struct-of-arrays record batch the C-ABI consumes (``bkid_batch``, include/breakid_b200.h) and,
for the small configs, also as a real BAM (``bamio.write_bam``) so the reference CPU binary can
be run on byte-identical input.

Everything is written with torch tensor ops so the same code generates config 1 on the CPU in
this container and the 6.2e8-record whole-genome configs on the B200 itself.

Planting recipe (the one the reference actually calls, SURVEY.md §8d): junction "left part ends
at A:a on +, right part starts at B:b"; spanning pair = read1 flag 97 at a-L-d, read2 flag 145 at
b+d'; split read = primary ``kM(L-k)S`` at a-k+1 with ``SA:Z:B,b,+,kS(L-k)M,60,0;`` plus a
0x100 record at B:b with the complementary cigar.  INV: both mates forward (65/129), split tail
on the minus strand.
"""
from __future__ import annotations

import dataclasses
import math
from typing import Dict, List, Optional

import numpy as np
import torch

HG19_LENS = [249250621, 243199373, 198022430, 191154276, 180915260, 171115067, 159138663,
             146364022, 141213431, 135534747, 135006516, 133851895, 115169878, 107349540,
             102531392, 90354753, 81195210, 78077248, 59128983, 63025520, 48129895, 51304566,
             155270560, 59373566]


def chrom_name(tid: int) -> str:
    """tid -> name convention the reference silently requires (src/util_bam.cc:128-142)."""
    if tid == 23:
        return "chrY"
    if tid == 22:
        return "chrX"
    return "chr%d" % (tid + 1)


# BAM flag bits
PAIRED, PROPER, UNMAP, MUNMAP, REVERSE, MREVERSE, READ1, READ2, SECONDARY, QCFAIL, DUP, SUPP = (
    0x1, 0x2, 0x4, 0x8, 0x10, 0x20, 0x40, 0x80, 0x100, 0x200, 0x400, 0x800)

OP_M, OP_I, OP_D, OP_N, OP_S, OP_H, OP_P, OP_EQ, OP_X = range(9)


@dataclasses.dataclass
class SynthConfig:
    chrom_lens: List[int]
    coverage: float = 30.0
    read_len: int = 150
    insert_mean: float = 350.0
    insert_sd: float = 30.0
    n_tra: int = 3
    n_inv: int = 3
    n_dup: int = 2
    n_del: int = 2
    span_per_sv: int = 15
    split_per_sv: int = 8
    chimeric_frac: float = 0.01      # random chimeric (noise) pairs, fraction of all pairs
    near_frac: float = 0.002         # improper pairs closer than the scan distance
    dup_frac: float = 0.05
    lowq_frac: float = 0.05          # fraction of improper records with MAPQ < 20
    sv_jitter: int = 0               # +-jitter on split-read breakpoints (exercises the +-2 vote)
    split_k_min: Optional[int] = None  # bases on the A side of a split read: U[split_k_min, split_k_max)
    split_k_max: Optional[int] = None  # (defaults L/2+1 .. L-20; config 5 uses 20 .. 131 = clip lengths U(20,130))
    min_sv_sep: int = 6000
    seed: int = 1
    n_pairs: Optional[int] = None    # override coverage-derived pair count


@dataclasses.dataclass
class SynthData:
    """Coordinate-sorted record batch (file order) + SA side table + truth."""
    cfg: SynthConfig
    cols: Dict[str, torch.Tensor]          # flag i16(u16 bits), mapq u8, tid,pos,mtid,mpos,isize,endpos i32, name_id i64
    sa_rec: torch.Tensor                   # i64 record index (file order) of every SA-bearing record
    cig_off: torch.Tensor                  # i64 [n_sa+1] into cig_ops (BAM u32 ops of that record)
    cig_ops: torch.Tensor                  # i64 (value fits u32)
    sa_off: torch.Tensor                   # i64 [n_sa+1] into sa_txt
    sa_txt: torch.Tensor                   # u8
    truth: Dict[str, torch.Tensor]         # planted junctions: type, A, a, B, b

    @property
    def n(self) -> int:
        return int(self.cols["flag"].numel())


def _segments(off: torch.Tensor, data: torch.Tensor, order: torch.Tensor):
    """variable-length segments data[off[k]:off[k+1]] re-laid out in the row order `order` -> (new offsets, new data)"""
    ln = (off[1:] - off[:-1])[order]
    new_off = torch.zeros(order.numel() + 1, dtype=off.dtype, device=off.device)
    new_off[1:] = torch.cumsum(ln, 0)
    total = int(new_off[-1])
    if total == 0:
        return new_off, data[:0].clone()
    seg = torch.repeat_interleave(torch.arange(order.numel(), device=off.device), ln)
    src = off[:-1][order][seg] + (torch.arange(total, device=off.device) - new_off[:-1][seg])
    return new_off, data[src]


def permute(d: SynthData, order) -> SynthData:
    """the same records in a new file order: new record i is old record order[i] (a permutation of range(n)).  The SA side
    table is re-laid out in ascending new record index, as a decoder of the permuted file would list it."""
    order = torch.as_tensor(order, dtype=torch.int64, device=d.cols["flag"].device)
    assert order.numel() == d.n
    new_of = torch.empty_like(order)
    new_of[order] = torch.arange(d.n, dtype=torch.int64, device=order.device)
    cols = {k: v[order] for k, v in d.cols.items()}
    sa_new = new_of[d.sa_rec]
    rows = torch.argsort(sa_new, stable=True)
    cig_off, cig_ops = _segments(d.cig_off, d.cig_ops, rows)
    sa_off, sa_txt = _segments(d.sa_off, d.sa_txt, rows)
    return SynthData(cfg=d.cfg, cols=cols, sa_rec=sa_new[rows], cig_off=cig_off, cig_ops=cig_ops, sa_off=sa_off, sa_txt=sa_txt,
                     truth=d.truth)


def _digits(v: torch.Tensor):
    """decimal digit count of non-negative int64 tensor (>=1)."""
    n = torch.ones_like(v)
    p = 10
    for _ in range(18):
        n = n + (v >= p).to(v.dtype)
        p *= 10
    return n


def format_fields(parts, device) -> (torch.Tensor, torch.Tensor):
    """Vectorised text formatting.  ``parts`` is a list of either ('i', int64 tensor[n]) for a
    decimal integer, ('s', bytes) for a constant string, or ('t', u8 tensor[n, w], len tensor[n])
    for per-row strings.  Returns (offsets[n+1], flat u8 text)."""
    n = None
    for p in parts:
        if p[0] != 's':
            n = p[1].shape[0]
    lens = torch.zeros(n, dtype=torch.int64, device=device)
    plen = []
    for p in parts:
        if p[0] == 'i':
            l = _digits(p[1])
        elif p[0] == 's':
            l = torch.full((n,), len(p[1]), dtype=torch.int64, device=device)
        else:
            l = p[2].to(torch.int64)
        plen.append(l)
        lens += l
    off = torch.zeros(n + 1, dtype=torch.int64, device=device)
    off[1:] = torch.cumsum(lens, 0)
    out = torch.zeros(int(off[-1]), dtype=torch.uint8, device=device)
    cur = off[:-1].clone()
    for p, l in zip(parts, plen):
        if p[0] == 'i':
            v = p[1]
            maxd = int(l.max()) if n else 1
            for d in range(maxd):      # d-th digit from the left
                has = l > d
                e = (l - 1 - d).clamp(min=0)
                div = torch.pow(torch.tensor(10, dtype=torch.int64, device=device), e)
                dig = (v // div) % 10
                out[(cur + d)[has]] = (dig[has] + 48).to(torch.uint8)
        elif p[0] == 's':
            b = torch.tensor(list(p[1]), dtype=torch.uint8, device=device)
            for d in range(len(p[1])):
                out[cur + d] = b[d]
        else:
            w = p[1].shape[1]
            for d in range(w):
                has = l > d
                out[(cur + d)[has]] = p[1][:, d][has]
        cur = cur + l
    return off, out


def _chr_name_table(n_chr: int, device):
    names = [chrom_name(t).encode() for t in range(n_chr)]
    w = max(len(x) for x in names)
    tab = torch.zeros((n_chr, w), dtype=torch.uint8, device=device)
    ln = torch.zeros(n_chr, dtype=torch.int64, device=device)
    for t, x in enumerate(names):
        tab[t, :len(x)] = torch.tensor(list(x), dtype=torch.uint8)
        ln[t] = len(x)
    return tab, ln


def generate(cfg: SynthConfig, device="cpu") -> SynthData:
    g = torch.Generator(device=device)
    g.manual_seed(cfg.seed)
    dev = torch.device(device)
    L = cfg.read_len
    lens = torch.tensor(cfg.chrom_lens, dtype=torch.int64, device=dev)
    n_chr = len(cfg.chrom_lens)
    genome = int(lens.sum())
    n_pairs = cfg.n_pairs if cfg.n_pairs is not None else int(cfg.coverage * genome / (2 * L))
    cum = torch.zeros(n_chr + 1, dtype=torch.int64, device=dev)
    cum[1:] = torch.cumsum(lens, 0)

    def rand(n):
        return torch.rand(n, generator=g, device=dev, dtype=torch.float64)

    def randint(lo, hi, n):
        return torch.randint(lo, hi, (n,), generator=g, device=dev, dtype=torch.int64)

    margin = 2000

    def rand_loc(n):
        """uniform genome location -> (tid, 0-based pos) at least `margin` from chromosome ends."""
        gp = (rand(n) * genome).to(torch.int64).clamp(max=genome - 1)
        tid = torch.searchsorted(cum, gp, right=True) - 1
        pos = gp - cum[tid]
        pos = torch.minimum(torch.maximum(pos, torch.tensor(margin, device=dev)), lens[tid] - margin - 1)
        return tid, pos

    cols = {k: [] for k in ("flag", "mapq", "tid", "pos", "mtid", "mpos", "isize", "endpos", "name_id")}
    # side info for SA-bearing records, aligned with the records appended to cols
    sa_mark: List[torch.Tensor] = []      # per-record: index into the SA arrays or -1
    sa_cig0, sa_cig1 = [], []             # two BAM cigar ops per SA record
    sa_parts: List[dict] = []

    def emit(flag, mapq, tid, pos, mtid, mpos, isize, endpos, name_id, sa_idx=None):
        n = flag.numel()
        cols["flag"].append(flag.to(torch.int16))
        cols["mapq"].append(mapq.to(torch.uint8))
        cols["tid"].append(tid.to(torch.int32)); cols["pos"].append(pos.to(torch.int32))
        cols["mtid"].append(mtid.to(torch.int32)); cols["mpos"].append(mpos.to(torch.int32))
        cols["isize"].append(isize.to(torch.int32)); cols["endpos"].append(endpos.to(torch.int32))
        cols["name_id"].append(name_id)
        sa_mark.append(sa_idx if sa_idx is not None else torch.full((n,), -1, dtype=torch.int64, device=dev))

    next_name = 0

    # ---------------- A. proper pairs ----------------
    n_chim = int(n_pairs * cfg.chimeric_frac)
    n_near = int(n_pairs * cfg.near_frac)
    n_prop = n_pairs - n_chim - n_near
    tid, p1 = rand_loc(n_prop)
    ins = (torch.randn(n_prop, generator=g, device=dev, dtype=torch.float64) * cfg.insert_sd
           + cfg.insert_mean).round().to(torch.int64).clamp(min=L + 1, max=2 * margin - 1)
    p2 = p1 + ins - L
    over = p2 + L > lens[tid]
    p2 = torch.where(over, p1, p2)
    ins = torch.where(over, torch.full_like(ins, L), ins)
    dup = rand(n_prop) < cfg.dup_frac
    dflag = dup.to(torch.int64) * DUP
    nid = torch.arange(n_prop, device=dev, dtype=torch.int64) + next_name
    next_name += n_prop
    m60 = torch.full((n_prop,), 60, dtype=torch.int64, device=dev)
    emit(dflag + (PAIRED | PROPER | MREVERSE | READ1), m60, tid, p1, tid, p2, ins, p1 + L, nid)
    emit(dflag + (PAIRED | PROPER | REVERSE | READ2), m60, tid, p2, tid, p1, -ins, p2 + L, nid)

    # ---------------- B. improper noise ----------------
    def improper(t1, q1, t2, q2, n):
        nonlocal next_name
        s1 = randint(0, 2, n); s2 = randint(0, 2, n)
        lowq = rand(n) < cfg.lowq_frac
        mq1 = torch.where(lowq, randint(0, 20, n), randint(20, 61, n))
        mq2 = torch.where(rand(n) < cfg.lowq_frac, randint(0, 20, n), randint(20, 61, n))
        dup = (rand(n) < cfg.dup_frac).to(torch.int64) * DUP
        nid = torch.arange(n, device=dev, dtype=torch.int64) + next_name
        next_name += n
        same = t1 == t2
        isz = torch.where(same, q2 - q1, torch.zeros_like(q1))
        emit(dup + PAIRED + READ1 + s1 * REVERSE + s2 * MREVERSE, mq1, t1, q1, t2, q2, isz, q1 + L, nid)
        emit(dup + PAIRED + READ2 + s2 * REVERSE + s1 * MREVERSE, mq2, t2, q2, t1, q1, -isz, q2 + L, nid)

    if n_chim:
        t1, q1 = rand_loc(n_chim); t2, q2 = rand_loc(n_chim)
        improper(t1, q1, t2, q2, n_chim)
    if n_near:
        t1, q1 = rand_loc(n_near)
        q2 = (q1 + randint(-1500, 1500, n_near)).clamp(min=0)
        q2 = torch.minimum(q2, lens[t1] - L - 1)
        improper(t1, q1, t1, q2, n_near)

    # ---------------- C/D. planted SVs ----------------
    n_sv = cfg.n_tra + cfg.n_inv + cfg.n_dup + cfg.n_del
    truth = {k: torch.zeros(n_sv, dtype=torch.int64, device=dev) for k in ("type", "A", "a", "B", "b")}
    if n_sv:
        typ = torch.cat([torch.full((c,), t, dtype=torch.int64, device=dev) for t, c in
                         ((1, cfg.n_tra), (2, cfg.n_inv), (3, cfg.n_dup), (4, cfg.n_del))])
        # junction sites on a jittered grid so no two planted breakpoints are close
        n_site = 2 * n_sv
        grid = genome // n_site
        assert grid > 3 * cfg.min_sv_sep, "genome too small for the requested number of SVs"
        perm = torch.randperm(n_site, generator=g, device=dev)
        gp = perm * grid + grid // 4 + (rand(n_site) * (grid // 2)).to(torch.int64)
        stid = torch.searchsorted(cum, gp, right=True) - 1
        spos = (gp - cum[stid]).clamp(min=margin)
        spos = torch.minimum(spos, lens[stid] - margin)
        A, a = stid[:n_sv].clone(), spos[:n_sv].clone()      # a, b are 1-based SAM coordinates
        B, b = stid[n_sv:].clone(), spos[n_sv:].clone()
        # same-chromosome types: place B on A's chromosome at a fixed large offset
        off = cfg.min_sv_sep + (rand(n_sv) * cfg.min_sv_sep).to(torch.int64)
        same = typ != 1
        B = torch.where(same, A, B)
        b_del = torch.minimum(a + off, lens[A] - margin)       # DEL / INV: b > a
        b_dup = (a - off).clamp(min=margin)                    # DUP: b < a
        b = torch.where(typ == 3, b_dup, torch.where(same, b_del, b))
        # translocations whose two sites fell on one chromosome: move B to the next chromosome
        clash = (typ == 1) & (A == B)
        B = torch.where(clash, (A + 1) % n_chr, B)
        b = torch.where(clash, torch.minimum(b, lens[B] - margin), b)
        truth = {"type": typ, "A": A, "a": a, "B": B, "b": b}

        # spanning pairs
        m = cfg.span_per_sv
        sv = torch.arange(n_sv, device=dev).repeat_interleave(m)
        ns = sv.numel()
        d1 = randint(0, 250, ns); d2 = randint(0, 250, ns)
        inv = typ[sv] == 2
        r1pos = a[sv] - L - d1 - 1                                  # 0-based
        r2pos = torch.where(inv, b[sv] - L - d2 - 1, b[sv] + d2 - 1)
        f1 = torch.where(inv, torch.full_like(sv, PAIRED | READ1), torch.full_like(sv, PAIRED | MREVERSE | READ1))
        f2 = torch.where(inv, torch.full_like(sv, PAIRED | READ2), torch.full_like(sv, PAIRED | REVERSE | READ2))
        nid = torch.arange(ns, device=dev, dtype=torch.int64) + next_name
        next_name += ns
        m60 = torch.full((ns,), 60, dtype=torch.int64, device=dev)
        z = torch.zeros(ns, dtype=torch.int64, device=dev)
        emit(f1, m60, A[sv], r1pos, B[sv], r2pos, z, r1pos + L, nid)
        emit(f2, m60, B[sv], r2pos, A[sv], r1pos, z, r2pos + L, nid)

        # split reads: primary (+mate) and the 0x100 record
        s = cfg.split_per_sv
        sv = torch.arange(n_sv, device=dev).repeat_interleave(s)
        ns = sv.numel()
        k = randint(cfg.split_k_min if cfg.split_k_min is not None else L // 2 + 1,
                    cfg.split_k_max if cfg.split_k_max is not None else L - 20, ns)   # bases on the A side
        jit = randint(-cfg.sv_jitter, cfg.sv_jitter + 1, ns) if cfg.sv_jitter else torch.zeros(ns, dtype=torch.int64, device=dev)
        aa = a[sv] + jit
        bb = b[sv] + jit
        inv = typ[sv] == 2
        ppos1 = aa - k + 1                                           # 1-based start of primary
        spos1 = torch.where(inv, bb - (L - k) + 1, bb)               # 1-based start of the 0x100 record
        nid = torch.arange(ns, device=dev, dtype=torch.int64) + next_name
        next_name += ns
        m60 = torch.full((ns,), 60, dtype=torch.int64, device=dev)
        mate = ppos1 - 1 + 200                                       # proper mate downstream
        base = len(sa_cig0) and 0
        sa_base = sum(x.numel() for x in sa_cig0)
        idx_p = torch.arange(ns, device=dev, dtype=torch.int64) + sa_base
        idx_s = idx_p + ns
        # primary: kM(L-k)S
        emit(torch.full_like(sv, PAIRED | PROPER | MREVERSE | READ1), m60, A[sv], ppos1 - 1, A[sv], mate,
             torch.full_like(sv, 200 + L), ppos1 - 1 + k, nid, idx_p)
        # its mate (plain proper read)
        emit(torch.full_like(sv, PAIRED | PROPER | REVERSE | READ2), m60, A[sv], mate, A[sv], ppos1 - 1,
             torch.full_like(sv, -(200 + L)), mate + L, nid)
        # 0x100 record: kS(L-k)M, or (L-k)MkS reversed for INV
        fsec = torch.where(inv, torch.full_like(sv, PAIRED | PROPER | MREVERSE | READ1 | SECONDARY | REVERSE),
                           torch.full_like(sv, PAIRED | PROPER | MREVERSE | READ1 | SECONDARY))
        emit(fsec, m60, B[sv], spos1 - 1, A[sv], mate, z[:ns] if ns <= z.numel() else torch.zeros(ns, dtype=torch.int64, device=dev),
             spos1 - 1 + (L - k), nid, idx_s)
        # cigars
        pc0 = (k << 4) | OP_M; pc1 = ((L - k) << 4) | OP_S
        sc0 = torch.where(inv, ((L - k) << 4) | OP_M, (k << 4) | OP_S)
        sc1 = torch.where(inv, (k << 4) | OP_S, ((L - k) << 4) | OP_M)
        sa_cig0 += [pc0, sc0]; sa_cig1 += [pc1, sc1]
        sa_parts.append(dict(rtid=torch.cat([B[sv], A[sv]]), rpos=torch.cat([spos1, ppos1]),
                             minus=torch.cat([inv, torch.zeros_like(inv)]),
                             n0=torch.cat([torch.where(inv, L - k, k), k]),
                             o0=torch.cat([torch.where(inv, torch.full_like(k, OP_M), torch.full_like(k, OP_S)), torch.full_like(k, OP_M)]),
                             n1=torch.cat([torch.where(inv, k, L - k), L - k]),
                             o1=torch.cat([torch.where(inv, torch.full_like(k, OP_S), torch.full_like(k, OP_M)), torch.full_like(k, OP_S)])))

    # ---------------- merge + coordinate sort ----------------
    C = {}
    for k in list(cols.keys()):
        C[k] = torch.cat(cols.pop(k))
    mark = torch.cat(sa_mark)
    del sa_mark
    key = (C["tid"].to(torch.int64) << 32) | C["pos"].to(torch.int64)
    order = torch.sort(key, stable=True).indices
    del key
    out = {}
    for k in list(C.keys()):
        out[k] = C.pop(k)[order]
    mark = mark[order]
    del order
    sa_rec = torch.nonzero(mark >= 0).flatten()
    sa_src = mark[sa_rec]                           # index into generation-order SA arrays
    n_sa = sa_rec.numel()
    if n_sa:
        c0 = torch.cat(sa_cig0)[sa_src]; c1 = torch.cat(sa_cig1)[sa_src]
        cig_ops = torch.stack([c0, c1], 1).flatten()
        cig_off = torch.arange(n_sa + 1, device=dev, dtype=torch.int64) * 2
        P = {k: torch.cat([p[k] for p in sa_parts])[sa_src] for k in sa_parts[0]}
        tab, tl = _chr_name_table(n_chr, dev)
        opch = torch.tensor([ord(c) for c in "MIDNSHP=X"], dtype=torch.uint8, device=dev)
        strand = torch.where(P["minus"], torch.tensor(ord('-'), device=dev), torch.tensor(ord('+'), device=dev)).to(torch.uint8)
        one = torch.ones(n_sa, dtype=torch.int64, device=dev)
        sa_off, sa_txt = format_fields([
            ('t', tab[P["rtid"]], tl[P["rtid"]]), ('s', b','), ('i', P["rpos"]), ('s', b','),
            ('t', strand[:, None], one), ('s', b','),
            ('i', P["n0"]), ('t', opch[P["o0"]][:, None], one), ('i', P["n1"]), ('t', opch[P["o1"]][:, None], one),
            ('s', b',60,0;')], dev)
    else:
        cig_ops = torch.zeros(0, dtype=torch.int64, device=dev)
        cig_off = torch.zeros(1, dtype=torch.int64, device=dev)
        sa_off = torch.zeros(1, dtype=torch.int64, device=dev)
        sa_txt = torch.zeros(0, dtype=torch.uint8, device=dev)
    return SynthData(cfg=cfg, cols=out, sa_rec=sa_rec, cig_off=cig_off, cig_ops=cig_ops,
                     sa_off=sa_off, sa_txt=sa_txt, truth=truth)


# ----------------------------------------------------------------------------------------------
# name hashing for synthetic read names "r%010d" (must equal bkid_name_hash on that string)
# ----------------------------------------------------------------------------------------------
_M64 = (1 << 64) - 1


def name_of(name_id: int) -> bytes:
    return b"r%010d" % name_id


def name_hash_py(s: bytes):
    a, b = 0xcbf29ce484222325, 0x9E3779B97F4A7C15
    for c in s:
        a = ((a ^ c) * 0x100000001b3) & _M64
        b = ((b ^ c) * 0xff51afd7ed558ccd) & _M64
        b ^= b >> 32
    return a, b


def _mul64(x: torch.Tensor, k: int) -> torch.Tensor:
    """wrapping 64-bit multiply of an int64 tensor (bit pattern = uint64) by constant k."""
    k = k & _M64
    ks = k - (1 << 64) if k >= (1 << 63) else k
    return x * ks      # torch int64 multiplication wraps modulo 2^64


def name_hash_ids(name_id: torch.Tensor) -> torch.Tensor:
    """Vectorised bkid_name_hash of the synthetic names; returns int64 tensor [n, 2] (lo, hi bit
    patterns)."""
    dev = name_id.device
    n = name_id.numel()
    a = torch.full((n,), 0xcbf29ce484222325 - (1 << 64), dtype=torch.int64, device=dev)
    b = torch.full((n,), 0x9E3779B97F4A7C15 - (1 << 64), dtype=torch.int64, device=dev)

    def step(a, b, c):
        a = _mul64(a ^ c, 0x100000001b3)
        b = _mul64(b ^ c, 0xff51afd7ed558ccd)
        b = b ^ ((b >> 32) & 0xFFFFFFFF)        # logical shift
        return a, b

    a, b = step(a, b, torch.full((n,), ord('r'), dtype=torch.int64, device=dev))
    p = 10 ** 9
    for _ in range(10):
        c = (name_id // p) % 10 + 48
        a, b = step(a, b, c)
        p //= 10
    return torch.stack([a, b], 1)


# ----------------------------------------------------------------------------------------------
# genome / nib / annotation files
# ----------------------------------------------------------------------------------------------
NIB_MAGIC = 0x6BE93D3A
_NIB_CODE = {"T": 0, "C": 1, "A": 2, "G": 3, "N": 4}


def random_nib_bytes(length: int, seed: int, device="cpu", homopolymer_at=()) -> torch.Tensor:
    """packed 4-bit payload (no header) of a uniform ACGT chromosome; high nibble first
    (reference src/nibtools.cc:49-64).  ``homopolymer_at`` = 0-based positions where a run of 14
    identical bases is forced (exercises is_rpt)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    nb = (length + 1) // 2
    codes = torch.randint(0, 4, (nb * 2,), generator=g, device=device, dtype=torch.uint8)
    for p in homopolymer_at:
        codes[p:p + 14] = codes[p]
    if length % 2:
        codes[-1] = 0
    return (codes[0::2] << 4) | codes[1::2]


_NIB_ASCII = np.frombuffer(b"TCAGNNNNTCAGNNNN", np.uint8)          # nib code -> base (src/nibtools.cc:55-61; bit 3 = mask flag)
_BAM_CODE = {ord("A"): 1, ord("C"): 2, ord("G"): 4, ord("T"): 8}
_COMP = bytes.maketrans(b"ACGTN", b"TGCAN")


def nib_ascii(payload, length: int) -> np.ndarray:
    """packed 4-bit nib payload -> ASCII bases (uint8 array of `length`)"""
    p = payload.cpu().numpy() if hasattr(payload, "cpu") else np.asarray(payload)
    codes = np.empty(p.shape[0] * 2, np.uint8)
    codes[0::2] = p >> 4; codes[1::2] = p & 0xf
    return _NIB_ASCII[codes[:length]]


def pack_bam_seq(ascii_bases: bytes) -> bytes:
    """ASCII bases -> BAM 4-bit packing ("=ACMGRSVTWYHKDBN", high nibble first)"""
    c = [_BAM_CODE.get(b, 15) for b in ascii_bases]
    if len(c) % 2:
        c.append(0)
    return bytes((c[i] << 4) | c[i + 1] for i in range(0, len(c), 2))


def split_read_sequences(hb, genome: List[np.ndarray], corrupt=(), seed: int = 0):
    """Read bases for the SA-tagged records of a synthetic batch, consistent with the genome: matched operations copy the
    reference under the record, the soft clip carries the bases the SA tag points at (reverse-complemented when the two
    alignments are on different strands).  Records listed in ``corrupt`` (indices into the SA table) get random clip
    bases instead -- split alignments the validator must reject.  Returns (seq table dict for HostBatch, list of ASCII reads)."""
    rng = np.random.RandomState(seed)
    s = hb.side
    names = {n: t for t, n in enumerate(hb.target_names)}
    reads, packed, lens = [], [], []
    for k in range(hb.n_sa):
        i = int(s["sa_rec"][k])
        tid, pos, flag = int(hb.cols["tid"][i]), int(hb.cols["pos"][i]), int(hb.cols["flag"][i])
        ops = s["cig_ops"][int(s["cig_off"][k]):int(s["cig_off"][k + 1])]
        f = bytes(s["sa_txt"][int(s["sa_off"][k]):int(s["sa_off"][k + 1])]).split(b";")[0].split(b",")
        sa_tid, sa_pos, sa_minus = names.get(f[0].decode(), -1), int(f[1]), f[2] == b"-"
        sa_m, num = 0, b""
        for ch in f[3]:
            if 48 <= ch <= 57: num += bytes([ch])
            else:
                if ch in b"M=X": sa_m += int(num)
                num = b""
        window = bytes(genome[sa_tid][sa_pos - 1:sa_pos - 1 + sa_m]) if sa_tid >= 0 else b"N" * sa_m
        if sa_minus != bool(flag & REVERSE):
            window = window.translate(_COMP)[::-1]
        out, cur = b"", pos
        for op in ops:
            ln, o = int(op) >> 4, int(op) & 0xf
            if o in (OP_M, OP_EQ, OP_X):
                out += bytes(genome[tid][cur:cur + ln]); cur += ln
            elif o == OP_S:
                clip = window
                if k in corrupt:
                    clip = bytes(rng.choice(np.frombuffer(b"ACGT", np.uint8), ln))
                out += (clip + b"N" * ln)[:ln]
            elif o == OP_I:
                out += b"N" * ln
            elif o in (OP_D, OP_N):
                cur += ln
        reads.append(out); packed.append(pack_bam_seq(out)); lens.append(len(out))
    off = np.concatenate([[0], np.cumsum([len(p) for p in packed])]).astype(np.uint32)
    seq4 = np.frombuffer(b"".join(packed), np.uint8).copy() if packed else np.zeros(0, np.uint8)
    return {"seq_off": off, "seq4": seq4, "seq_len": np.array(lens, np.int32)}, reads


def write_nib(path: str, payload: torch.Tensor, length: int):
    with open(path, "wb") as f:
        f.write(np.array([NIB_MAGIC, length], dtype="<u4").tobytes())
        f.write(payload.cpu().numpy().tobytes())


def write_ref_names(path: str, n_chr: int):
    with open(path, "w") as f:
        for t in range(n_chr):
            f.write(chrom_name(t) + "\n")


def write_refgene(path: str, chrom_lens: List[int], genes_per_mb: float = 4.0, seed: int = 7):
    """Synthetic UCSC refGene.txt (16 tab-separated columns, parsed by the reference at
    src/RefSeqTranscript.cc:19-79).  Every transcript has a CDS (the reference underflows on
    CDS-less overlaps, src/BreakID.cc:1757) ; a few NR_ rows exercise the skip rule."""
    rng = np.random.RandomState(seed)
    rows = []
    gid = 0
    for tid, clen in enumerate(chrom_lens):
        ng = max(1, int(clen / 1e6 * genes_per_mb))
        starts = np.sort(rng.randint(1000, max(1001, clen - 60000), ng))
        for s in starts:
            gid += 1
            glen = int(rng.randint(8000, 50000))
            ne = int(rng.randint(2, 9))
            cuts = np.sort(rng.choice(np.arange(100, glen - 100), 2 * ne, replace=False))
            es = s + cuts[0::2]; ee = s + cuts[1::2]
            tx_s, tx_e = int(es[0]), int(ee[-1])
            cds_s = int(es[0] + (ee[0] - es[0]) // 3)
            cds_e = int(ee[-1] - (ee[-1] - es[-1]) // 3)
            strand = "+" if rng.rand() < 0.5 else "-"
            name = ("NR_%06d" % gid) if gid % 17 == 0 else ("NM_%06d" % gid)
            rows.append("\t".join([
                "0", name, chrom_name(tid), strand, str(tx_s), str(tx_e), str(cds_s), str(cds_e), str(ne),
                ",".join(map(str, es)) + ",", ",".join(map(str, ee)) + ",", "0", "GENE%d" % gid,
                "cmpl", "cmpl", ",".join(["0"] * ne) + ","]))
    with open(path, "w") as f:
        f.write("\n".join(rows) + "\n")


def config1(seed: int = 1) -> SynthConfig:
    """BASELINE.json configs[0]: 1 Mb two-chromosome genome, 30x, 10 planted SVs."""
    return SynthConfig(chrom_lens=[600000, 400000], seed=seed)


def config2(scale: float = 1.0, seed: int = 2) -> SynthConfig:
    """BASELINE.json configs[1]: hg19-shaped 3.1 Gb genome, 30x 2x150 bp, 2000 SVs, 1 % chimeric
    noise.  ``scale`` < 1 shrinks every chromosome (bounded samples for the CPU arms)."""
    lens = [max(200000, int(l * scale)) for l in HG19_LENS]
    nsv = max(8, int(2000 * scale))
    return SynthConfig(chrom_lens=lens, n_tra=nsv // 4, n_inv=nsv // 4, n_dup=nsv // 4, n_del=nsv - 3 * (nsv // 4), seed=seed)


def config4(scale: float = 1.0, seed: int = 4) -> SynthConfig:
    """BASELINE.json configs[3]: tumour-shaped 100x BAM with 500 planted translocations (gene fusions; the
    annotation path runs on the host over a synthetic refGene, ``write_refgene``)."""
    lens = [max(200000, int(l * scale)) for l in HG19_LENS]
    return SynthConfig(chrom_lens=lens, coverage=100.0, n_tra=max(4, int(500 * scale)), n_inv=0, n_dup=0, n_del=0,
                       span_per_sv=40, split_per_sv=20, seed=seed)


def config5(scale: float = 1.0, seed: int = 5, split_per_sv: int = 5000) -> SynthConfig:
    """BASELINE.json configs[4]: split-read refinement stress.  1000 x scale breakpoint hotspots, each with
    ``split_per_sv`` split reads (2 SA-tagged records per split read => 1e7 SA-tagged records at scale 1), clip
    lengths U(20,130) on 150 bp reads, breakpoints jittered +-3 bp (exercises the +-2 vote), thin 2x background."""
    lens = [max(200000, int(l * scale)) for l in HG19_LENS]
    nsv = max(4, int(1000 * scale))
    return SynthConfig(chrom_lens=lens, coverage=2.0, n_tra=nsv // 4, n_inv=nsv // 4, n_dup=nsv // 4, n_del=nsv - 3 * (nsv // 4),
                       split_per_sv=split_per_sv, sv_jitter=3, split_k_min=20, split_k_max=131, seed=seed)
