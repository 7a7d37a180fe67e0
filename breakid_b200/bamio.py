"""Minimal BAM / SAM *writer* for synthetic workloads (test / bench tooling, not on the hot path).

Writes the record batch of ``synth.SynthData`` in its own record order as a real BGZF-compressed BAM so
that the unmodified reference CPU binary can be run on byte-identical input.  ``sort_order`` is the @HD SO: tag
("coordinate" for the batches synth.generate makes; "unsorted" / "queryname" for synth.permute'd ones).  The `.bai` index is
NOT written here: tests build it with ``oracle/_ref/bamindex`` (the reference's own vendored
htslib), the product only checks that the index file exists (reference src/BreakID.cc:411-416).
"""
from __future__ import annotations

import struct
import zlib
from typing import List

import numpy as np

from . import synth

_BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def _bgzf_block(data: bytes, level: int) -> bytes:
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    bsize = len(comp) + 25
    return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize)
            + comp + struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data)))


def reg2bin(beg: np.ndarray, end: np.ndarray) -> np.ndarray:
    """UCSC binning scheme (SAM spec §5.3); end is exclusive."""
    end = end - 1
    out = np.zeros_like(beg)
    done = np.zeros(beg.shape, dtype=bool)
    for shift, base in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        hit = ((beg >> shift) == (end >> shift)) & ~done
        out[hit] = base + (beg[hit] >> shift)
        done |= hit
    return out


def write_bam(path: str, d: synth.SynthData, random_qual: bool = True, level: int = 1,
              chunk: int = 200_000, sa_seq=None, sort_order: str = "coordinate") -> None:
    """``sort_order`` = the @HD SO: value; the records are written in the batch's order whatever it says.
    ``sa_seq`` = optional seq table (seq_off / seq4 / seq_len, see synth.split_read_sequences): real read bases for
    the SA-tagged records (all other records carry a constant sequence)."""
    cfg = d.cfg
    L = cfg.read_len
    c = {k: v.cpu().numpy() for k, v in d.cols.items()}
    n = c["flag"].shape[0]
    flag = c["flag"].astype(np.uint16)
    sa_rec = d.sa_rec.cpu().numpy()
    cig_off = d.cig_off.cpu().numpy(); cig_ops = d.cig_ops.cpu().numpy().astype(np.uint32)
    sa_off = d.sa_off.cpu().numpy(); sa_txt = d.sa_txt.cpu().numpy()
    is_sa = np.zeros(n, dtype=bool); is_sa[sa_rec] = True
    sa_slot = np.full(n, -1, dtype=np.int64); sa_slot[sa_rec] = np.arange(sa_rec.shape[0])

    NAME = 12                       # "r%010d" + NUL
    seq_b = (L + 1) // 2
    fixed = 32 + NAME + 4 + seq_b + L          # record bytes after block_size, 1 cigar op, no aux
    rng = np.random.RandomState(cfg.seed + 12345)

    # header
    text = "@HD\tVN:1.4\tSO:%s\n" % sort_order + "".join(
        "@SQ\tSN:%s\tLN:%d\n" % (synth.chrom_name(t), l) for t, l in enumerate(cfg.chrom_lens))
    hdr = b"BAM\x01" + struct.pack("<i", len(text)) + text.encode() + struct.pack("<i", len(cfg.chrom_lens))
    for t, l in enumerate(cfg.chrom_lens):
        nm = synth.chrom_name(t).encode() + b"\x00"
        hdr += struct.pack("<i", len(nm)) + nm + struct.pack("<i", l)

    out = open(path, "wb")
    pending = bytearray(hdr)

    from concurrent.futures import ThreadPoolExecutor
    import os as _os
    pool = ThreadPoolExecutor(max(1, min(32, _os.cpu_count() or 1)))     # zlib releases the GIL
    futures = []

    def flush(final=False):
        nonlocal pending
        mv = memoryview(pending)
        o = 0
        blks = []
        while len(pending) - o >= 0xff00 or (final and o < len(pending)):
            blk = bytes(mv[o:o + 0xff00])
            blks.append(blk)
            o += len(blk)
        mv.release()
        futures.extend(pool.submit(_bgzf_block, b, level) for b in blks)      # compression overlaps the record assembly
        while len(futures) > 4096:                                             # bound the backlog: write the oldest blocks
            out.write(futures.pop(0).result())
        pending = pending[o:]

    flush()
    digits = np.array([10 ** (9 - i) for i in range(10)], dtype=np.int64)
    head_dt = np.dtype([
        ("block_size", "<i4"), ("tid", "<i4"), ("pos", "<i4"), ("l_name", "u1"), ("mapq", "u1"),
        ("bin", "<u2"), ("n_cigar", "<u2"), ("flag", "<u2"), ("l_seq", "<i4"),
        ("mtid", "<i4"), ("mpos", "<i4"), ("isize", "<i4"), ("name", "u1", NAME)])
    hw = head_dt.itemsize                               # 36 + NAME
    row_w = hw + 4 + seq_b + L                          # a record without aux, one cigar op: every non-SA record
    cig1 = np.frombuffer(struct.pack("<I", (L << 4) | 0), dtype=np.uint8)
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        m = e - s
        sa_m = is_sa[s:e]
        idx_sa = np.nonzero(sa_m)[0]
        # fixed part of every record as a structured block
        rec = np.zeros(m, dtype=head_dt)
        rec["block_size"] = fixed
        rec["tid"] = c["tid"][s:e]; rec["pos"] = c["pos"][s:e]
        rec["l_name"] = NAME; rec["mapq"] = c["mapq"][s:e]
        rec["bin"] = reg2bin(c["pos"][s:e].astype(np.int64), c["endpos"][s:e].astype(np.int64))
        rec["n_cigar"] = 1; rec["flag"] = flag[s:e]; rec["l_seq"] = L
        rec["mtid"] = c["mtid"][s:e]; rec["mpos"] = c["mpos"][s:e]; rec["isize"] = c["isize"][s:e]
        nid = c["name_id"][s:e]
        nm = np.zeros((m, NAME), dtype=np.uint8)
        nm[:, 0] = ord("r")
        nm[:, 1:11] = ((nid[:, None] // digits[None, :]) % 10 + 48).astype(np.uint8)
        rec["name"] = nm
        # all records laid out as fixed-width rows (column slices, no index arrays); the few SA-tagged records are
        # re-serialised with their own cigar / tag bytes and spliced in between the runs of plain rows
        rows = np.empty((m, row_w), dtype=np.uint8)
        rows[:, :hw] = rec.view(np.uint8).reshape(m, hw)
        rows[:, hw:hw + 4] = cig1
        rows[:, hw + 4:hw + 4 + seq_b] = 0x11
        rows[:, hw + 4 + seq_b:] = rng.randint(2, 41, (m, L)).astype(np.uint8) if random_qual else 30
        if idx_sa.size == 0:
            pending += rows.tobytes()
        else:
            prev = 0
            for j in idx_sa:
                if j > prev:
                    pending += rows[prev:j].tobytes()
                k = sa_slot[s + j]
                ops = cig_ops[cig_off[k]:cig_off[k + 1]]
                sq = b"\x11" * seq_b if sa_seq is None else bytes(sa_seq["seq4"][int(sa_seq["seq_off"][k]):int(sa_seq["seq_off"][k + 1])])
                assert len(sq) == seq_b
                blob = ops.astype("<u4").tobytes() + sq + (b"\x1e" * L) + b"SAZ" + sa_txt[sa_off[k]:sa_off[k + 1]].tobytes() + b"\x00"
                r1 = rec[j:j + 1].copy()
                r1["n_cigar"] = ops.shape[0]
                r1["block_size"] = hw - 4 + len(blob)
                pending += r1.tobytes() + blob
                prev = j + 1
            if prev < m:
                pending += rows[prev:].tobytes()
        flush()
    flush(final=True)
    for fu in futures:
        out.write(fu.result())
    pool.shutdown()
    out.write(_BGZF_EOF)
    out.close()


_NT16 = np.frombuffer(b"=ACMGRSVTWYHKDBN", dtype=np.uint8)


def write_sam(path: str, d: synth.SynthData, random_qual: bool = True, chunk: int = 200_000, sa_seq=None,
              sort_order: str = "coordinate") -> None:
    """The records ``write_bam`` writes (same arguments, same names, cigars, SA tags, bases and qualities) as SAM text:
    RNEXT is "=" when the mate is on the record's own target, SEQ spells the 4-bit codes, QUAL is Phred + 33."""
    cfg = d.cfg
    L = cfg.read_len
    c = {k: v.cpu().numpy() for k, v in d.cols.items()}
    n = c["flag"].shape[0]
    sa_rec = d.sa_rec.cpu().numpy()
    cig_off = d.cig_off.cpu().numpy(); cig_ops = d.cig_ops.cpu().numpy().astype(np.uint32)
    sa_off = d.sa_off.cpu().numpy(); sa_txt = d.sa_txt.cpu().numpy()
    sa_slot = np.full(n, -1, dtype=np.int64); sa_slot[sa_rec] = np.arange(sa_rec.shape[0])
    rng = np.random.RandomState(cfg.seed + 12345)          # the qualities write_bam draws, in the same order
    names = [synth.chrom_name(t) for t in range(len(cfg.chrom_lens))]
    with open(path, "wb") as out:
        out.write(("@HD\tVN:1.4\tSO:%s\n" % sort_order + "".join("@SQ\tSN:%s\tLN:%d\n" % (names[t], l) for t, l in enumerate(cfg.chrom_lens))).encode())
        plain = "%dM" % L
        seq_plain = b"A" * L
        for s in range(0, n, chunk):
            e = min(n, s + chunk)
            m = e - s
            q = (rng.randint(2, 41, (m, L)).astype(np.uint8) if random_qual else np.full((m, L), 30, np.uint8)) + 33
            qb = q.tobytes()
            tid = c["tid"][s:e].tolist(); pos = c["pos"][s:e].tolist(); mapq = c["mapq"][s:e].tolist(); flag = c["flag"][s:e].tolist()
            mtid = c["mtid"][s:e].tolist(); mpos = c["mpos"][s:e].tolist(); isize = c["isize"][s:e].tolist(); nid = c["name_id"][s:e].tolist()
            parts = []
            for j in range(m):
                t, mt = tid[j], mtid[j]
                k = sa_slot[s + j]
                rn = names[t] if t >= 0 else "*"
                rx = "*" if mt < 0 else "=" if mt == t else names[mt]
                if k < 0:
                    parts.append(("r%010d\t%d\t%s\t%d\t%d\t%s\t%s\t%d\t%d\t" % (nid[j], flag[j], rn, pos[j] + 1, mapq[j], plain, rx, mpos[j] + 1, isize[j])).encode())
                    parts.append(seq_plain); parts.append(b"\t"); parts.append(qb[j * L:(j + 1) * L]); parts.append(b"\n")
                    continue
                ops = cig_ops[cig_off[k]:cig_off[k + 1]]
                cig = "".join("%d%s" % (int(o) >> 4, "MIDNSHP=X"[int(o) & 15]) for o in ops)
                if sa_seq is None:
                    sq = seq_plain
                else:
                    b = np.asarray(sa_seq["seq4"][int(sa_seq["seq_off"][k]):int(sa_seq["seq_off"][k + 1])], np.uint8)
                    sq = _NT16[np.stack([b >> 4, b & 15], 1).reshape(-1)[:L]].tobytes()
                parts.append(("r%010d\t%d\t%s\t%d\t%d\t%s\t%s\t%d\t%d\t" % (nid[j], flag[j], rn, pos[j] + 1, mapq[j], cig, rx, mpos[j] + 1, isize[j])).encode())
                parts.append(sq); parts.append(b"\t" + b"?" * L + b"\tSA:Z:"); parts.append(sa_txt[sa_off[k]:sa_off[k + 1]].tobytes()); parts.append(b"\n")
            out.write(b"".join(parts))


def write_dataset(dirpath: str, d: synth.SynthData, random_qual: bool = True, nib: bool = True,
                  genes_per_mb: float = 4.0, sort_order: str = "coordinate", sam: bool = False) -> dict:
    """Lay down everything a BreakID run needs: <dir>/reads.bam, <dir>/nib/{ref_names.txt,
    hg19_<chr>.nib}, <dir>/ref_files/refGene.txt, and with ``sam`` also <dir>/reads.sam (the same records as text).
    Returns the paths."""
    import os
    os.makedirs(os.path.join(dirpath, "nib"), exist_ok=True)
    os.makedirs(os.path.join(dirpath, "ref_files"), exist_ok=True)
    cfg = d.cfg
    bam = os.path.join(dirpath, "reads.bam")
    write_bam(bam, d, random_qual=random_qual, sort_order=sort_order)
    paths = {}
    if sam:
        paths["sam"] = os.path.join(dirpath, "reads.sam")
        write_sam(paths["sam"], d, random_qual=random_qual, sort_order=sort_order)
    synth.write_ref_names(os.path.join(dirpath, "nib", "ref_names.txt"), len(cfg.chrom_lens))
    if nib:
        for t, l in enumerate(cfg.chrom_lens):
            pay = synth.random_nib_bytes(l, cfg.seed * 1000 + t)
            synth.write_nib(os.path.join(dirpath, "nib", "hg19_%s.nib" % synth.chrom_name(t)), pay, l)
    synth.write_refgene(os.path.join(dirpath, "ref_files", "refGene.txt"), cfg.chrom_lens, genes_per_mb=genes_per_mb)
    return dict({"bam": bam, "nib": os.path.join(dirpath, "nib"), "refgene": os.path.join(dirpath, "ref_files", "refGene.txt")}, **paths)
