"""SAM input (bkid_push_sam, BreakID -i reads.sam / -i -): alignment text parsed on the device.

The expected result is defined by construction: the run on the BAM that holds the same records.  A small SAM-line ->
BAM-record encoder below (SAM spec 1.4 / 4.2) gives that BAM for any text; the CPU tests prove it against
bamio.write_bam, the GPU tests compare every column of push_sam with the host BAM decoder and push_bgzf of the encoded
BAM, and the calls with the oracle."""
import os
import re
import struct
import subprocess

import numpy as np
import pytest

from breakid_b200 import api, bamio, synth
from test_bgzf_decode import _bgzf_write, _raw_bam

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "breakid_b200", "host", "BreakID")
DENSE = (("flag", np.uint16), ("mapq", np.uint8), ("tid", np.int32), ("pos", np.int32), ("isize", np.int32), ("endpos", np.int32))
ALL = DENSE + api._XCOLS + api._SIDE + api._SEQ
TARGETS = [("chr1", 500000), ("chr2", 400000)]


# ------------------------------------------------------------------------------------------------ the encoder (oracle)
def _aux(field: bytes) -> bytes:
    tag, ty, val = field[:2], field[3:4], field[5:]
    if ty == b"A":
        return tag + b"A" + val
    if ty == b"i":
        return tag + b"i" + struct.pack("<i", int(val))
    if ty == b"f":
        return tag + b"f" + struct.pack("<f", float(val))
    if ty in (b"Z", b"H"):
        return tag + ty + val + b"\0"
    sub, *vals = val.split(b",")
    fmt = {b"c": "b", b"C": "B", b"s": "h", b"S": "H", b"i": "i", b"I": "I", b"f": "f"}[sub]
    conv = float if sub == b"f" else int
    return tag + b"B" + sub + struct.pack("<i", len(vals)) + b"".join(struct.pack("<" + fmt, conv(v)) for v in vals)


def sam_to_bam(line: bytes, names) -> bytes:
    """one SAM alignment line (without its newline) -> the BAM record (block_size included) holding the same record"""
    if line.endswith(b"\r"):
        line = line[:-1]
    f = line.split(b"\t")
    qname, flag, rname, pos, mapq, cigar, rnext, pnext, tlen, seq, qual = f[:11]
    tids = {n.encode(): t for t, n in enumerate(names)}
    tid = -1 if rname == b"*" else tids[rname]
    mtid = -1 if rnext == b"*" else tid if rnext == b"=" else tids[rnext]
    ops = [] if cigar == b"*" else [(int(n), "MIDNSHP=X".index(op.decode())) for n, op in re.findall(rb"(\d+)([MIDNSHP=X])", cigar)]
    l_seq = 0 if seq == b"*" else len(seq)
    codes = [max(0, "=ACMGRSVTWYHKDBN".find(chr(ch).upper())) if chr(ch).upper() in "=ACMGRSVTWYHKDBN" else 15 for ch in (seq if l_seq else b"")]
    codes += [0] * (len(codes) & 1)
    packed = bytes((codes[k] << 4) | codes[k + 1] for k in range(0, len(codes), 2))
    qb = b"\xff" * l_seq if qual == b"*" else bytes(q - 33 for q in qual)
    nm = qname + b"\0"
    body = struct.pack("<iiBBHHHiiii", tid, int(pos) - 1, len(nm), int(mapq), 4680, len(ops), int(flag), l_seq, mtid, int(pnext) - 1, int(tlen)) + nm
    body += b"".join(struct.pack("<I", (n << 4) | op) for n, op in ops) + packed + qb + b"".join(_aux(x) for x in f[11:])
    return struct.pack("<i", len(body)) + body


def encode_bam(path, text: bytes, targets):
    """the BAM holding the records of the SAM alignment lines `text`"""
    names = [n for n, _ in targets]
    lines = text.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    payload, first = _raw_bam([sam_to_bam(ln, names)[4:] for ln in lines], targets)
    _bgzf_write(path, payload)


def sam_header(targets):
    return ("@HD\tVN:1.4\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % t for t in targets)).encode()


def _hb_equal(a, b):
    for part in ("cols", "x", "side"):
        pa, pb = getattr(a, part), getattr(b, part)
        assert sorted(pa) == sorted(pb), part
        for k in pa:
            assert np.array_equal(np.asarray(pa[k]), np.asarray(pb[k])), (part, k)
    assert (a.seq is None) == (b.seq is None)
    if a.seq is not None:
        for k in a.seq:
            assert np.array_equal(a.seq[k], b.seq[k]), k


# ------------------------------------------------------------------------------------------------ hostile records
def hostile_lines(rng, n, crlf=False):
    """every record kind of test_bgzf_decode._hostile_records as SAM text, plus 254-character names, * SEQ with a CIGAR,
    * CIGAR with a SEQ, RNEXT = and *, SA:i before SA:Z, empty SA, OC without SA, B arrays on both sides of SA, IUPAC and
    lower-case bases and the unmapped tail"""
    out = []
    pos = 100
    for i in range(n):
        pos += int(rng.randint(0, 50))
        k = i % 16
        name = "read_%d_%s" % (i, "x" * int(rng.randint(0, 60)))
        if k == 12:
            name = ("L%d_" % i + "y" * 254)[:254]
        flag = int(rng.choice([99, 147, 65, 129, 97, 145, 1089, 4, 77, 141, 1, 2]))
        l_seq = int(rng.choice([1, 100, 151]))
        cig = "%dM" % l_seq
        aux = ["NM:i:1", "MD:Z:%d" % int(rng.randint(1, 150)), "AS:i:77"]
        if k == 1: aux.append("SA:Z:chr2,%d,+,40M60S,60,0;" % (pos + 7))
        if k == 2: aux += ["OC:Z:60M40S", "SA:Z:chr1,%d,-,60S40M,13,1;chr2,5,+,10M,0,0;" % (pos + 999)]
        if k == 3: aux.append("SA:Z:")                                    # empty SA: not an SA record
        if k == 4: aux += ["XB:B:s,1,2,3,4,5", "SA:Z:chrX,9,+,50M50S,60,0;", "YB:B:c,-1,2"]
        if k == 5: aux += ["XF:f:1.5", "XH:H:1A2B", "XA:A:q", "XS:i:-3"]
        if k == 6:
            l_seq = 10 + 30 + 5 + 20 + 35 + 10 + 5
            cig = "10S30M5I20M1000N35M8D10=5X3H"
        if k == 7: cig = "*"                                              # * CIGAR with a SEQ
        if k == 8: flag |= 4
        if k == 9: aux = []
        if k == 10: aux += ["SA:Z:chr1,1,+,1S1M,0,0;", "SA:Z:ignored,2,+,1M,0,0;"]    # the first SA:Z wins
        if k == 11: aux += ["XB:B:I," + ",".join("0" for _ in range(300)), "SA:i:5", "SA:Z:chr2,77,-,5M,1,0;", "OC:Z:4M1D"]
        if k == 13: aux += ["OC:Z:9M"]                                    # OC without SA
        seq = "".join(rng.choice(list("ACGTNacgtRYKM=."), l_seq))
        qual = "*" if k in (5, 7) else "".join(chr(33 + int(q)) for q in rng.randint(0, 41, l_seq))
        if k == 14: seq, qual = "*", "*"                                  # * SEQ with a CIGAR
        tid = 0 if i < n * 2 // 3 else 1
        if i == n * 2 // 3:
            pos = 5
        mt = int(rng.choice([-1, 0, 1]))
        rnext = "*" if mt < 0 else "=" if (mt == tid and k % 2) else TARGETS[mt][0]
        out.append("\t".join([name, str(flag), TARGETS[tid][0], str(pos + 1), str(int(rng.randint(0, 61))), cig, rnext,
                              str(int(rng.randint(0, 5000))), str(int(rng.randint(-900, 900))), seq, qual] + aux))
    out.append("unmapped_tail\t77\t*\t0\t0\t*\t*\t0\t0\t" + "A" * 30 + "\t" + "I" * 30)
    eol = "\r\n" if crlf else "\n"
    return (eol.join(out)).encode()                                       # no final newline


# ------------------------------------------------------------------------------------------------ CPU
def test_sam_header_parse(tmp_path):
    p = tmp_path / "h.sam"
    text = b"line one\tx\n"
    p.write_bytes(b"@HD\tVN:1.6\n@SQ\tSN:chrA\tLN:1000\tM5:x\n@CO\thello\n@SQ\tLN:25\tSN:chrB\r\n@RG\tID:1\n" + text)
    f = api.SamFile(str(p))
    assert f.target_names == ["chrA", "chrB"] and f.target_len == [1000, 25]
    assert f.first_line == 6 and f.first_record == p.stat().st_size - len(text) and f.text() == text
    f.close()
    for bad, msg in ((b"@SQ\tSN:a\tLN:5\n@SQ\tSN:a\tLN:6\n", "duplicate"), (b"@SQ\tSN:a\n", "without LN"),
                     (b"@SQ\tSN:a\tLN:5x\n", "not a number"), (b"@SQ\tSN:a\tLN:\n", "not a number"), (b"@SQ\tLN:5\n", "without SN"),
                     (b"@SQ\tSN:a\tLN:99999999999\n", "not a number")):
        q = tmp_path / "bad.sam"
        q.write_bytes(bad + b"r\t0\t*\t0\t0\t*\t*\t0\t0\t*\t*\n")
        with pytest.raises(IOError, match=msg):
            api.SamFile(str(q))
    q = tmp_path / "only_header.sam"                                     # header only, last line without newline
    q.write_bytes(b"@SQ\tSN:a\tLN:5\n@SQ\tSN:b\tLN:6")
    f = api.SamFile(str(q))
    assert f.target_names == ["a", "b"] and f.first_record == f.size and f.text() == b""
    q = tmp_path / "no_header.sam"
    q.write_bytes(b"r\t4\t*\t0\t0\t*\t*\t0\t0\t*\t*\n")
    f = api.SamFile(str(q))
    assert f.target_names == [] and f.first_record == 0 and f.first_line == 1
    g = api.SamFile(buf=sam_header(TARGETS))                             # the same parser on a buffer (stdin)
    assert g.target_names == ["chr1", "chr2"] and g.target_len == [500000, 400000] and g.first_line == 4
    with pytest.raises(IOError):
        api.SamFile(str(tmp_path / "missing.sam"))


def test_write_sam_equals_write_bam_through_the_encoder(tmp_path, small_data):
    """every line of bamio.write_sam(d) encodes to the record bamio.write_bam(d) wrote: the host BAM decoder reads the
    same columns from both BAMs (sparse table, SA side table and the read bases of the SA records included)"""
    d, hb, nibs = small_data
    genome = [synth.nib_ascii(p, l) for p, l in nibs]
    seq, _ = synth.split_read_sequences(hb, genome)
    pb, ps, pe = str(tmp_path / "w.bam"), str(tmp_path / "w.sam"), str(tmp_path / "e.bam")
    bamio.write_bam(pb, d, sa_seq=seq)
    bamio.write_sam(ps, d, sa_seq=seq)
    f = api.SamFile(ps)
    targets = list(zip(f.target_names, f.target_len))
    encode_bam(pe, f.text(), targets)
    a, b = api.HostBatch.from_bam(pb), api.HostBatch.from_bam(pe)
    assert a.n == hb.n and b.n == hb.n and a.seq is not None
    _hb_equal(a, b)


def test_hostile_encoder_roundtrip(tmp_path):
    """the hostile text encodes to a BAM the host decoder reads (the GPU tests compare against it)"""
    text = hostile_lines(np.random.RandomState(3), 400)
    p = str(tmp_path / "h.bam")
    encode_bam(p, text, TARGETS)
    hb = api.HostBatch.from_bam(p)
    assert hb.n == 401 and hb.n_sa > 0 and int((hb.cols["tid"] == -1).sum()) == 1


def test_driver_refusals_before_any_device(tmp_path):
    nib = str(tmp_path)
    txt = tmp_path / "notes.txt"
    txt.write_text("neither a BAM nor SAM\njust text\n")
    r = subprocess.run([DRIVER, "-i", str(txt), "-o", str(tmp_path / "o"), "-n", nib], capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and "can not open bam-file" in r.stderr
    r = subprocess.run([DRIVER, "-i", "-", "-gpu", "0,1", "-o", str(tmp_path / "o"), "-n", nib], input="", capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and "stdin needs one GPU" in r.stderr
    sam = tmp_path / "reads.sam"
    sam.write_bytes(sam_header(TARGETS) + b"r\t4\t*\t0\t0\t*\t*\t0\t0\t*\t*\n")
    r = subprocess.run([DRIVER, "-i", str(sam), "-o", str(tmp_path / "o"), "-n", nib], capture_output=True, text=True, timeout=60,
                       env=dict(os.environ, BKID_HOST_DECODE="1"))
    assert r.returncode == 1 and "host decode reads BAM only" in r.stderr
    assert "- for stdin" in subprocess.run([DRIVER, "-h"], capture_output=True, text=True, timeout=60).stderr


# ------------------------------------------------------------------------------------------------ GPU
def _ctx(names=TARGETS, **kw):
    return api.Context([l for _, l in names], [n for n, _ in names], device=0, **kw)


def _cols(c):
    return {k: c.fetch_column(k, dt) for k, dt in ALL}


def _assert_cols(got, exp, what=""):
    for k in exp:
        assert np.array_equal(got[k], exp[k]), (what, k)


def _push_sam(text, chunk_kb=None, **kw):
    if chunk_kb:
        os.environ["BKID_SAM_CHUNK_KB"] = str(chunk_kb)
    try:
        c = _ctx(**kw)
        n = c.push_sam(text)
    finally:
        os.environ.pop("BKID_SAM_CHUNK_KB", None)
    return c, n


@pytest.mark.gpu
@pytest.mark.parametrize("crlf", [False, True])
@pytest.mark.parametrize("chunk_kb", [None, 1, 16])
def test_columns_equal_bam_of_the_same_records(tmp_path, chunk_kb, crlf):
    text = hostile_lines(np.random.RandomState(3), 3000, crlf)
    p = str(tmp_path / "h.bam")
    encode_bam(p, text, TARGETS)
    hb = api.HostBatch.from_bam(p)
    f = api.BgzfFile(p)
    ref = _ctx()
    ref.push_bgzf(f)
    exp = _cols(ref)
    for k, dt in DENSE:                                          # the host decoder agrees with push_bgzf
        assert np.array_equal(exp[k], hb.cols[k].astype(dt)), k
    c, n = _push_sam(text, chunk_kb)
    assert n == hb.n == 3001
    st = c.decode_stats()
    assert st["n_records"] == n and st["uncompressed_bytes"] == len(text) and st["compressed_bytes"] == 0 and st["inflate_ms"] == 0
    if chunk_kb:
        assert st["n_chunks"] > 1
    _assert_cols(_cols(c), exp, chunk_kb)
    c.close(); ref.close(); f.close()


@pytest.mark.gpu
def test_split_pushes_and_append_after_bgzf(tmp_path):
    text = hostile_lines(np.random.RandomState(5), 2000) + b"\n"
    lines = text.split(b"\n")[:-1]
    one, _ = _push_sam(text)
    exp = _cols(one)
    rng = np.random.RandomState(1)
    for parts in range(1, 8):
        cuts = sorted(rng.choice(np.arange(1, len(lines)), parts - 1, replace=False).tolist()) if parts > 1 else []
        c = _ctx()
        first = 1
        for a, b in zip([0] + cuts, cuts + [len(lines)]):
            assert c.push_sam(b"\n".join(lines[a:b]) + b"\n", first_line=first) == b - a
            first += b - a
        _assert_cols(_cols(c), exp, parts)
        c.close()
    # push_sam after push_bgzf appends: the result is the BAM of both texts
    head = hostile_lines(np.random.RandomState(6), 700) + b"\n"
    p1, p2 = str(tmp_path / "a.bam"), str(tmp_path / "ab.bam")
    encode_bam(p1, head, TARGETS)
    encode_bam(p2, head + text, TARGETS)
    c = _ctx()
    f = api.BgzfFile(p1)
    c.push_bgzf(f)
    c.push_sam(text)
    ref = _ctx()
    g = api.BgzfFile(p2)
    ref.push_bgzf(g)
    _assert_cols(_cols(c), _cols(ref), "append")
    for x in (c, ref, one, f, g):
        x.close()


BAD = [  # (line, what the message names)
    ("r\t0\tchr1\t5\t60\t10M\t*\t0\t0\tAAAAAAAAAA", "fewer than 11"),
    ("", "empty line"),
    ("@SQ\tSN:chr3\tLN:5", "header line"),
    ("y" * 255 + "\t0\tchr1\t5\t60\t*\t*\t0\t0\t*\t*", "QNAME"),
    ("r\t65536\tchr1\t5\t60\t*\t*\t0\t0\t*\t*", "FLAG"),
    ("r\t-1\tchr1\t5\t60\t*\t*\t0\t0\t*\t*", "FLAG"),
    ("r\t0\tchrZ\t5\t60\t*\t*\t0\t0\t*\t*", "RNAME"),
    ("r\t0\tchr1\t2147483648\t60\t*\t*\t0\t0\t*\t*", "POS"),
    ("r\t0\tchr1\t5\t256\t*\t*\t0\t0\t*\t*", "MAPQ"),
    ("r\t0\tchr1\t5\t60\t10Q\t*\t0\t0\t*\t*", "CIGAR"),
    ("r\t0\tchr1\t5\t60\t0M\t*\t0\t0\t*\t*", "CIGAR"),
    ("r\t0\tchr1\t5\t60\t268435456M\t*\t0\t0\t*\t*", "CIGAR"),
    ("r\t0\tchr1\t5\t60\t" + "1M" * 65536 + "\t*\t0\t0\t*\t*", "CIGAR"),
    ("r\t0\tchr1\t5\t60\tM\t*\t0\t0\t*\t*", "CIGAR"),
    ("r\t0\tchr1\t5\t60\t*\tchr9\t0\t0\t*\t*", "RNEXT"),
    ("r\t0\tchr1\t5\t60\t*\t=\tx\t0\t*\t*", "PNEXT"),
    ("r\t0\tchr1\t5\t60\t*\t=\t1\t2147483648\t*\t*", "TLEN"),
    ("r\t0\tchr1\t5\t60\t*\t=\t1\t-2147483649\t*\t*", "TLEN"),
    ("r\t0\tchr1\t5\t60\t*\t=\t1\t0\tAC*G\t*", "SEQ"),
    ("r\t0\tchr1\t5\t60\t*\t=\t1\t0\tAC1G\t*", "SEQ"),
    ("r\t0\tchr1\t5\t60\t*\t=\t1\t0\tACGT\tIII", "QUAL"),
    ("r\t0\tchr1\t5\t60\t*\t=\t1\t0\t*\tI", "QUAL"),
    ("r\t0\tchr1\t5\t60\t5M\t=\t1\t0\tACGT\t*", "CIGAR query length"),
    ("r\t0\tchr1\t5\t60\t*\t=\t1\t0\t*\t*\tXX:Q:1", "optional field"),
    ("r\t0\tchr1\t5\t60\t*\t=\t1\t0\t*\t*\tX:i:1", "optional field"),
    ("r\t0\tchr1\t5\t60\t*\t=\t1\t0\t*\t*\tNM:i:1\t", "optional field"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_kb", [None, 4])
def test_rejections_leave_the_context_unchanged(chunk_kb):
    good = hostile_lines(np.random.RandomState(8), 300) + b"\n"
    glines = good.split(b"\n")[:-1]
    if chunk_kb:
        os.environ["BKID_SAM_CHUNK_KB"] = str(chunk_kb)
    try:
        c = _ctx()
        c.push_sam(good)
        before = _cols(c)
        for j, (bad, what) in enumerate(BAD):
            k = 37 + 9 * j                                      # the failing line's index in the pushed text
            text = b"\n".join(glines[:k] + [bad.encode()] + glines[k:]) + b"\n"
            with pytest.raises(api.BkidError, match=re.escape("SAM line %d: " % (1000 + k)) + ".*" + re.escape(what)):
                c.push_sam(text, first_line=1000)
            _assert_cols(_cols(c), before, bad[:40])
        assert c.push_sam(good) == len(glines)                  # a following valid push works
        after = _cols(c)
        assert np.array_equal(after["pos"], np.concatenate([before["pos"], before["pos"]]))
        c.close()
    finally:
        os.environ.pop("BKID_SAM_CHUNK_KB", None)


def _nibs_set(c, nibs):
    for t, (p, l) in enumerate(nibs):
        c.set_nib(t, p, l)


def _sam_text(path):
    f = api.SamFile(path)
    t = f.text()
    f.close()
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "exclude_q20s15", "validate", "shuffled"])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("data", ["small", "config1"])
def test_calls_equal_oracle(request, tmp_path, data, mode, variant):
    import oracle_py as O
    d, hb, nibs = request.getfixturevalue("small_data" if data == "small" else "config1_data")
    kw = {"qual": 20, "sd_mult": 15} if variant == "exclude_q20s15" else {}
    seq = None
    if variant == "validate":
        genome = [synth.nib_ascii(p, l) for p, l in nibs]
        rng = np.random.RandomState(3)
        hb = api.HostBatch(hb.cols, hb.name_hash, hb.side, hb.target_len, hb.target_names)
        seq, _ = synth.split_read_sequences(hb, genome, corrupt=set(np.nonzero(rng.rand(hb.n_sa) < 0.3)[0].tolist()), seed=9)
        hb.set_seq(seq)
        kw["validate_align"] = 1
    p = str(tmp_path / "reads.sam")
    if variant == "shuffled":
        bamio.write_sam(p, synth.permute(d, np.random.RandomState(7).permutation(hb.n)), sort_order="unsorted")
    else:
        bamio.write_sam(p, d, sa_seq=seq)
    names = list(zip(hb.target_names, hb.target_len))
    iv = np.array([(t, 0, 3) for t in range(len(names))] + [(t, l // 3, l // 3 + 4000) for t, (_, l) in enumerate(names)], np.int64)

    def run(push, sort=False):
        c = _ctx(names, fast=mode, **kw)
        push(c)
        if sort:
            assert c.sort_records() is False
        if variant == "exclude_q20s15":
            c.set_exclude(iv[:, 0], iv[:, 1], iv[:, 2])
        _nibs_set(c, nibs)
        res = c.run()
        got = c.fetch_clusters()
        c.close()
        return res, got

    r1, got = run(lambda c: c.push_sam(_sam_text(p)), sort=variant == "shuffled")
    r2, exp = run(lambda c: c.push(hb))                         # the batch itself: tested against the oracle elsewhere
    assert r1 == r2 and got.tobytes() == exp.tobytes()
    assert len(exp) >= (1 if variant == "exclude_q20s15" else 4)
    if variant in ("plain", "shuffled"):
        m, s, dist, oc = O.run(hb, nibs, mode=mode)
        assert r1[:3] == (m, s, dist) and got.tobytes() == oc.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 5])
def test_sharded_ranges_equal_oracle(tmp_path, small_data, world):
    """rank r pushes the newline-aligned byte range [cut_r, cut_r+1) of a coordinate-sorted SAM"""
    import oracle_py as O
    d, hb, nibs = small_data
    p = str(tmp_path / "reads.sam")
    bamio.write_sam(p, d)
    text = _sam_text(p)
    cuts = [0]
    for r in range(1, world):
        q = max(cuts[-1], len(text) * r // world)
        if q > 0 and text[q - 1:q] != b"\n":
            q = text.index(b"\n", q) + 1
        cuts.append(q)
    cuts.append(len(text))
    names = list(zip(hb.target_names, hb.target_len))
    ctxs = []
    for r in range(world):
        c = _ctx(names)
        c.push_sam(text[cuts[r]:cuts[r + 1]])
        _nibs_set(c, nibs)
        ctxs.append(c)
    res = api.dist_run_local(ctxs, 0)
    m, s, dd, exp = O.run(hb, nibs, mode=0)
    for r, c in enumerate(ctxs):
        assert res[r][:3] == (m, s, dd)
        assert c.fetch_clusters().tobytes() == exp.tobytes(), r
        c.close()


def _driver(inp, out, ps, extra=(), stdin=None):
    return subprocess.run([DRIVER, "-i", inp, "-o", out, "-n", ps["nib"], "-r", ps["refgene"]] + list(extra),
                          timeout=600, capture_output=True, text=stdin is None, input=stdin, env=dict(os.environ))


@pytest.mark.gpu
def test_driver_on_sam(tmp_path, small_data):
    import reference_calls as R
    d, hb, nibs = small_data
    ps = bamio.write_dataset(str(tmp_path / "s"), d, sam=True)
    pg = bamio.write_dataset(str(tmp_path / "g"), synth.permute(d, np.argsort(d.cols["name_id"].cpu().numpy(), kind="stable")),
                             sort_order="queryname", sam=True)
    base = str(tmp_path / "s")

    def files(prefix, flags, inp):
        fs = ("_fusion.txt", "_params.txt") + (("_fusion_all.txt",) if "-all" in flags else ())
        return {k: open(prefix + k).read().replace("inp_file\t" + inp + "\n", "inp_file\tIN\n").replace("out_file\t" + prefix + "\n", "out_file\tOUT\n")
                for k in fs}

    def decoder(prefix):
        return dict(ln.split("\t") for ln in open(prefix + "_b200_timings.txt").read().splitlines())

    # SAM first: no .bai exists yet
    got = {}
    for flags in ([], ["-fast"], ["-all"]):
        o = base + "/sam" + "".join(flags)
        g = _driver(ps["sam"], o, ps, flags)
        assert g.returncode == 0, g.stderr[-500:]
        got[o] = (tuple(flags), files(o, flags, ps["sam"]))
    for o, inp, pp, extra, stdin in ((str(tmp_path / "g" / "sorted"), pg["sam"], pg, ["-sort"], None),
                                     (base + "/stdin", "-", ps, ["-sort"], open(ps["sam"], "rb").read()),
                                     (base + "/multi", ps["sam"], ps, ["-gpu", "0,0,0"], None)):
        g = _driver(inp, o, pp, extra + ["-all"], stdin=stdin)
        assert g.returncode == 0, g.stderr[-500:]
        got[o] = (("-all",), files(o, ["-all"], inp))
    assert not os.path.exists(ps["bam"] + ".bai")
    for o in got:
        tm = decoder(o)
        assert tm["decoder"] == "sam" and int(tm["records"]) == hb.n, o
    # the BAM of the same records
    R.index(ps["bam"])
    want = {}
    for flags in ([], ["-fast"], ["-all"]):
        o = base + "/ref" + "".join(flags)
        g = _driver(ps["bam"], o, ps, flags)
        assert g.returncode == 0, g.stderr[-500:]
        want[tuple(flags)] = files(o, flags, ps["bam"])
    R.match_oracle(base + "/ref-all", d)
    for o, (flags, fs) in got.items():
        assert fs == want[flags], o
