"""BAM on a pipe (bkid_push_bgzf_stream, BreakID -i - / -i <fifo>): a BGZF stream decoded on the device piece by piece.

The expected result is defined by construction: for any cut of the stream into pieces, the context ends in exactly the
state bkid_push_bgzf leaves for the same bytes held as a file.  The CPU tests pin the host block walker to
bkid_host_bgzf_open's table under every kind of cut and the prefix header parser to the file parser; the GPU tests
compare every column with push_bgzf, the calls with the oracle and the driver's files with the run on the file."""
import gzip
import os
import struct
import subprocess
import threading

import numpy as np
import pytest

from breakid_b200 import api, bamio, synth
from test_bgzf_decode import _bgzf_write, _hostile_records, _raw_bam, _record, _write_hostile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "breakid_b200", "host", "BreakID")
DENSE = (("flag", np.uint16), ("mapq", np.uint8), ("tid", np.int32), ("pos", np.int32), ("isize", np.int32), ("endpos", np.int32))
ALL = DENSE + api._XCOLS + api._SIDE + api._SEQ
TARGETS = [("chr1", 500000), ("chr2", 400000)]


def _block_starts(raw):
    """(start, end) of every BGZF block of a whole file, from its own BSIZE fields"""
    out, o = [], 0
    while o < len(raw):
        xlen = struct.unpack_from("<H", raw, o + 10)[0]
        x, bsize = 0, 0
        while x + 4 <= xlen:
            si1, si2, slen = raw[o + 12 + x], raw[o + 13 + x], struct.unpack_from("<H", raw, o + 14 + x)[0]
            if (si1, si2) == (66, 67):
                bsize = struct.unpack_from("<H", raw, o + 16 + x)[0] + 1
            x += 4 + slen
        out.append((o, o + bsize))
        o += bsize
    return out


def _walk_in_pieces(raw, cuts):
    """feed raw to the walker as a pipe would deliver it (cut at `cuts`): the stream's block table, offsets made absolute"""
    table, buf, base = [], b"", 0
    for a, b in zip([0] + list(cuts), list(cuts) + [len(raw)]):
        buf += raw[a:b]
        tb, used = api.bgzf_walk(buf)
        tb["payload_off"] += np.uint64(base)
        table.append(tb)
        buf, base = buf[used:], base + used
    assert buf == b"" and base == len(raw)
    return np.concatenate(table)


def _cut_kinds(raw, rng):
    blk = _block_starts(raw)
    k = [s + int(rng.randint(1, 18)) for s, _ in blk[1::7]]                          # inside the 18-byte header
    x = [s + 12 + int(rng.randint(1, 6)) for s, _ in blk[2::7]]                      # inside XLEN's subfields
    p = [s + 18 + int(rng.randint(0, max(1, e - s - 26))) for s, e in blk[3::7]]    # inside the payload
    t = [e - int(rng.randint(1, 9)) for _, e in blk[4::7]]                           # inside CRC32 / ISIZE
    e = [e for _, e in blk[:-1]]                                                     # exactly on block ends
    r = sorted(set(int(v) for v in rng.randint(1, len(raw), 60)))                    # random
    return {"header": k, "xlen": x, "payload": p, "trailer": t, "block_end": e, "random": r}


# ------------------------------------------------------------------------------------------------ CPU
def test_walker_equals_open_under_every_cut(tmp_path):
    p, payload, first = _write_hostile(tmp_path)
    raw = open(p, "rb").read()
    f = api.BgzfFile(p)
    want = f.block_table()
    f.close()
    whole, used = api.bgzf_walk(raw)
    assert used == len(raw) and np.array_equal(whole, want)
    for kind, cuts in _cut_kinds(raw, np.random.RandomState(1)).items():
        assert len(cuts) > 3, kind
        assert np.array_equal(_walk_in_pieces(raw, sorted(set(cuts))), want), kind
        for c in cuts[:20]:                                # each cut alone: the blocks before it, the partial one left
            tb, used = api.bgzf_walk(raw[:c])
            ends = (want["payload_off"] + want["payload_len"] + 8).astype(np.int64)
            n = int((ends <= c).sum())
            assert np.array_equal(tb, want[:n]) and used == (int(ends[n - 1]) if n else 0), (kind, c)


def test_walker_rejects_garbage_and_plain_gzip(tmp_path):
    p, _, _ = _write_hostile(tmp_path, n=2000)
    raw = open(p, "rb").read()
    blk = _block_starts(raw)
    with pytest.raises(IOError, match="not a BGZF"):
        api.bgzf_walk(b"this is not a BAM at all" * 4)
    with pytest.raises(IOError, match="plain gzip"):
        api.bgzf_walk(gzip.compress(b"hello world" * 100))
    s = blk[3][0]
    with pytest.raises(IOError):                            # garbage between two blocks
        api.bgzf_walk(raw[:s] + b"\0garbage\0" * 3 + raw[s:])
    bad = bytearray(raw)                                    # the BC subfield renamed
    bad[blk[2][0] + 12] = ord("X")
    with pytest.raises(IOError, match="BC"):
        api.bgzf_walk(bytes(bad))
    assert api.bgzf_walk(b"")[1] == 0 and api.bgzf_walk(raw[:17])[1] == 0          # too short to judge: wait for more


def _many_sq_bam(tmp_path, n_sq=3366, n_rec=200, block=4096):
    targets = [("contig_%05d_%s" % (i, "q" * (i % 37)), 1000 + i) for i in range(n_sq)]
    recs = [_record(i % n_sq, 10 + i, "r%d" % i, 99, 60, [(50, 0)], 50, i % n_sq, 400, 300, b"NMC\x01") for i in range(n_rec)]
    payload, first = _raw_bam(recs, targets)
    p = str(tmp_path / "many_sq.bam")
    _bgzf_write(p, payload, block=block)
    return p, targets, first


def test_prefix_header_parse_needs_more_until_complete(tmp_path):
    p, targets, first = _many_sq_bam(tmp_path)
    raw = open(p, "rb").read()
    f = api.BgzfFile(p)
    table = f.block_table()
    assert f.first_record == first and f.target_names == [n for n, _ in targets]
    f.close()
    ustart = np.concatenate([[0], np.cumsum(table["usize"].astype(np.int64))])
    need = int(np.searchsorted(ustart, first, side="left"))  # blocks that hold the header
    assert need > 20
    for k in list(range(0, need)) + [need, need + 1, len(table)]:
        end = int(table["payload_off"][k - 1] + table["payload_len"][k - 1] + 8) if k else 0
        tb, used = api.bgzf_walk(raw[:end + 5])
        assert used == end and len(tb) == k
        got = api.bgzf_parse_header(raw[:end + 5], tb)
        if k < need:
            assert got is None, k
        else:
            names, lens, fr = got
            assert fr == first and names == [n for n, _ in targets] and lens == [l for _, l in targets], k
    with pytest.raises(IOError, match="not a BAM"):
        blk = bamio._bgzf_block(b"SAM?" + bytes(40), 6)
        api.bgzf_parse_header(blk, api.bgzf_walk(blk)[0])


def _run(args, **kw):
    return subprocess.run([DRIVER] + args, capture_output=True, timeout=120, **kw)


def test_driver_refusals_before_any_device(tmp_path):
    p, _, _ = _write_hostile(tmp_path, n=300)
    raw = open(p, "rb").read()
    o, nib = str(tmp_path / "o"), str(tmp_path)
    r = _run(["-i", "-", "-gpu", "0,1", "-o", o, "-n", nib], input=raw)
    assert r.returncode == 1 and b"stdin needs one GPU" in r.stderr
    r = _run(["-i", "-", "-o", o, "-n", nib], input=raw, env=dict(os.environ, BKID_HOST_DECODE="1"))
    assert r.returncode == 1 and b"host decode" in r.stderr
    r = _run(["-i", "-", "-o", o, "-n", nib], input=gzip.compress(b"@HD\tVN:1.6\n" * 50))
    assert r.returncode == 1 and b"can not read bam-file: - (" in r.stderr
    fifo = str(tmp_path / "in.fifo")
    os.mkfifo(fifo)                                          # nobody writes it: the refusal must come before the open
    r = _run(["-i", fifo, "-gpu", "0,1", "-o", o, "-n", nib])
    assert r.returncode == 1 and b"needs one GPU" in r.stderr
    assert b"- for stdin" in _run(["-h"]).stderr


# ------------------------------------------------------------------------------------------------ GPU
def _ctx(names=TARGETS, **kw):
    return api.Context([l for _, l in names], [n for n, _ in names], device=0, **kw)


def _cols(c):
    return {k: c.fetch_column(k, dt) for k, dt in ALL}


def _assert_cols(got, exp, what=""):
    assert sorted(got) == sorted(exp)
    for k in exp:
        assert np.array_equal(got[k], exp[k]), (what, k)


def _stream(c, raw, cuts, first, end=True):
    """push raw to c as the driver does when the pipe delivers it cut at `cuts`: every whole block read so far"""
    c.bgzf_stream_begin(first)
    buf, n = b"", 0
    for a, b in zip([0] + list(cuts), list(cuts) + [len(raw)]):
        buf += raw[a:b]
        tb, used = api.bgzf_walk(buf)
        if len(tb):
            n += c.push_bgzf_stream(buf[:used], tb)
        buf = buf[used:]
    if end:
        assert buf == b""
        assert c.bgzf_stream_end() == n
    return n


def _file_cols(p, names=TARGETS):
    f = api.BgzfFile(p)
    c = _ctx(names)
    n = c.push_bgzf(f)
    cols = _cols(c)
    c.close(); f.close()
    return n, cols


def _with_chunk(chunk_kb, fn):
    if chunk_kb:
        os.environ["BKID_BGZF_CHUNK_KB"] = str(chunk_kb)
    try:
        return fn()
    finally:
        os.environ.pop("BKID_BGZF_CHUNK_KB", None)


def _big_record_bam(tmp_path, rng):
    """a 700 KB record (spans many blocks and is longer than most pieces) among hostile ones, behind a 120 KB header"""
    recs = _hostile_records(rng, 1500)
    big = _record(0, 60000, "bigrec", 99, 60, [(50, 0)], 0, 0, 61000, 300, b"XBBc" + struct.pack("<i", 700000) + bytes(range(256)) * 2734 + bytes(96))
    text = "@HD\tVN:1.4\tSO:coordinate\n" + "".join("@CO\t%s\n" % ("h" * 90) for _ in range(1300)) + "".join("@SQ\tSN:%s\tLN:%d\n" % t for t in TARGETS)
    out = b"BAM\x01" + struct.pack("<i", len(text)) + text.encode() + struct.pack("<i", len(TARGETS))
    for nm, ln in TARGETS:
        out += struct.pack("<i", len(nm) + 1) + nm.encode() + b"\0" + struct.pack("<i", ln)
    first = len(out)
    for r in recs[:700] + [big] + recs[700:]:
        out += struct.pack("<i", len(r)) + r
    p = str(tmp_path / "big.bam")
    _bgzf_write(p, out, vary=True)
    return p, first


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_kb", [None, 64])
def test_stream_equals_push_bgzf_under_every_cut(tmp_path, chunk_kb):
    p, payload, first = _write_hostile(tmp_path, n=6000)
    raw = open(p, "rb").read()
    n_file, exp = _file_cols(p)
    blk = _block_starts(raw)
    rng = np.random.RandomState(2)
    cases = dict(_cut_kinds(raw, rng))
    cases["one_block_per_piece"] = [e for _, e in blk[:-1]]
    cases["inside_header"] = [9, 40, 300, first // 2]       # the BAM header arrives over several pieces
    pb, first_b = _big_record_bam(tmp_path, np.random.RandomState(4))
    raw_b = open(pb, "rb").read()
    n_b, exp_b = _file_cols(pb)
    for kind, cuts in cases.items():
        c = _ctx()
        n = _with_chunk(chunk_kb, lambda: _stream(c, raw, sorted(set(cuts)), first))
        assert n == n_file
        _assert_cols(_cols(c), exp, (kind, chunk_kb))
        st = c.decode_stats()                                # accumulated over the session
        assert st["n_records"] == n_file and st["uncompressed_bytes"] == len(payload), kind
        c.close()
    # a BAM header of 300 @SQ lines in blocks of 512 bytes, one block (or a few) per piece: the header skip carries over
    pm, tm, first_m = _many_sq_bam(tmp_path, n_sq=300, n_rec=400, block=512)
    raw_m = open(pm, "rb").read()
    n_m, exp_m = _file_cols(pm, tm)
    blk_m = _block_starts(raw_m)
    assert first_m > 10 * 512
    for cuts in ([e for _, e in blk_m[:-1]], [e for _, e in blk_m[2:-1:3]]):
        c = _ctx(tm)
        assert _with_chunk(chunk_kb, lambda: _stream(c, raw_m, cuts, first_m)) == n_m == 400
        _assert_cols(_cols(c), exp_m, ("many @SQ", chunk_kb))
        c.close()
    # a record over many blocks, pieces of 100 KB (shorter than the record)
    for cuts in (list(range(50000, len(raw_b), 100000)), sorted(set(int(v) for v in np.random.RandomState(7).randint(1, len(raw_b), 40)))):
        c = _ctx()
        assert _with_chunk(chunk_kb, lambda: _stream(c, raw_b, cuts, first_b)) == n_b == 1502
        _assert_cols(_cols(c), exp_b, ("big", chunk_kb))
        c.close()


@pytest.mark.gpu
def test_stored_blocks_empty_blocks_and_no_records(tmp_path):
    rng = np.random.RandomState(5)
    payload, first = _raw_bam(_hostile_records(rng, 2500), TARGETS)
    # level 0 (stored blocks), as samtools view -u writes them
    p0 = str(tmp_path / "stored.bam")
    _bgzf_write(p0, payload, level=0)
    raw0 = open(p0, "rb").read()
    n, exp = _file_cols(p0)
    c = _ctx()
    assert _stream(c, raw0, list(range(70000, len(raw0), 150001)), first) == n
    _assert_cols(_cols(c), exp, "stored")
    c.close()
    # empty blocks in the middle of the stream, with and without the EOF marker at the end
    blocks = [bamio._bgzf_block(payload[o:o + 30000], 6) for o in range(0, len(payload), 30000)]
    for eof in (True, False):
        raw = b"".join(b + (bamio._BGZF_EOF if i % 3 == 1 else b"") for i, b in enumerate(blocks)) + (bamio._BGZF_EOF if eof else b"")
        pe = str(tmp_path / "empty_blocks.bam")
        open(pe, "wb").write(raw)
        n, exp = _file_cols(pe)
        c = _ctx()
        assert _stream(c, raw, [e for _, e in _block_starts(raw)[:-1]], first) == n
        _assert_cols(_cols(c), exp, ("empty blocks", eof))
        c.close()
    # no records at all
    hp, hfirst = _raw_bam([], TARGETS)
    ph = str(tmp_path / "header_only.bam")
    _bgzf_write(ph, hp, block=100)
    rawh = open(ph, "rb").read()
    c = _ctx()
    assert _stream(c, rawh, [50, 150], hfirst) == 0
    assert c.fetch_column("flag", np.uint16).shape[0] == 0
    c.close()


@pytest.mark.gpu
def test_stream_after_push_batch_two_streams_and_sort(tmp_path, small_data):
    d, hb, nibs = small_data
    names = list(zip(hb.target_names, hb.target_len))
    p = str(tmp_path / "reads.bam")
    bamio.write_bam(p, d)
    raw = open(p, "rb").read()
    f = api.BgzfFile(p)
    first = f.first_record
    cuts = list(range(1 << 20, len(raw), 1 << 20))
    # after push_batch (with the read bases of its SA records, so that every seq column is defined), two streams in a row
    genome = [synth.nib_ascii(pl, l) for pl, l in nibs]
    hbs = api.HostBatch(hb.cols, hb.name_hash, hb.side, hb.target_len, hb.target_names)
    hbs.set_seq(synth.split_read_sequences(hbs, genome)[0])
    ref, c = _ctx(names), _ctx(names)
    ref.push(hbs); ref.push_bgzf(f); ref.push_bgzf(f)
    c.push(hbs)
    _stream(c, raw, cuts, first)
    _stream(c, raw, cuts[1:], first)
    _assert_cols(_cols(c), _cols(ref), "after push_batch + 2 streams")
    ref.close(); c.close(); f.close()
    # a shuffled BAM: stream + sort == push_bgzf + sort
    ps = str(tmp_path / "shuffled.bam")
    bamio.write_bam(ps, synth.permute(d, np.random.RandomState(3).permutation(hb.n)), sort_order="unsorted")
    raw = open(ps, "rb").read()
    g = api.BgzfFile(ps)
    ref, c = _ctx(names), _ctx(names)
    ref.push_bgzf(g)
    assert ref.sort_records() is False
    _stream(c, raw, list(range(300000, len(raw), 700000)), g.first_record)
    assert c.sort_records() is False
    _assert_cols(_cols(c), _cols(ref), "sorted")
    ref.close(); c.close(); g.close()


def _counts(c):
    return {k: c.fetch_column(k, dt).shape[0] for k, dt in ALL}


@pytest.mark.gpu
def test_rejections_restore_the_context_at_begin(tmp_path):
    p, payload, first = _write_hostile(tmp_path, n=5000)
    raw = open(p, "rb").read()
    blk = _block_starts(raw)
    f = api.BgzfFile(p)
    table = f.block_table()
    f.close()
    ustart = np.concatenate([[0], np.cumsum(table["usize"].astype(np.int64))])
    rec_starts, o = set(), first
    while o < len(payload):
        rec_starts.add(o)
        o += 4 + struct.unpack_from("<i", payload, o)[0]
    n_file, exp = _file_cols(p)
    c = _ctx()
    _stream(c, raw, [len(raw) // 2], first)                  # the state at begin: one stream already decoded
    before = _cols(c)
    assert _counts(c)["flag"] == n_file

    def rejected(fn, match):
        with pytest.raises(api.BkidError, match=match):
            fn()
        _assert_cols(_cols(c), before, match)

    # truncation: the stream stops inside a block header, a payload or a trailer (the walker leaves that block), or
    # right after a block whose end is not a record end; in each case a record is still carried at end
    for k, where in ((len(blk) * 2 // 3, lambda s, e: s + 9), (len(blk) // 2, lambda s, e: s + 40), (len(blk) // 3, lambda s, e: e - 3),
                     (len(blk) // 4, lambda s, e: e)):
        s, e = blk[k]
        assert int(ustart[k + 1] if where(s, e) == e else ustart[k]) not in rec_starts
        cut = where(s, e)
        rejected(lambda: (_stream(c, raw[:cut], list(range(100000, cut, 100000)), first, end=False), c.bgzf_stream_end()),
                 "truncated BAM record")
    # a CRC error in a late piece, after earlier pieces appended records: the block is named by its stream index
    k = len(blk) - 5
    bad = bytearray(raw)
    bad[int(table["payload_off"][k] + table["payload_len"][k])] ^= 0x20
    cuts = [blk[10][1], blk[len(blk) // 2][1], blk[k - 2][1]]

    def crc():
        c.bgzf_stream_begin(first)
        buf = bytes(bad)
        appended = 0
        for a, b in zip([0] + cuts, cuts + [len(buf)]):
            tb, used = api.bgzf_walk(buf[a:b])
            appended += c.push_bgzf_stream(buf[a:a + used], tb)
            assert appended > 0
    rejected(crc, "CRC32 mismatch in BGZF block %d" % k)
    # a block table that lies outside its piece; a corrupt record (block_size < 32)
    tb, used = api.bgzf_walk(raw)

    def outside():
        c.bgzf_stream_begin(first)
        t = tb.copy()
        t["payload_off"][7] += np.uint64(len(raw))
        c.push_bgzf_stream(raw, t)
    rejected(outside, "corrupt BGZF block table")
    bad_payload = bytearray(payload)
    struct.pack_into("<i", bad_payload, sorted(rec_starts)[2000], 12)
    pb = str(tmp_path / "bad_record.bam")
    _bgzf_write(pb, bytes(bad_payload), vary=True)
    rawb = open(pb, "rb").read()
    rejected(lambda: _stream(c, rawb, [len(rawb) // 3, len(rawb) * 2 // 3], first), "corrupt BAM record")
    # call order
    rejected(lambda: c.push_bgzf_stream(raw), "without bkid_bgzf_stream_begin")
    rejected(lambda: c.bgzf_stream_end(), "without bkid_bgzf_stream_begin")
    c.bgzf_stream_begin(first)
    c.push_bgzf_stream(raw[:blk[40][1]])
    g = api.BgzfFile(p)
    for other in (lambda: c.bgzf_stream_begin(first), lambda: c.push_bgzf(g), lambda: c.push_sam(b""), lambda: c.sort_records(),
                  lambda: c.insert_stats(), lambda: c.run(), lambda: c.push(api.HostBatch.from_bam(p))):
        with pytest.raises(api.BkidError, match="stream session is open"):
            other()
    c.reset()                                                # closes the session
    assert _counts(c)["flag"] == 0
    # after the rejections a fresh stream decodes correctly
    _stream(c, raw, [len(raw) // 3], first)
    _assert_cols(_cols(c), exp, "after rejections")
    c.close()
    # begin on a context that holds borrowed device columns
    from test_sort_records import _device_batch
    keep = []
    b = _device_batch(api.HostBatch.from_bam(p), keep)
    c = _ctx()
    c.push_device(b)
    with pytest.raises(api.BkidError, match="borrowed"):
        c.bgzf_stream_begin(first)
    c.close()
    g.close()


def _nibs_set(c, nibs):
    for t, (pl, l) in enumerate(nibs):
        c.set_nib(t, pl, l)


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
        genome = [synth.nib_ascii(pl, l) for pl, l in nibs]
        rng = np.random.RandomState(3)
        hb = api.HostBatch(hb.cols, hb.name_hash, hb.side, hb.target_len, hb.target_names)
        seq, _ = synth.split_read_sequences(hb, genome, corrupt=set(np.nonzero(rng.rand(hb.n_sa) < 0.3)[0].tolist()), seed=9)
        hb.set_seq(seq)
        kw["validate_align"] = 1
    p = str(tmp_path / "reads.bam")
    if variant == "shuffled":
        bamio.write_bam(p, synth.permute(d, np.random.RandomState(7).permutation(hb.n)), sort_order="unsorted")
    else:
        bamio.write_bam(p, d, sa_seq=seq)
    raw = open(p, "rb").read()
    f = api.BgzfFile(p)
    first = f.first_record
    f.close()
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

    cuts = sorted(set(int(v) for v in np.random.RandomState(11).randint(1, len(raw), 9)))
    r1, got = run(lambda c: _stream(c, raw, cuts, first), sort=variant == "shuffled")
    r2, exp = run(lambda c: c.push(hb))
    assert r1 == r2 and got.tobytes() == exp.tobytes()
    assert len(exp) >= (1 if variant == "exclude_q20s15" else 4)
    if variant in ("plain", "shuffled"):
        m, s, dist, oc = O.run(hb, nibs, mode=mode)
        assert r1[:3] == (m, s, dist) and got.tobytes() == oc.tobytes()


def _driver(inp, out, ps, extra=(), stdin=None, env=None):
    return subprocess.run([DRIVER, "-i", inp, "-o", out, "-n", ps["nib"], "-r", ps["refgene"]] + list(extra),
                          timeout=600, capture_output=True, input=stdin, env=dict(os.environ, **(env or {})))


def _files(prefix, flags, inp):
    fs = ("_fusion.txt", "_params.txt") + (("_fusion_all.txt",) if "-all" in flags else ())
    return {k: open(prefix + k).read().replace("inp_file\t" + inp + "\n", "inp_file\tIN\n").replace("out_file\t" + prefix + "\n", "out_file\tOUT\n")
            for k in fs}


def _timings(prefix):
    return dict(ln.split("\t") for ln in open(prefix + "_b200_timings.txt").read().splitlines())


def _via_fifo(path_in, fifo, run):
    """run(fifo) while a thread writes path_in's bytes into the FIFO"""
    os.mkfifo(fifo)
    data = open(path_in, "rb").read()

    def feed():
        with open(fifo, "wb") as w:
            w.write(data)
    t = threading.Thread(target=feed)
    t.start()
    try:
        return run(fifo)
    finally:
        t.join(timeout=600)


@pytest.mark.gpu
def test_driver_on_a_stream(tmp_path, small_data):
    import reference_calls as R
    d, hb, nibs = small_data
    ps = bamio.write_dataset(str(tmp_path / "s"), d, sam=True)
    pg = bamio.write_dataset(str(tmp_path / "g"), synth.permute(d, np.argsort(d.cols["name_id"].cpu().numpy(), kind="stable")),
                             sort_order="queryname")
    base = str(tmp_path / "s")
    raw = open(ps["bam"], "rb").read()
    stored = base + "/stored.bam"                            # the same bytes uncompressed, as samtools view -u writes them
    _bgzf_write(stored, gzip.decompress(raw), level=0)
    got = {}
    for flags, env in (([], {}), (["-fast"], {}), (["-all"], {"BKID_STREAM_PIECE_KB": "64"})):
        o = base + "/pipe" + "".join(flags)
        g = _driver("-", o, ps, flags, stdin=raw, env=env)
        assert g.returncode == 0, g.stderr[-800:]
        got[o] = (tuple(flags), _files(o, flags, "-"))
        tm = _timings(o)
        assert tm["decoder"] == "device" and tm["stream"] == "1" and int(tm["records"]) == hb.n
        assert int(tm["pieces"]) > (1 if env else 0)
    o = base + "/stored"
    g = _driver("-", o, ps, ["-all"], stdin=open(stored, "rb").read())
    assert g.returncode == 0, g.stderr[-800:]
    got[o] = (("-all",), _files(o, ["-all"], "-"))
    o = str(tmp_path / "g" / "sorted")
    g = _driver("-", o, pg, ["-sort", "-all"], stdin=open(pg["bam"], "rb").read())
    assert g.returncode == 0, g.stderr[-800:]
    got[o] = (("-all",), _files(o, ["-all"], "-"))
    for kind in ("bam", "sam"):
        fifo = base + "/in_%s.fifo" % kind
        o = base + "/fifo_" + kind
        g = _via_fifo(ps[kind], fifo, lambda q: _driver(q, o, ps, ["-all"]))
        assert g.returncode == 0, g.stderr[-800:]
        got[o] = (("-all",), _files(o, ["-all"], fifo))
        assert _timings(o)["decoder"] == ("device" if kind == "bam" else "sam")
    assert not os.path.exists(ps["bam"] + ".bai")            # no index is needed for a stream
    # a truncated stream exits 1 and writes no call file
    o = base + "/trunc"
    g = _driver("-", o, ps, [], stdin=raw[:len(raw) * 2 // 3])
    assert g.returncode == 1 and b"can not read bam-file: - (" in g.stderr and not os.path.exists(o + "_fusion.txt")
    # the run on the file
    R.index(ps["bam"])
    want = {}
    for flags in ([], ["-fast"], ["-all"]):
        o = base + "/ref" + "".join(flags)
        g = _driver(ps["bam"], o, ps, flags)
        assert g.returncode == 0, g.stderr[-800:]
        want[tuple(flags)] = _files(o, flags, ps["bam"])
    R.match_oracle(base + "/ref-all", d)
    for o, (flags, fs) in got.items():
        assert fs == want[flags], o
