"""bkid_sort_records / BreakID -sort: unsorted input is coordinate sorted on the device.

The expected result of every GPU test is the batch sorted on the host with numpy (a stable sort by
(tid as uint32, pos + 1, reverse strand)) and pushed directly; columns and calls are compared byte for byte, and the calls
on the host-sorted batch against the CPU oracle.  The CPU tests pin the key to the samtools 1.3.1 expression and check the
test helpers that write unsorted input (synth.permute, bamio.write_bam(sort_order=...))."""
import os
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "breakid_b200", "host", "BreakID")
COLS = (("flag", np.uint16), ("mapq", np.uint8), ("tid", np.int32), ("pos", np.int32), ("isize", np.int32), ("endpos", np.int32),
        ("x_rec", np.uint32), ("x_mtid", np.int32), ("x_mpos", np.int32), ("x_name_hash", np.uint64),
        ("sa_rec", np.uint32), ("cig_off", np.uint32), ("cig_ops", np.uint32), ("sa_off", np.uint32), ("sa_txt", np.uint8),
        ("oc_off", np.uint32), ("oc_txt", np.uint8))
SEQ_COLS = (("seq_off", np.uint32), ("seq4", np.uint8), ("seq_len", np.int32))


# ------------------------------------------------------------------------------------------------ host-side helpers
def coordinate_order(tid, pos, flag):
    """stable order by the lexicographic key (tid as uint32, pos + 1, flag & 0x10)"""
    return np.lexsort(((np.asarray(flag).astype(np.int64) >> 4) & 1, np.asarray(pos, np.int64) + 1, np.asarray(tid).astype(np.uint32)))


def samtools_key(tid, pos, flag):
    """the literal key of samtools 1.3.1 bam_sort.c: (uint64_t)tid << 32 | (pos + 1) << 1 | bam_is_rev"""
    t = np.asarray(tid).astype(np.uint32).astype(np.uint64)
    p = (np.asarray(pos, np.int64) + 1).astype(np.uint64)
    r = ((np.asarray(flag).astype(np.uint64) >> np.uint64(4)) & np.uint64(1))
    return (t << np.uint64(32)) | (p << np.uint64(1)) | r


def _segs(off, data, rows):
    off = off.astype(np.int64)
    parts = [data[off[k]:off[k + 1]] for k in rows]
    new_off = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.uint32)
    return new_off, (np.concatenate(parts).astype(data.dtype) if parts else data[:0].copy())


def permute_hb(hb, order):
    """HostBatch of the same records in file order `order` (new record i = old record order[i]); side tables and the
    optional seq table re-laid out in ascending new record index"""
    from breakid_b200 import api
    order = np.asarray(order, np.int64)
    new_of = np.empty_like(order); new_of[order] = np.arange(order.shape[0])
    cols = {k: v[order] for k, v in hb.cols.items()}
    nh = hb.name_hash.reshape(-1, 2)[order].reshape(-1)
    sa_new = new_of[hb.side["sa_rec"].astype(np.int64)]
    rows = np.argsort(sa_new, kind="stable")
    side = {"sa_rec": sa_new[rows].astype(np.uint32)}
    for o, d in (("cig_off", "cig_ops"), ("sa_off", "sa_txt"), ("oc_off", "oc_txt")):
        side[o], side[d] = _segs(hb.side[o], hb.side[d], rows)
    if hb.seq is not None:
        side["seq_off"], side["seq4"] = _segs(hb.seq["seq_off"], hb.seq["seq4"], rows)
        side["seq_len"] = hb.seq["seq_len"][rows]
    return api.HostBatch(cols, nh, side, hb.target_len, hb.target_names)


def host_sorted(hb):
    return permute_hb(hb, coordinate_order(hb.cols["tid"], hb.cols["pos"], hb.cols["flag"]))


def input_orders(d, hb, seed=1):
    """the five input orders of the tests: (name, order, already sorted)"""
    rng = np.random.RandomState(seed)
    n = hb.n
    rev = (hb.cols["flag"].astype(np.int64) >> 4) & 1
    name_id = d.cols["name_id"].cpu().numpy()
    return [("random", rng.permutation(n), False),
            ("name_grouped", np.argsort(name_id, kind="stable"), False),
            ("reversed", np.arange(n)[::-1].copy(), False),
            ("sorted", np.arange(n), True),
            ("sorted_rev_first", np.lexsort((1 - rev, hb.cols["pos"], hb.cols["tid"].astype(np.uint32))), True)]


# ------------------------------------------------------------------------------------------------ CPU
def test_lexicographic_key_equals_samtools_key():
    rng = np.random.RandomState(4)
    n = 20000
    tid = rng.randint(-1, 5, n).astype(np.int32)
    pos = rng.randint(-1, 300, n).astype(np.int32)
    pos[tid < 0] = -1                                          # the unmapped tail
    flag = (rng.randint(0, 2, n) * 0x10 | 0x1).astype(np.uint16)
    pl = rng.rand(n) < 0.1                                     # placed-unmapped mates: same tid / pos as their mate, 0x4
    flag[pl] |= 0x4
    pos[:50] = 0; pos[50:100] = -1
    for t, p in ((0, 0), (0, -1), (-1, -1)):
        m = (tid == t) & (pos == p)
        assert (m & ((flag & 0x10) != 0)).any() and (m & ((flag & 0x10) == 0)).any()
    key = samtools_key(tid, pos, flag)
    o1 = coordinate_order(tid, pos, flag)
    o2 = np.argsort(key, kind="stable")
    assert np.array_equal(o1, o2)
    # the order a check of "already sorted" accepts is (tid as uint32, pos); the tail stays last
    s = o1
    assert (tid[s][-int((tid < 0).sum()):] == -1).all()


def test_permute_roundtrip_is_exact(small_data):
    from breakid_b200 import synth
    d, hb, nibs = small_data
    for name, order, _ in input_orders(d, hb):
        p = synth.permute(d, order)
        inv = np.empty_like(order); inv[order] = np.arange(order.shape[0])
        back = synth.permute(p, inv)
        for k in d.cols:
            assert torch.equal(back.cols[k], d.cols[k]), (name, k)
        for k in ("sa_rec", "cig_off", "cig_ops", "sa_off", "sa_txt"):
            assert torch.equal(getattr(back, k), getattr(d, k)), (name, k)
        assert torch.equal(p.cols["pos"], d.cols["pos"][torch.from_numpy(order)])
        assert bool((p.sa_rec[1:] > p.sa_rec[:-1]).all())


def test_host_decoder_reads_name_grouped_bam(tmp_path, small_data):
    from breakid_b200 import api, bamio, synth
    d, hb, nibs = small_data
    order = np.argsort(d.cols["name_id"].cpu().numpy(), kind="stable")
    p = synth.permute(d, order)
    bam = str(tmp_path / "reads.bam")
    bamio.write_bam(bam, p, sort_order="queryname")
    b = api.HostBatch.from_bam(bam, 4)
    a = permute_hb(hb, order)
    assert a.n == b.n and a.n_sa == b.n_sa and a.n_x == b.n_x
    for k in a.cols:
        assert np.array_equal(a.cols[k], b.cols[k]), k
    for k in a.x:
        assert np.array_equal(a.x[k], b.x[k]), k
    for k in a.side:
        assert np.array_equal(a.side[k], b.side[k]), k
    with open(bam, "rb") as f:
        import gzip
        assert b"SO:queryname" in gzip.GzipFile(fileobj=f).read(4096)


def test_driver_sort_refuses_several_gpus(tmp_path):
    r = subprocess.run([DRIVER, "-sort", "-gpu", "0,1", "-i", str(tmp_path / "x.bam"), "-o", str(tmp_path / "o"), "-n", str(tmp_path)],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 1
    assert "-sort works on one GPU only" in r.stderr
    h = subprocess.run([DRIVER, "-h"], capture_output=True, text=True, timeout=60)
    assert "-sort" in h.stderr


# ------------------------------------------------------------------------------------------------ GPU
def _ctx(hb, **kw):
    from breakid_b200 import api
    return api.Context(hb.target_len, hb.target_names, device=0, **kw)


def _columns(c, seq=False):
    return {k: c.fetch_column(k, dt) for k, dt in COLS + (SEQ_COLS if seq else ())}


def _push(c, hb, how):
    from test_multi_gloo import _slice
    if how == "three":
        t = hb.cols["tid"]
        same = np.nonzero(t[1:] == t[:-1])[0] + 1            # cuts inside a tid run
        cut = [0, int(same[len(same) // 3]), int(same[2 * len(same) // 3]), hb.n]
        for a, b in zip(cut[:-1], cut[1:]):
            c.push(_slice(hb, a, b))
    else:
        c.push(hb, narrow=(how == "narrow"))


def _assert_columns(got, exp):
    for k in exp:
        assert got[k].dtype == exp[k].dtype and np.array_equal(got[k], exp[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["narrow", "wide", "three"])
@pytest.mark.parametrize("which", ["random", "name_grouped", "reversed", "sorted", "sorted_rev_first"])
def test_columns_equal_host_sorted_batch(small_data, which, how):
    d, hb, nibs = small_data
    name, order, already = [o for o in input_orders(d, hb) if o[0] == which][0]
    inp = permute_hb(hb, order)
    exp_hb = inp if already else host_sorted(inp)
    ref = _ctx(hb); _push(ref, exp_hb, how); exp = _columns(ref); ref.close()
    c = _ctx(hb); _push(c, inp, how)
    assert c.sort_records() == already
    _assert_columns(_columns(c), exp)
    if already:                                  # nothing moved: not re-sorted into samtools order
        assert np.array_equal(c.fetch_column("flag", np.uint16), inp.cols["flag"])
    c.close()


def _edge_data():
    from breakid_b200 import api
    from test_chrom_edges import build_edge_batch, nibs_for
    d = build_edge_batch()
    return d, api.HostBatch.from_synth(d), nibs_for(d)


def _variant_kw(variant):
    return {"qual": 20, "sd_mult": 15} if variant == "q20s15" else {}


def _run(hb, nibs, mode, variant, sort, exclude=None, **kw):
    c = _ctx(hb, fast=mode, **_variant_kw(variant), **kw)
    c.push(hb)
    if sort:
        c.sort_records()
    if exclude is not None:
        c.set_exclude(exclude[:, 0], exclude[:, 1], exclude[:, 2])
    for t, (p, l) in enumerate(nibs):
        c.set_nib(t, p, l)
    res = c.run()
    got = c.fetch_clusters()
    c.close()
    return res, got


def _exclude_for(hb):
    iv = []
    for t, l in enumerate(hb.target_len):
        iv += [(t, 0, 3), (t, int(l) // 3, int(l) // 3 + 4000)]
    return np.array(iv, np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "exclude", "q20s15", "validate"])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("data", ["small", "config1", "edges"])
def test_calls_equal_host_sorted_and_oracle(request, data, mode, variant):
    import oracle_py as O
    from breakid_b200 import synth
    from test_gpu_parity import _prefilter
    if data == "edges":
        d, hb, nibs = _edge_data()
    else:
        d, hb, nibs = request.getfixturevalue("small_data" if data == "small" else "config1_data")
    if variant == "validate":
        if data == "edges":
            pytest.skip("the edge batch's split reads are covered by the other variants")
        from breakid_b200 import api
        hb = api.HostBatch(hb.cols, hb.name_hash, hb.side, hb.target_len, hb.target_names)
        genome = [synth.nib_ascii(p, l) for p, l in nibs]
        rng = np.random.RandomState(3)
        seq, _ = synth.split_read_sequences(hb, genome, corrupt=set(np.nonzero(rng.rand(hb.n_sa) < 0.3)[0].tolist()), seed=9)
        hb.set_seq(seq)
    order = np.random.RandomState(7).permutation(hb.n)
    shuf = permute_hb(hb, order)
    srt = host_sorted(shuf)
    kw = {"validate_align": 1} if variant == "validate" else {}
    ex = _exclude_for(hb) if variant == "exclude" else None
    r1, got = _run(shuf, nibs, mode, variant, True, ex, **kw)
    r2, exp = _run(srt, nibs, mode, variant, False, ex, **kw)
    assert r1 == r2 and got.tobytes() == exp.tobytes()
    assert len(exp) >= (1 if ex is not None else 4)
    if variant == "validate":
        return                                                   # the validator's oracle is test_align's
    base = srt
    if ex is not None:
        tid, pos = srt.cols["tid"].astype(np.int64), srt.cols["pos"].astype(np.int64)
        keep = np.ones(srt.n, bool)
        for t, b, e in ex:
            keep &= ~((tid == t) & (pos >= max(b, 0)) & (pos < e))
        base = _prefilter(srt, keep)
    m, s, dist, oc = O.run(base, nibs, mode=mode, **_variant_kw(variant))
    assert r1[:3] == (m, s, dist)
    assert got.tobytes() == oc.tobytes()


@pytest.mark.gpu
def test_device_decode_of_unsorted_bam(tmp_path, small_data):
    from breakid_b200 import api, bamio, synth
    d, hb, nibs = small_data
    order = np.random.RandomState(11).permutation(hb.n)
    bam = str(tmp_path / "reads.bam")
    bamio.write_bam(bam, synth.permute(d, order), sort_order="unsorted")
    exp_hb = host_sorted(permute_hb(hb, order))
    ref = _ctx(hb); ref.push(exp_hb); exp = _columns(ref); ref.close()
    f = api.BgzfFile(bam)
    c = _ctx(hb)
    c.push_bgzf(f)
    assert c.sort_records() is False
    got = _columns(c)
    fl = exp["flag"]                                        # isize is only defined on the records insert statistics read
    read = ((fl & 1) != 0) & ((fl & 2) != 0) & ((fl & (0x4 | 0x100 | 0x200 | 0x400)) == 0)
    assert np.array_equal(got.pop("isize")[read], exp.pop("isize")[read])
    _assert_columns(got, exp)
    for t, (p, l) in enumerate(nibs):
        c.set_nib(t, p, l)
    r1 = c.run(); got = c.fetch_clusters(); c.close(); f.close()
    r2, want = _run(exp_hb, nibs, 0, "plain", False)
    assert r1 == r2 and got.tobytes() == want.tobytes() and len(got) >= 4


def _device_batch(hb, keep):
    """api.Batch of device tensors holding hb's columns (wide form) and its sparse / SA tables"""
    from breakid_b200 import api
    b = api.Batch()
    b.n = hb.n
    for k, _ in api._COLS:
        t = torch.from_numpy(hb.cols[k].view(np.int16) if k == "flag" else hb.cols[k]).cuda(); keep.append(t); setattr(b, k, t.data_ptr())
    b.n_x = hb.n_x
    for k, _ in api._XCOLS:
        a = hb.x[k]
        t = torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a.view(np.int32)).cuda(); keep.append(t); setattr(b, k, t.data_ptr())
    b.n_sa = hb.n_sa
    for k, _ in api._SIDE:
        a = hb.side[k]
        t = torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a).cuda(); keep.append(t); setattr(b, k, t.data_ptr())
    return b


@pytest.mark.gpu
def test_borrowed_columns_are_not_written(small_data):
    d, hb, nibs = small_data
    inp = permute_hb(hb, np.random.RandomState(5).permutation(hb.n))
    keep = []
    b = _device_batch(inp, keep)
    before = [int(t.view(torch.uint8).to(torch.int64).sum()) for t in keep]
    c = _ctx(hb)
    c.push_device(b)
    assert c.sort_records() is False
    torch.cuda.synchronize()
    assert [int(t.view(torch.uint8).to(torch.int64).sum()) for t in keep] == before
    exp_hb = host_sorted(inp)
    ref = _ctx(hb); ref.push(exp_hb, narrow=False); exp = _columns(ref); ref.close()
    _assert_columns(_columns(c), exp)
    for t, (p, l) in enumerate(nibs):
        c.set_nib(t, p, l)
    r1 = c.run(); got = c.fetch_clusters(); c.close()
    r2, want = _run(exp_hb, nibs, 0, "plain", False)
    assert r1 == r2 and got.tobytes() == want.tobytes()


@pytest.mark.gpu
def test_sorted_narrow_context_keeps_narrow_classify(small_data):
    from breakid_b200 import api
    d, hb, nibs = small_data
    inp = permute_hb(hb, np.random.RandomState(6).permutation(hb.n))
    names = []
    for h, sort in ((host_sorted(inp), False), (inp, True)):
        c = _ctx(hb); c.push(h, narrow=True)
        if sort:
            c.sort_records()
        api.profile_kernels(True); api.profile_report()
        c.insert_stats()
        rep = api.profile_report(); api.profile_kernels(False)
        names.append(sorted(k for k in rep if "k1_classify" in k))
        c.close()
    assert names[0] == names[1] and any("k1_classify<true, true>" in k for k in names[0]), names


@pytest.mark.gpu
def test_edge_cases(small_data):
    from breakid_b200 import api
    d, hb, nibs = small_data
    c = _ctx(hb)
    assert c.sort_records() is True                           # n = 0
    from test_multi_gloo import _slice
    one = _slice(hb, 5, 6)
    c.push(one)
    assert c.sort_records() is True
    _assert_columns(_columns(c), _columns_of(one))
    c.reset()
    # all unmapped: tid = pos = -1 (sorted already), then shuffled flags make no difference to the order
    cols = {k: v[:1000].copy() for k, v in hb.cols.items()}
    cols["tid"][:] = -1; cols["pos"][:] = -1; cols["flag"][:] = 0x1 | 0x4 | 0x8
    cols["flag"][::3] |= 0x10
    un = api.HostBatch(cols, hb.name_hash[:2000], _no_side(), hb.target_len, hb.target_names)
    c.push(un)
    assert c.sort_records() is True
    _assert_columns(_columns(c), _columns_of(un))
    c.reset()
    # push -> sort -> push -> sort
    a = permute_hb(hb, np.random.RandomState(8).permutation(hb.n))
    h = hb.n // 2
    c.push(_slice(a, 0, h))
    assert c.sort_records() is False
    c.push(_slice(a, h, hb.n))
    assert c.sort_records() is False
    _assert_columns(_columns(c), _columns_of(host_sorted(a)))
    # argument errors leave the context as it was
    bad = {k: v[:10].copy() for k, v in hb.cols.items()}
    bad["tid"][3] = len(hb.target_names)
    c2 = _ctx(hb); c2.push(api.HostBatch(bad, hb.name_hash[:20], _no_side(), hb.target_len, hb.target_names), narrow=False)
    before = _columns(c2)
    with pytest.raises(api.BkidError):
        c2.sort_records()
    _assert_columns(_columns(c2), before)
    c2.close(); c.close()


def _no_side():
    z = np.zeros(1, np.uint32)
    return {"sa_rec": np.zeros(0, np.uint32), "cig_off": z, "cig_ops": np.zeros(0, np.uint32), "sa_off": z, "sa_txt": np.zeros(0, np.uint8)}


def _columns_of(h):
    c = _ctx(h); c.push(h); out = _columns(c); c.close()
    return out


@pytest.mark.gpu
def test_more_than_2_30_records_against_torch_sort():
    """about 1.1e9 records built on the device, pushed as borrowed columns (group path: targets cut into groups of
    < 2^30 records); tid / pos / flag / mapq against torch.sort(stable=True) of the same key, sparse rows renumbered"""
    from breakid_b200 import api
    n, nt = 1_100_000_000, 24
    dev = "cuda"
    g = torch.Generator(device=dev); g.manual_seed(1)
    tid = torch.randint(-1, nt, (n,), device=dev, dtype=torch.int32, generator=g)
    pos = torch.randint(0, 1 << 27, (n,), device=dev, dtype=torch.int32, generator=g)
    flag = (torch.randint(0, 2, (n,), device=dev, dtype=torch.int32, generator=g) * 0x10 | 0x3).to(torch.int16)
    mapq = (torch.arange(n, device=dev, dtype=torch.int64) % 251).to(torch.uint8)
    isize16 = torch.zeros(n, device=dev, dtype=torch.int16)
    span16 = torch.full((n,), 100, device=dev, dtype=torch.int16)
    nx = 1000
    x_rec = torch.unique(torch.randint(0, n, (nx,), device=dev, dtype=torch.int64, generator=g))
    nx = int(x_rec.numel())
    cols = [tid, pos, flag, mapq, isize16, span16]
    x_rec32 = x_rec.to(torch.int32)                     # < 2^31
    x_m = torch.arange(nx, device=dev, dtype=torch.int32)
    x_nh = torch.arange(2 * nx, device=dev, dtype=torch.int64)
    sa_off = torch.zeros(1, device=dev, dtype=torch.int32)
    b = api.Batch()
    b.n = n; b.flag = flag.data_ptr(); b.mapq = mapq.data_ptr(); b.tid = tid.data_ptr(); b.pos = pos.data_ptr()
    b.isize16 = isize16.data_ptr(); b.span16 = span16.data_ptr()
    b.n_x = nx; b.x_rec = x_rec32.data_ptr(); b.x_mtid = x_m.data_ptr(); b.x_mpos = x_m.data_ptr(); b.x_name_hash = x_nh.data_ptr()
    b.n_sa = 0; b.cig_off = b.sa_off = b.oc_off = sa_off.data_ptr()
    c = api.Context([1 << 28] * nt, ["chr%d" % (i + 1) for i in range(nt)], device=0)
    c.push_device(b)
    assert c.sort_records() is False
    rank = torch.where(tid < 0, torch.full_like(tid, nt), tid).to(torch.int64)
    key = (rank << 33) | ((pos.to(torch.int64) + 1) << 1) | ((flag.to(torch.int64) >> 4) & 1)
    del rank
    skey, perm = torch.sort(key, stable=True)
    del key, skey
    for k, ref in (("tid", tid), ("pos", pos), ("flag", flag), ("mapq", mapq)):
        got = c.fetch_column(k, {"flag": np.uint16, "mapq": np.uint8}.get(k, np.int32))
        exp = ref[perm].cpu().numpy()
        assert np.array_equal(got.view(exp.dtype), exp), k
        del got, exp
    inv = torch.empty_like(perm); inv[perm] = torch.arange(n, device=dev)
    new_x = inv[x_rec]
    ordx = torch.argsort(new_x)
    assert np.array_equal(c.fetch_column("x_rec", np.uint32).astype(np.int64), new_x[ordx].cpu().numpy())
    assert np.array_equal(c.fetch_column("x_mtid", np.int32), x_m[ordx].cpu().numpy())
    c.close()


# ------------------------------------------------------------------------------------------------ the driver
def _driver(bam, out, nib, refgene, extra=(), env=None):
    return subprocess.run([DRIVER, "-i", bam, "-o", out, "-n", nib, "-r", refgene, "-all"] + list(extra),
                          timeout=600, capture_output=True, text=True, env=env)


@pytest.mark.gpu
def test_driver_sort_on_name_grouped_bam(tmp_path, small_data):
    import reference_calls as R
    from breakid_b200 import bamio, synth
    d, hb, nibs = small_data
    order = np.argsort(d.cols["name_id"].cpu().numpy(), kind="stable")
    ps = bamio.write_dataset(str(tmp_path / "sorted"), d)
    R.index(ps["bam"])
    pu = bamio.write_dataset(str(tmp_path / "grouped"), synth.permute(d, order), sort_order="queryname")
    ref = str(tmp_path / "sorted" / "out")
    g = _driver(ps["bam"], ref, ps["nib"], ps["refgene"])
    assert g.returncode == 0, g.stderr[-500:]
    R.match_oracle(ref, d)
    files = ("_fusion.txt", "_fusion_all.txt", "_params.txt")
    want = {s: open(ref + s).read().replace(str(tmp_path / "sorted"), "@") for s in files}
    for tag, env in (("dev", None), ("host", dict(os.environ, BKID_HOST_DECODE="1"))):
        o = str(tmp_path / "grouped" / ("out_" + tag))
        g = _driver(pu["bam"], o, pu["nib"], pu["refgene"], ["-sort"], env)
        assert g.returncode == 0, (tag, g.stderr[-500:])
        for s in files:
            assert open(o + s).read().replace(str(tmp_path / "grouped"), "@").replace("out_" + tag, "out") == want[s], (tag, s)
        tm = dict(ln.split("\t") for ln in open(o + "_b200_timings.txt").read().splitlines())
        assert tm["input_was_sorted"] == "0" and float(tm["sort_ms"]) > 0
    # -sort on the sorted BAM: the same files
    o = str(tmp_path / "sorted" / "out_s")
    g = _driver(ps["bam"], o, ps["nib"], ps["refgene"], ["-sort"])
    assert g.returncode == 0, g.stderr[-500:]
    for s in files:
        assert open(o + s).read().replace(str(tmp_path / "sorted"), "@").replace("out_s", "out") == want[s], s
    # without -sort the unsorted, unindexed BAM fails as before
    g = _driver(pu["bam"], str(tmp_path / "grouped" / "nosort"), pu["nib"], pu["refgene"])
    assert g.returncode == 1 and "please index bam-file first" in g.stderr
