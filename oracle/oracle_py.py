"""ctypes access to the CPU oracle (oracle/liboracle.so) and, when built, to the real reference
(oracle/_ref/libbreakid_ref.so, oracle/_ref/BreakID_ref).  TEST INFRASTRUCTURE ONLY: imported by
tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs; never by the
product package."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_ORACLE = os.path.join(HERE, "liboracle.so")
LIB_REF = os.path.join(HERE, "_ref", "libbreakid_ref.so")
REF_BIN = os.path.join(HERE, "_ref", "BreakID_ref")
REF_INDEX = os.path.join(HERE, "_ref", "bamindex")
REF_INSTALL = os.path.join(HERE, "_ref", "install")

sys.path.insert(0, os.path.dirname(HERE))
from breakid_b200.api import CLUSTER_DTYPE, EVIDENCE_DTYPE, PAIR_DTYPE  # noqa: E402  (POD layouts are shared)

L, D, I = C.c_long, C.c_double, C.c_int
u8p = np.ctypeslib.ndpointer(np.uint8, flags="C")
u16p = np.ctypeslib.ndpointer(np.uint16, flags="C")
u32p = np.ctypeslib.ndpointer(np.uint32, flags="C")
i32p = np.ctypeslib.ndpointer(np.int32, flags="C")
u64p = np.ctypeslib.ndpointer(np.uint64, flags="C")
f64p = np.ctypeslib.ndpointer(np.float64, flags="C")

_o = None
_r = None


def build(ref: bool = True):
    tgt = ["oracle"] + (["ref"] if ref and os.path.isdir("/root/reference") else [])
    subprocess.check_call(["make", "-s", "-C", HERE, "-j8"] + tgt)


def have_ref() -> bool:
    return os.path.exists(LIB_REF) and os.path.exists(REF_BIN)


def olib():
    global _o
    if _o is None:
        if not os.path.exists(LIB_ORACLE):
            build(ref=False)
        o = C.CDLL(LIB_ORACLE)
        o.orc_insert_stats.argtypes = [L, u16p, i32p, C.POINTER(D), C.POINTER(D)] + [C.POINTER(C.c_int64)] * 3
        o.orc_set_refine_consts.argtypes = [I, I]
        o.orc_dist.restype = D
        o.orc_dist.argtypes = [D, D, I]
        o.orc_scan.restype = L
        o.orc_scan.argtypes = [L, u16p, u8p, i32p, i32p, i32p, i32p, u64p, I, u32p, C.POINTER(C.c_char_p), L, D, C.POINTER(C.c_void_p)]
        o.orc_bucket_rank_table.argtypes = [I, C.POINTER(C.c_char_p), i32p]
        o.orc_std_sort_perm.argtypes = [L, u32p, u32p]
        o.orc_model_sort_perm.argtypes = [L, u32p, u32p]
        o.orc_remove_isolated.restype = L
        o.orc_remove_isolated.argtypes = [L, u32p, u32p, D, u32p]
        for f in (o.orc_cluster_fast, o.orc_cluster_ahc, o.orc_model_cluster_ahc):
            f.restype = L
            f.argtypes = [L, u32p, u32p, D, u32p, i32p, C.POINTER(I)]
        for f in (o.orc_ahc_tree, o.orc_model_ahc_tree):
            f.restype = L
            f.argtypes = [L, f64p, f64p, L, i32p, i32p, i32p]
        o.orc_set_ahc_model.argtypes = [I]
        o.orc_model_ahc_flags.argtypes = [C.POINTER(L), C.POINTER(L)]
        o.orc_model_heapsort_count.restype = L
        o.orc_is_complementary.argtypes = [C.c_char_p, C.c_char_p, I]
        rec = [L, u16p, u8p, i32p, i32p, i32p, u64p, L, u32p, u32p, u32p, u32p, u8p, u32p, u8p]
        o.orc_find_sa_reads.restype = L
        o.orc_find_sa_reads.argtypes = rec + [I, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
        o.orc_find_bp.argtypes = rec + [I, C.c_char_p, C.c_uint32, C.c_uint32, I, C.c_uint32, C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        o.orc_single_base_depth.restype = D
        o.orc_single_base_depth.argtypes = [L, u16p, u8p, i32p, i32p, i32p, I, C.c_uint64]
        o.orc_neighbor_41.argtypes = [u8p, C.c_uint64, C.c_int32, C.c_char_p]
        o.orc_longest_repeat.argtypes = [C.c_char_p]
        o.orc_run.restype = L
        o.orc_run.argtypes = [L, u16p, u8p, i32p, i32p, i32p, i32p, i32p, i32p, u64p,
                              L, u32p, u32p, u32p, u32p, u8p, u32p, u8p,
                              I, u32p, C.POINTER(C.c_char_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64),
                              I, I, I, C.POINTER(D), C.POINTER(D), C.POINTER(D), C.POINTER(C.c_void_p)]
        o.orc_free.argtypes = [C.c_void_p]
        _o = o
    return _o


def rlib():
    global _r
    if _r is None:
        r = C.CDLL(LIB_REF)
        r.ref_insert_stats.argtypes = [C.c_char_p, C.POINTER(D), C.POINTER(D)]
        r.ref_scan.restype = L
        r.ref_scan.argtypes = [C.c_char_p, I, D, C.c_char_p, C.POINTER(C.c_void_p)]
        r.ref_remove_isolated.restype = L
        r.ref_remove_isolated.argtypes = [L, u32p, u32p, D, u32p]
        for f in (r.ref_cluster_fast, r.ref_cluster_ahc):
            f.restype = L
            f.argtypes = [L, u32p, u32p, D, u32p, i32p, C.POINTER(I), I]
        r.ref_std_sort_perm.argtypes = [L, u32p, I, u32p]
        r.ref_find_sa_reads.restype = L
        r.ref_find_sa_reads.argtypes = [C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
        r.ref_find_bp.argtypes = [C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint32, C.c_char_p, C.c_uint32, C.c_uint32,
                                  C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        r.ref_single_base_depth.restype = D
        r.ref_single_base_depth.argtypes = [C.c_char_p, C.c_char_p, C.c_uint64]
        r.ref_is_complementary.argtypes = [C.c_char_p, C.c_char_p, I]
        r.ref_neighbor_41.argtypes = [C.c_char_p, C.c_char_p, C.c_int32, C.c_char_p]
        r.ref_longest_repeat.argtypes = [C.c_char_p]
        r.ref_ahc_tree.restype = L
        r.ref_ahc_tree.argtypes = [L, f64p, f64p, L, i32p, i32p, i32p]
        r.ref_free.argtypes = [C.c_void_p]
        _r = r
    return _r


class quiet:
    """silence the reference's std::cout chatter (fd level)"""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        self.null = os.open(os.devnull, os.O_WRONLY)
        os.dup2(self.null, 1)

    def __exit__(self, *a):
        os.dup2(self.saved, 1)
        os.close(self.null)
        os.close(self.saved)


def _take(ptr, n, dtype, free):
    out = np.zeros(n, dtype)
    if n:
        C.memmove(out.ctypes.data, ptr, n * dtype.itemsize)
    free(ptr)
    return out


def _names(hb):
    return (C.c_char_p * len(hb.target_names))(*[s.encode() for s in hb.target_names])


def _recargs(hb):
    c, s = hb.cols, hb.side
    return [hb.n, c["flag"], c["mapq"], c["tid"], c["pos"], c["endpos"], hb.name_hash, hb.n_sa, s["sa_rec"], s["cig_off"],
            _nz(s["cig_ops"], np.uint32), s["sa_off"], _nz(s["sa_txt"], np.uint8), s["oc_off"], _nz(s["oc_txt"], np.uint8)]


def _nz(a, dt):
    return a if a.shape[0] else np.zeros(1, dt)


# ---------------------------------------------------------------- oracle on a HostBatch
def insert_stats(hb):
    m, s = D(), D()
    a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
    olib().orc_insert_stats(hb.n, hb.cols["flag"], hb.cols["isize"], C.byref(m), C.byref(s), C.byref(a), C.byref(b), C.byref(c))
    return m.value, s.value, a.value, b.value, c.value


def dist(mean, sd, times=2, sd_mult=3):
    olib().orc_set_sd_mult(int(sd_mult))
    try:
        return olib().orc_dist(mean, sd, times)
    finally:
        olib().orc_set_sd_mult(3)


def scan(hb, qual, w):
    out = C.c_void_p()
    c = hb.cols
    n = olib().orc_scan(hb.n, c["flag"], c["mapq"], c["tid"], c["pos"], c["mtid"], c["mpos"], hb.name_hash,
                        len(hb.target_names), hb.target_len, _names(hb), qual, w, C.byref(out))
    return _take(out, n, PAIR_DTYPE, olib().orc_free)


def remove_isolated(p1, p2, w):
    p1 = np.ascontiguousarray(p1, np.uint32); p2 = np.ascontiguousarray(p2, np.uint32)
    out = np.zeros(p1.shape[0] + 2, np.uint32)
    n = olib().orc_remove_isolated(p1.shape[0], p1, p2, w, out)
    return out[:n]


def cluster(mode, p1, p2, thr, model=False):
    p1 = np.ascontiguousarray(p1, np.uint32); p2 = np.ascontiguousarray(p2, np.uint32)
    oi = np.zeros(p1.shape[0] + 2, np.uint32); oc = np.zeros(p1.shape[0] + 2, np.int32)
    r = I()
    f = olib().orc_cluster_fast if mode else (olib().orc_model_cluster_ahc if model else olib().orc_cluster_ahc)
    n = f(p1.shape[0], p1, p2, thr, oi, oc, C.byref(r))
    return oi[:n], oc[:n], r.value


class ahc_model:
    """inside the block, the per-bucket AHC of run() and of OracleEngine.cluster is the component model instead of the
    literal O(N^3) restatement"""

    def __enter__(self):
        olib().orc_set_ahc_model(1)

    def __exit__(self, *a):
        olib().orc_set_ahc_model(0)


def ahc_flags(p1, p2, thr):
    """(components the device's speculative AHC pass flags, decisions that flag them) on these points (post-mask order),
    predicted by the component model"""
    cluster(0, p1, p2, thr, model=True)
    f, d = L(), L()
    olib().orc_model_ahc_flags(C.byref(f), C.byref(d))
    return f.value, d.value


def heapsort_count():
    """depth-exhausted segments the sort model has finished with the literal heapsort so far (cumulative)"""
    return olib().orc_model_heapsort_count()


def banded_edit(q: bytes, r: bytes, w: int) -> int:
    L = olib()
    L.orc_banded_edit.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int]
    L.orc_banded_edit.restype = C.c_int
    return int(L.orc_banded_edit(q, len(q), r, len(r), w))


def sort_perm(key, model=False):
    key = np.ascontiguousarray(key, np.uint32)
    perm = np.zeros(key.shape[0], np.uint32)
    (olib().orc_model_sort_perm if model else olib().orc_std_sort_perm)(key.shape[0], key, perm)
    return perm


_refine = [2, 10]                             # the values in force in liboracle (bp_err, mismatch)


class refine_consts:
    """inside the block, every refinement entry point of the oracle (run, find_sa_reads, find_bp and the shard pieces of
    OracleEngine) votes with a window of +-bp_err and accepts complementary cigars within `mismatch` bases: the literals
    2 and 10 of src/BreakID.cc:444-445 and :891, bkid_params.bp_pos_error and mismatch_num on the device.  None keeps
    the value in force; the values in force before the block come back when it ends"""

    def __init__(self, bp_err=None, mismatch=None):
        self.bp_err, self.mismatch = bp_err, mismatch

    def __enter__(self):
        self.saved = tuple(_refine)
        _refine[:] = [self.saved[0] if self.bp_err is None else int(self.bp_err),
                      self.saved[1] if self.mismatch is None else int(self.mismatch)]
        olib().orc_set_refine_consts(*_refine)

    def __exit__(self, *a):
        _refine[:] = self.saved
        olib().orc_set_refine_consts(*_refine)


def find_sa_reads(hb, tid, start, end, mismatch=None):
    out = C.c_void_p()
    with refine_consts(mismatch=mismatch):
        n = olib().orc_find_sa_reads(*_recargs(hb), tid, start, end, C.byref(out))
    return _take(out, n, EVIDENCE_DTYPE, olib().orc_free)


def find_bp(hb, tid1, s1, e1, tid2, s2, e2, bp_err=None, mismatch=None):
    a, b = C.c_int32(), C.c_int32()
    with refine_consts(bp_err, mismatch):
        v = olib().orc_find_bp(*_recargs(hb), tid1, hb.target_names[tid1].encode(), s1, e1, tid2, s2, e2, C.byref(a), C.byref(b))
    return v, a.value, b.value


def single_base_depth(hb, tid, pos):
    c = hb.cols
    return olib().orc_single_base_depth(hb.n, c["flag"], c["mapq"], c["tid"], c["pos"], c["endpos"], tid, pos)


def neighbor_41(packed, nbases, bp):
    buf = C.create_string_buffer(42)
    olib().orc_neighbor_41(np.ascontiguousarray(packed, np.uint8), nbases, bp, buf)
    return buf.value


def run(hb, nibs=None, qual=20, times=2, mode=0, sd_mult=3, bp_err=None, mismatch=None):
    """whole hot path; nibs = list of (packed uint8 array, n_bases) per tid or None.  sd_mult replaces the literal 3 of
    src/BreakID.cc:103 (the -s extension), bp_err and mismatch the literals 2 and 10 of the refinement (refine_consts;
    None: the values in force)"""
    olib().orc_set_sd_mult(int(sd_mult))
    try:
        with refine_consts(bp_err, mismatch):
            return _run(hb, nibs, qual, times, mode)
    finally:
        olib().orc_set_sd_mult(3)


def _run(hb, nibs, qual, times, mode):
    c, s = hb.cols, hb.side
    nt = len(hb.target_names)
    if nibs is not None:                          # an entry (None, 0): no nib for that tid, its 41-mers stay empty
        keep = [None if p is None else np.ascontiguousarray(p, np.uint8) for p, _ in nibs]
        ptrs = (C.c_void_p * nt)(*[None if k is None else k.ctypes.data for k in keep])
        lens = (C.c_uint64 * nt)(*[int(l) for _, l in nibs])
    else:
        ptrs, lens = None, None
    m, sd, d = D(), D(), D()
    out = C.c_void_p()
    n = olib().orc_run(hb.n, c["flag"], c["mapq"], c["tid"], c["pos"], c["mtid"], c["mpos"], c["isize"], c["endpos"], hb.name_hash,
                       hb.n_sa, s["sa_rec"], s["cig_off"], _nz(s["cig_ops"], np.uint32), s["sa_off"], _nz(s["sa_txt"], np.uint8),
                       s["oc_off"], _nz(s["oc_txt"], np.uint8), nt, hb.target_len, _names(hb),
                       C.cast(ptrs, C.POINTER(C.c_void_p)) if ptrs is not None else None,
                       C.cast(lens, C.POINTER(C.c_uint64)) if lens is not None else None,
                       qual, times, mode, C.byref(m), C.byref(sd), C.byref(d), C.byref(out))
    if n < 0:
        olib().orc_free(out)
        raise RuntimeError("oracle: reference 'error cigar' fatal path")
    return m.value, sd.value, d.value, _take(out, n, CLUSTER_DTYPE, olib().orc_free)


# ---------------------------------------------------------------- the real reference
def ref_index(bam):
    subprocess.check_call([REF_INDEX, bam])


def ref_install_refgene(path):
    import shutil
    os.makedirs(os.path.join(REF_INSTALL, "ref_files"), exist_ok=True)
    shutil.copy(path, os.path.join(REF_INSTALL, "ref_files", "refGene.txt"))


def ref_run_binary(bam, prefix, nib_dir, fast=False, all_=True, qual=None, timeout=3600, extra=(), sd_mult=None):
    """the reference binary.  sd_mult: the binary built by `make -C oracle ref_s`, in which the literal 3 of
    src/BreakID.cc:103 is read from BREAKID_SD_MULT (the reference has no -s flag: an unknown flag makes it crash)"""
    env = None
    exe = REF_BIN
    if sd_mult is not None:
        exe = REF_BIN + "_s"
        env = dict(os.environ, BREAKID_SD_MULT=str(int(sd_mult)))
    cmd = [exe, "-i", bam, "-o", prefix, "-n", nib_dir]
    if fast:
        cmd.append("-fast")
    if all_:
        cmd.append("-all")
    if qual is not None:
        cmd += ["-q", str(qual)]
    cmd += list(extra)
    return subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)


def ref_scan(bam, qual, w, nib_dir):
    out = C.c_void_p()
    with quiet():
        n = rlib().ref_scan(bam.encode(), qual, w, nib_dir.encode(), C.byref(out))
    return _take(out, n, PAIR_DTYPE, rlib().ref_free)


def ref_find_sa_reads(bam, chr_, start, end):
    out = C.c_void_p()
    with quiet():
        n = rlib().ref_find_sa_reads(bam.encode(), chr_.encode(), start, end, C.byref(out))
    return _take(out, n, EVIDENCE_DTYPE, rlib().ref_free)
