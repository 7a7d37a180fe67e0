"""ctypes binding of include/breakid_b200.h (the C ABI of the CUDA library) and of the host BAM
decoder.  Python here is test / bench plumbing: the product is ``libbreakid_b200.so`` (CUDA) and
the C++ host driver ``BreakID`` (breakid_b200/host).  There is no CPU fallback: if the CUDA library
is missing or no device is usable, loading / ``Context()`` raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_CUDA = os.path.join(_HERE, "csrc", "libbreakid_b200.so")
LIB_HOST = os.path.join(_HERE, "host", "libbreakid_host.so")


class Header(C.Structure):
    _fields_ = [("n_targets", C.c_int32), ("target_len", C.POINTER(C.c_uint32)),
                ("target_name", C.POINTER(C.c_char_p))]


class Params(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("qual", "times", "fast", "min_reads", "bp_pos_error",
                                         "mismatch_num", "sd_mult", "validate_align")]


class Batch(C.Structure):
    _fields_ = [("n", C.c_int64), ("flag", C.c_void_p), ("mapq", C.c_void_p),
                ("tid", C.c_void_p), ("pos", C.c_void_p), ("isize", C.c_void_p), ("endpos", C.c_void_p),
                ("n_x", C.c_int64), ("x_rec", C.c_void_p), ("x_mtid", C.c_void_p), ("x_mpos", C.c_void_p), ("x_name_hash", C.c_void_p),
                ("n_sa", C.c_int64), ("sa_rec", C.c_void_p), ("cig_off", C.c_void_p), ("cig_ops", C.c_void_p),
                ("sa_off", C.c_void_p), ("sa_txt", C.c_void_p), ("oc_off", C.c_void_p), ("oc_txt", C.c_void_p),
                ("isize16", C.c_void_p), ("span16", C.c_void_p), ("n_tid_runs", C.c_int64), ("tid_run_start", C.c_void_p), ("tid_run_tid", C.c_void_p),
                ("seq_off", C.c_void_p), ("seq4", C.c_void_p), ("seq_len", C.c_void_p)]


PAIR_DTYPE = np.dtype([
    ("name_lo", "<u8"), ("name_hi", "<u8"), ("p1_tid", "<i4"), ("p2_tid", "<i4"),
    ("p1_pos", "<u4"), ("p2_pos", "<u4"), ("p1_chr_pos", "<u4"), ("p2_chr_pos", "<u4"),
    ("p1_flag", "<u2"), ("p2_flag", "<u2"), ("p1_mapq", "u1"), ("p2_mapq", "u1"),
    ("p1_strand", "u1"), ("p2_strand", "u1"), ("bucket", "<i4"), ("cluster", "<i4"),
    ("orig", "<u4"), ("_pad", "<u4")])
assert PAIR_DTYPE.itemsize == 64

CLUSTER_DTYPE = np.dtype([
    ("bucket", "<i4"), ("id", "<i4"), ("p1_tid", "<i4"), ("p2_tid", "<i4"),
    ("p1_mean_pos", "<u8"), ("p2_mean_pos", "<u8"),
    ("p1_min_pos", "<u4"), ("p1_max_pos", "<u4"), ("p2_min_pos", "<u4"), ("p2_max_pos", "<u4"),
    ("p1_exact_pos", "<u4"), ("p2_exact_pos", "<i4"),
    ("n_split_read", "<i8"), ("n_discordant_pair", "<i8"),
    ("p1_bp_depth", "<f8"), ("p2_bp_depth", "<f8"), ("p1_alle_freq", "<f4"), ("p2_alle_freq", "<f4"),
    ("fusion_type", "<i4"), ("is_rpt", "<i4"), ("p1_rpt", "S44"), ("p2_rpt", "S44")])
assert CLUSTER_DTYPE.itemsize == 192

EVIDENCE_DTYPE = np.dtype([
    ("name_lo", "<u8"), ("name_hi", "<u8"), ("primary_chr", "<i4"), ("secondary_chr", "<i4"),
    ("primary_start", "<u4"), ("secondary_start", "<u4"), ("primary_end", "<u4"), ("secondary_end", "<u4"),
    ("primary_bp", "<u4"), ("secondary_bp", "<u4"), ("primary_cigar_h", "<u8"), ("secondary_cigar_h", "<u8"),
    ("flag", "<u2"), ("secondary", "u1"), ("_pad", "u1", 5)])
assert EVIDENCE_DTYPE.itemsize == 72

TIMING_FIELDS_F = ("h2d", "insert_stats", "classify", "join", "bucket_sort", "mask", "cluster", "summarize",
                   "evidence", "refine", "total")
TIMING_FIELDS_I = ("n_records", "n_candidates", "n_pairs", "n_masked", "n_clustered", "n_clusters", "n_sa",
                   "n_evidence", "n_called", "kernel_launches")


class Timings(C.Structure):
    _fields_ = [(k, C.c_float) for k in TIMING_FIELDS_F] + [("_pad", C.c_float)] + \
               [(k, C.c_int64) for k in TIMING_FIELDS_I]


FUSION_TYPES = ["Unknown", "Translocation", "Inversion", "Duplication", "Deletion"]

_COLS = (("flag", np.uint16), ("mapq", np.uint8), ("tid", np.int32), ("pos", np.int32), ("isize", np.int32), ("endpos", np.int32))
_XCOLS = (("x_rec", np.uint32), ("x_mtid", np.int32), ("x_mpos", np.int32), ("x_name_hash", np.uint64))
_SIDE = (("sa_rec", np.uint32), ("cig_off", np.uint32), ("cig_ops", np.uint32), ("sa_off", np.uint32),
         ("sa_txt", np.uint8), ("oc_off", np.uint32), ("oc_txt", np.uint8))
_SEQ = (("seq_off", np.uint32), ("seq4", np.uint8), ("seq_len", np.int32))        # optional read bases of the SA records


class HostBatch:
    """numpy-backed record batch + header; owns the arrays a ``Batch`` struct points to.

    Built from dense per-record arrays (incl. ``mtid``, ``mpos`` and the [2n] ``name_hash``); the sparse
    mate/name table of the C ABI (records that are not proper pairs or carry an SA tag) is derived here.
    ``cols['mtid']``, ``cols['mpos']`` and ``name_hash`` stay available as dense arrays for the CPU oracle,
    zeroed outside the sparse table (nothing on the path reads them there)."""

    def __init__(self, cols: Dict[str, np.ndarray], name_hash: np.ndarray, side: Dict[str, np.ndarray],
                 target_len: Sequence[int], target_names: Sequence[str]):
        self.cols = {k: np.ascontiguousarray(cols[k], dtype=dt) for k, dt in _COLS}
        self.n = int(self.cols["flag"].shape[0])
        name_hash = np.ascontiguousarray(name_hash, dtype=np.uint64).reshape(-1)
        assert name_hash.shape[0] == 2 * self.n
        n_sa = int(side["sa_rec"].shape[0]) if "sa_rec" in side else 0
        in_x = (self.cols["flag"] & 2) == 0
        if n_sa:
            in_x[np.asarray(side["sa_rec"], dtype=np.int64)] = True
        xr = np.nonzero(in_x)[0]
        self.x = {"x_rec": xr.astype(np.uint32), "x_mtid": np.ascontiguousarray(np.asarray(cols["mtid"], np.int32)[xr]),
                  "x_mpos": np.ascontiguousarray(np.asarray(cols["mpos"], np.int32)[xr]),
                  "x_name_hash": np.ascontiguousarray(name_hash.reshape(-1, 2)[xr].reshape(-1))}
        self.n_x = int(xr.shape[0])
        for k in ("mtid", "mpos"):
            dense = np.zeros(self.n, np.int32)
            dense[xr] = self.x["x_" + k]
            self.cols[k] = dense
        nh = np.zeros((self.n, 2), np.uint64)
        nh[xr] = self.x["x_name_hash"].reshape(-1, 2)
        self.name_hash = nh.reshape(-1)
        side = dict(side)
        if "oc_off" not in side:
            side["oc_off"] = np.zeros(n_sa + 1, np.uint32)
            side["oc_txt"] = np.zeros(0, np.uint8)
        self.side = {k: np.ascontiguousarray(side[k], dtype=dt) for k, dt in _SIDE}
        self.seq = {k: np.ascontiguousarray(side[k], dtype=dt) for k, dt in _SEQ} if all(k in side for k, _ in _SEQ) else None
        self.n_sa = n_sa
        self.target_len = np.ascontiguousarray(target_len, dtype=np.uint32)
        self.target_names = [str(x) for x in target_names]

    def set_seq(self, seq: Optional[Dict[str, np.ndarray]]):
        """attach / remove the optional read bases of the SA records (seq_off, seq4, seq_len)"""
        self.seq = None if seq is None else {k: np.ascontiguousarray(seq[k], dtype=dt) for k, dt in _SEQ}

    # -- views -----------------------------------------------------------------------------
    def narrow(self) -> Dict[str, np.ndarray]:
        """narrow encodings of isize / endpos / tid (include/breakid_b200.h) for the columns that fit; cached"""
        if getattr(self, "_narrow", None) is None:
            c, nr = self.cols, {}
            if self.n:
                sp = c["endpos"].astype(np.int64) - c["pos"].astype(np.int64)
                if sp.min() >= 0 and sp.max() <= 65535:
                    nr["span16"] = sp.astype(np.uint16)
                fl = c["flag"]
                read = ((fl & 1) != 0) & ((fl & 2) != 0) & ((fl & (0x4 | 0x100 | 0x200 | 0x400)) == 0)       # src/BreakID.cc:1932
                iz = c["isize"]
                if not read.any() or (iz[read].min() >= -32768 and iz[read].max() <= 32767):
                    nr["isize16"] = np.clip(iz, -32768, 32767).astype(np.int16)
                start = np.nonzero(np.concatenate([[True], c["tid"][1:] != c["tid"][:-1]]))[0]
                if start.shape[0] <= 65536:
                    nr["tid_run_start"] = start.astype(np.uint32)
                    nr["tid_run_tid"] = np.ascontiguousarray(c["tid"][start])
            self._narrow = nr
        return self._narrow

    def struct(self, narrow: bool = True) -> Batch:
        b = Batch()
        b.n = self.n
        for k, _ in _COLS:
            setattr(b, k, self.cols[k].ctypes.data)
        if narrow:
            nr = self.narrow()
            if "span16" in nr:
                b.span16 = nr["span16"].ctypes.data; b.endpos = None
            if "isize16" in nr:
                b.isize16 = nr["isize16"].ctypes.data; b.isize = None
            if "tid_run_start" in nr:
                b.n_tid_runs = int(nr["tid_run_start"].shape[0]); b.tid_run_start = nr["tid_run_start"].ctypes.data
                b.tid_run_tid = nr["tid_run_tid"].ctypes.data; b.tid = None
        b.n_x = self.n_x
        for k, _ in _XCOLS:
            setattr(b, k, self.x[k].ctypes.data)
        b.n_sa = self.n_sa
        for k, _ in _SIDE:
            setattr(b, k, self.side[k].ctypes.data)
        if self.seq is not None:
            for k, _ in _SEQ:
                setattr(b, k, self.seq[k].ctypes.data)
        return b

    def header(self) -> Header:
        h = Header()
        h.n_targets = len(self.target_names)
        h.target_len = self.target_len.ctypes.data_as(C.POINTER(C.c_uint32))
        self._name_arr = (C.c_char_p * len(self.target_names))(*[s.encode() for s in self.target_names])
        h.target_name = C.cast(self._name_arr, C.POINTER(C.c_char_p))
        return h

    def nbytes(self) -> int:
        return sum(self.cols[k].nbytes for k, _ in _COLS) + sum(a.nbytes for a in self.x.values()) + sum(a.nbytes for a in self.side.values())

    # -- constructors ----------------------------------------------------------------------
    @staticmethod
    def from_synth(d, target_names=None) -> "HostBatch":
        """target_names: the header name of every tid (default synth.chrom_name)"""
        from . import synth
        cols = {k: d.cols[k].cpu().numpy() for k in ("mapq", "tid", "pos", "mtid", "mpos", "isize", "endpos")}
        cols["flag"] = d.cols["flag"].cpu().numpy().view(np.uint16)
        nh = synth.name_hash_ids(d.cols["name_id"]).cpu().numpy().view(np.uint64).reshape(-1)
        side = {"sa_rec": d.sa_rec.cpu().numpy(), "cig_off": d.cig_off.cpu().numpy(),
                "cig_ops": d.cig_ops.cpu().numpy(), "sa_off": d.sa_off.cpu().numpy(),
                "sa_txt": d.sa_txt.cpu().numpy()}
        names = [synth.chrom_name(t) for t in range(len(d.cfg.chrom_lens))] if target_names is None else list(target_names)
        return HostBatch(cols, nh, side, d.cfg.chrom_lens, names)

    @staticmethod
    def from_bam(path: str, threads: int = 8) -> "HostBatch":
        lib = host_lib()
        err = C.create_string_buffer(256)
        h = lib.bkid_host_read_bam(path.encode(), threads, err, 256)
        if not h:
            raise IOError("bkid_host_read_bam: " + err.value.decode())
        try:
            b = C.cast(lib.bkid_host_bam_batch(h), C.POINTER(Batch)).contents
            hd = C.cast(lib.bkid_host_bam_header(h), C.POINTER(Header)).contents
            n, n_sa = int(b.n), int(b.n_sa)

            def arr(ptr, count, dt):
                if count == 0:
                    return np.zeros(0, dt)
                return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), (count * np.dtype(dt).itemsize,)).view(dt).copy()

            cols = {k: arr(getattr(b, k), n, dt) for k, dt in _COLS}
            n_x = int(b.n_x)
            xr = arr(b.x_rec, n_x, np.uint32).astype(np.int64)
            for k in ("mtid", "mpos"):
                cols[k] = np.zeros(n, np.int32)
                cols[k][xr] = arr(getattr(b, "x_" + k), n_x, np.int32)
            nh2 = np.zeros((n, 2), np.uint64)
            nh2[xr] = arr(b.x_name_hash, 2 * n_x, np.uint64).reshape(-1, 2)
            nh = nh2.reshape(-1)
            cig_off = arr(b.cig_off, n_sa + 1, np.uint32)
            sa_off = arr(b.sa_off, n_sa + 1, np.uint32)
            oc_off = arr(b.oc_off, n_sa + 1, np.uint32)
            side = {"sa_rec": arr(b.sa_rec, n_sa, np.uint32), "cig_off": cig_off,
                    "cig_ops": arr(b.cig_ops, int(cig_off[-1]), np.uint32), "sa_off": sa_off,
                    "sa_txt": arr(b.sa_txt, int(sa_off[-1]), np.uint8), "oc_off": oc_off,
                    "oc_txt": arr(b.oc_txt, int(oc_off[-1]), np.uint8)}
            if b.seq_off:
                seq_off = arr(b.seq_off, n_sa + 1, np.uint32)
                side.update({"seq_off": seq_off, "seq4": arr(b.seq4, int(seq_off[-1]), np.uint8), "seq_len": arr(b.seq_len, n_sa, np.int32)})
            tl = [int(hd.target_len[i]) for i in range(hd.n_targets)]
            names = [hd.target_name[i].decode() for i in range(hd.n_targets)]
        finally:
            lib.bkid_host_bam_free(h)
        return HostBatch(cols, nh, side, tl, names)


_host = None
_cuda = None


def host_lib():
    global _host
    if _host is None:
        if not os.path.exists(LIB_HOST):
            raise RuntimeError("host library missing: %s (run __graft_entry__.build())" % LIB_HOST)
        L = C.CDLL(LIB_HOST)
        L.bkid_host_read_bam.restype = C.c_void_p
        L.bkid_host_read_bam.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int]
        L.bkid_host_bam_header.restype = C.c_void_p
        L.bkid_host_bam_header.argtypes = [C.c_void_p]
        L.bkid_host_bam_batch.restype = C.c_void_p
        L.bkid_host_bam_batch.argtypes = [C.c_void_p]
        L.bkid_host_bam_free.argtypes = [C.c_void_p]
        L.bkid_host_bam_batch_narrow.restype = C.c_void_p
        L.bkid_host_bam_batch_narrow.argtypes = [C.c_void_p]
        L.bkid_host_bgzf_open.restype = C.c_void_p
        L.bkid_host_bgzf_open.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        for f, rt in (("header", C.c_void_p), ("data", C.c_void_p), ("size", C.c_uint64), ("blocks", C.c_void_p), ("n_blocks", C.c_int64),
                      ("first_record", C.c_uint64), ("usize", C.c_uint64), ("first_l_qseq", C.c_int32)):
            fn = getattr(L, "bkid_host_bgzf_" + f)
            fn.restype = rt
            fn.argtypes = [C.c_void_p]
        L.bkid_host_bgzf_close.argtypes = [C.c_void_p]
        L.bkid_host_sam_open.restype = C.c_void_p
        L.bkid_host_sam_open.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        L.bkid_host_sam_parse.restype = C.c_void_p
        L.bkid_host_sam_parse.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p, C.c_int]
        for f, rt in (("header", C.c_void_p), ("data", C.c_void_p), ("size", C.c_uint64), ("first_record", C.c_uint64), ("first_line", C.c_int64)):
            fn = getattr(L, "bkid_host_sam_" + f)
            fn.restype = rt
            fn.argtypes = [C.c_void_p]
        L.bkid_host_sam_close.argtypes = [C.c_void_p]
        _host = L
    return _host


EXPORTS = ["bkid_abi_version", "bkid_last_error", "bkid_default_params", "bkid_create", "bkid_destroy",
           "bkid_reserve", "bkid_push_batch", "bkid_push_batch_device", "bkid_reset", "bkid_insert_stats",
           "bkid_scan", "bkid_cluster", "bkid_set_nib", "bkid_refine", "bkid_run", "bkid_fetch_clusters",
           "bkid_fetch_pairs", "bkid_fetch_class", "bkid_get_timings", "bkid_op_sort_perm",
           "bkid_op_remove_isolated", "bkid_op_cluster",
           "bkid_shard_insert_partial", "bkid_sd_upper_binade", "bkid_shard_sd_fast", "bkid_shard_sd_fast_collect", "bkid_shard_sd_prepare", "bkid_shard_sd_partial", "bkid_shard_set_stats", "bkid_shard_candidates", "bkid_shard_join",
           "bkid_shard_set_pairs", "bkid_shard_clusters", "bkid_shard_set_clusters", "bkid_shard_sa_rows", "bkid_shard_set_sa_rows",
           "bkid_shard_maxspan", "bkid_shard_set_maxspan", "bkid_shard_coverage", "bkid_shard_vote", "bkid_shard_depth",
           "bkid_shard_finish", "bkid_fetch_bucket_ranks", "bkid_device_copy",
           "bkid_push_bgzf", "bkid_push_bgzf_range", "bkid_get_decode_stats", "bkid_fetch_column", "bkid_set_exclude", "bkid_device_gather_rows", "bkid_op_banded_align", "bkid_profile_kernels", "bkid_profile_report",
           "bkid_comm_nccl_unique_id", "bkid_comm_nccl_init", "bkid_comm_nccl_init_all", "bkid_comm_local_create", "bkid_comm_destroy", "bkid_dist_run", "bkid_dist_run_threads",
           "bkid_op_summarize", "bkid_set_params", "bkid_lpt_owner_table", "bkid_sort_records", "bkid_push_sam"]

CAND_BYTES = 48
SAROW_BYTES = 88


def cuda_lib():
    """Load libbreakid_b200.so.  Raises (never falls back) when it has not been built."""
    global _cuda
    if _cuda is None:
        if not os.path.exists(LIB_CUDA):
            raise RuntimeError("CUDA library missing: %s (run __graft_entry__.build()); there is no CPU fallback" % LIB_CUDA)
        L = C.CDLL(LIB_CUDA)
        vp, i64p = C.c_void_p, C.POINTER(C.c_int64)
        dp = C.POINTER(C.c_double)
        L.bkid_abi_version.restype = C.c_int
        L.bkid_last_error.restype = C.c_char_p
        L.bkid_last_error.argtypes = [vp]
        L.bkid_default_params.argtypes = [C.POINTER(Params)]
        L.bkid_create.restype = vp
        L.bkid_create.argtypes = [C.c_int, C.POINTER(Header), C.POINTER(Params)]
        L.bkid_destroy.argtypes = [vp]
        L.bkid_reserve.argtypes = [vp] + [C.c_int64] * 6
        L.bkid_push_batch.argtypes = [vp, C.POINTER(Batch)]
        L.bkid_push_batch_device.argtypes = [vp, C.POINTER(Batch)]
        L.bkid_set_exclude.argtypes = [vp, C.c_int64, vp, vp, vp]
        L.bkid_op_banded_align.argtypes = [vp, C.c_int64, vp, vp, vp, vp, C.c_int32, vp]
        L.bkid_device_gather_rows.argtypes = [vp, vp, vp, vp, C.c_int64, C.c_int32]
        L.bkid_push_bgzf.argtypes = [vp, vp, C.c_uint64, vp, C.c_int64, C.c_uint64, C.POINTER(C.c_int64)]
        L.bkid_push_bgzf_range.argtypes = [vp, vp, C.c_uint64, vp, C.c_int64, C.c_uint64, C.c_int64, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.bkid_get_decode_stats.argtypes = [vp, C.POINTER(DecodeStats)]
        L.bkid_push_sam.argtypes = [vp, vp, C.c_uint64, C.c_int64, C.POINTER(C.c_int64)]
        L.bkid_fetch_column.argtypes = [vp, C.c_char_p, vp, C.c_int64, C.POINTER(C.c_int64)]
        L.bkid_reset.argtypes = [vp]
        L.bkid_sort_records.argtypes = [vp, C.POINTER(C.c_int32)]
        L.bkid_insert_stats.argtypes = [vp, dp, dp]
        L.bkid_scan.argtypes = [vp, C.c_double, i64p]
        L.bkid_cluster.argtypes = [vp, C.c_double, C.c_int, i64p]
        L.bkid_set_nib.argtypes = [vp, C.c_int32, vp, C.c_uint64]
        L.bkid_refine.argtypes = [vp, C.c_double, i64p]
        L.bkid_run.argtypes = [vp, dp, dp, dp, i64p]
        L.bkid_fetch_clusters.argtypes = [vp, vp, C.c_int64, i64p]
        L.bkid_fetch_pairs.argtypes = [vp, C.c_int, vp, C.c_int64, i64p]
        L.bkid_fetch_class.argtypes = [vp, vp, C.c_int64]
        L.bkid_get_timings.argtypes = [vp, C.POINTER(Timings)]
        L.bkid_op_sort_perm.argtypes = [vp, C.c_int64, vp, vp]
        L.bkid_op_remove_isolated.argtypes = [vp, C.c_int64, vp, vp, C.c_double, vp, i64p]
        L.bkid_op_cluster.argtypes = [vp, C.c_int, C.c_int64, vp, vp, C.c_double, vp, vp, i64p, C.POINTER(C.c_int32)]
        L.bkid_op_summarize.argtypes = [vp, C.c_int64, vp, C.c_double, i64p]
        L.bkid_set_params.argtypes = [vp, vp]
        L.bkid_lpt_owner_table.argtypes = [vp, C.c_int, C.c_int, vp]
        pvp = C.POINTER(C.c_void_p)
        u64p = C.POINTER(C.c_uint64)
        L.bkid_shard_insert_partial.argtypes = [vp, i64p, i64p, u64p, u64p]
        L.bkid_sd_upper_binade.argtypes = [C.c_uint64] * 4
        L.bkid_sd_upper_binade.restype = C.c_int
        L.bkid_shard_sd_fast.argtypes = [vp, C.c_double, C.c_int32]
        L.bkid_shard_sd_fast_collect.argtypes = [vp, u64p, u64p]
        L.bkid_shard_sd_prepare.argtypes = [vp, C.c_double]
        L.bkid_shard_sd_partial.argtypes = [vp, C.c_double, C.c_int64, i64p]
        L.bkid_shard_set_stats.argtypes = [vp, C.c_double, C.c_double]
        L.bkid_shard_candidates.argtypes = [vp, C.c_uint64, pvp, i64p]
        L.bkid_shard_join.argtypes = [vp, vp, C.c_int64, C.c_double, pvp, i64p]
        L.bkid_shard_set_pairs.argtypes = [vp, vp, C.c_int64]
        L.bkid_shard_clusters.argtypes = [vp, pvp, i64p]
        L.bkid_shard_set_clusters.argtypes = [vp, vp, C.c_int64]
        L.bkid_shard_sa_rows.argtypes = [vp, pvp, i64p]
        L.bkid_shard_set_sa_rows.argtypes = [vp, vp, C.c_int64]
        L.bkid_shard_maxspan.argtypes = [vp, C.POINTER(C.c_int32)]
        L.bkid_shard_set_maxspan.argtypes = [vp, C.c_int32]
        L.bkid_shard_coverage.argtypes = [vp, C.c_double, pvp, i64p]
        L.bkid_shard_vote.argtypes = [vp]
        L.bkid_shard_depth.argtypes = [vp, pvp, i64p]
        L.bkid_shard_finish.argtypes = [vp, i64p]
        L.bkid_fetch_bucket_ranks.argtypes = [vp, vp, C.c_int64, i64p]
        L.bkid_device_copy.argtypes = [vp, vp, vp, C.c_uint64]
        L.bkid_comm_nccl_unique_id.argtypes = [vp]
        L.bkid_comm_nccl_init.restype = vp
        L.bkid_comm_nccl_init.argtypes = [vp, C.c_int, C.c_int, C.c_int]
        L.bkid_comm_nccl_init_all.argtypes = [vp, C.c_int, vp]
        L.bkid_comm_local_create.argtypes = [C.c_int, vp]
        L.bkid_comm_destroy.argtypes = [vp]
        L.bkid_dist_run.argtypes = [vp, vp, C.c_int, dp, dp, dp, i64p, C.POINTER(C.c_float)]
        L.bkid_dist_run_threads.argtypes = [vp, vp, C.c_int, C.c_int, dp, dp, dp, i64p]
        L.bkid_profile_kernels.argtypes = [C.c_int]
        L.bkid_profile_report.argtypes = [C.c_char_p, C.c_int64]
        L.bkid_profile_report.restype = C.c_int64
        _cuda = L
    return _cuda


class BkidError(RuntimeError):
    pass


def dist_run_local(ctxs: Sequence["Context"], mode: int = 0):
    """the sharded hot path with the exchanges inside the library, every rank a host thread of this process
    (``bkid_comm_local_create`` + ``bkid_dist_run_threads``): contexts may share one device.  ctxs[r] holds the r-th slice
    of the coordinate-sorted stream.  Returns [(mean, sd, dist, n_called)] per rank; fetch the calls from any context."""
    L = cuda_lib()
    W = len(ctxs)
    comms = (C.c_void_p * W)()
    rc = L.bkid_comm_local_create(W, comms)
    if rc:
        raise BkidError("bkid_comm_local_create failed: %d" % rc)
    try:
        cp = (C.c_void_p * W)(*[c.ctx for c in ctxs])
        m, s, d = (C.c_double * W)(), (C.c_double * W)(), (C.c_double * W)()
        n = (C.c_int64 * W)()
        rc = L.bkid_dist_run_threads(cp, comms, W, mode, m, s, d, n)
        if rc:
            msgs = [(L.bkid_last_error(c.ctx) or b"").decode() for c in ctxs]
            raise BkidError("bkid_dist_run_threads: error %d: %s" % (rc, "; ".join(x for x in msgs if x)))
        return [(m[r], s[r], d[r], n[r]) for r in range(W)]
    finally:
        for r in range(W):
            L.bkid_comm_destroy(comms[r])


def profile_kernels(on: bool):
    """switch the per-kernel CUDA-event timing of the library on / off (bkid_profile_kernels)"""
    cuda_lib().bkid_profile_kernels(1 if on else 0)


def profile_report() -> dict:
    """{kernel name: (launches, milliseconds)} of everything launched since profiling was switched on (and reset)"""
    L = cuda_lib()
    buf = C.create_string_buffer(1 << 16)
    L.bkid_profile_report(buf, len(buf))
    out = {}
    for line in buf.value.decode().splitlines():
        nm, n, ms = line.split("\t")
        out[nm] = (int(n), float(ms))
    return out


class BgzfBlock(C.Structure):
    _fields_ = [("payload_off", C.c_uint64), ("payload_len", C.c_uint32), ("usize", C.c_uint32)]


class DecodeStats(C.Structure):
    _fields_ = [("n_chunks", C.c_int64), ("n_blocks", C.c_int64), ("compressed_bytes", C.c_int64), ("uncompressed_bytes", C.c_int64),
                ("n_records", C.c_int64), ("total_ms", C.c_float), ("inflate_ms", C.c_float), ("boundaries_ms", C.c_float),
                ("extract_ms", C.c_float), ("seed_repairs", C.c_int32), ("reserved", C.c_int32)]


class BgzfFile:
    """Host half of the device decode path: mapped BAM file + BGZF block table + parsed BAM header
    (``bkid_host_bgzf_open``, breakid_b200/host/bam_reader.h)."""

    def __init__(self, path: str):
        self.lib = host_lib()
        err = C.create_string_buffer(256)
        self.h = self.lib.bkid_host_bgzf_open(path.encode(), err, 256)
        if not self.h:
            raise IOError("bkid_host_bgzf_open: " + err.value.decode())
        hd = C.cast(self.lib.bkid_host_bgzf_header(self.h), C.POINTER(Header)).contents
        self.target_len = [int(hd.target_len[i]) for i in range(hd.n_targets)]
        self.target_names = [hd.target_name[i].decode() for i in range(hd.n_targets)]
        self.data = self.lib.bkid_host_bgzf_data(self.h)
        self.size = int(self.lib.bkid_host_bgzf_size(self.h))
        self.blocks = self.lib.bkid_host_bgzf_blocks(self.h)
        self.n_blocks = int(self.lib.bkid_host_bgzf_n_blocks(self.h))
        self.first_record = int(self.lib.bkid_host_bgzf_first_record(self.h))
        self.usize = int(self.lib.bkid_host_bgzf_usize(self.h))

    def block_table(self) -> np.ndarray:
        dt = np.dtype([("payload_off", np.uint64), ("payload_len", np.uint32), ("usize", np.uint32)])
        return np.ctypeslib.as_array(C.cast(self.blocks, C.POINTER(C.c_uint8)), (self.n_blocks * 16,)).view(dt).copy()

    def close(self):
        if self.h:
            self.lib.bkid_host_bgzf_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SamFile:
    """Host half of the SAM path: mapped SAM file (or a header in a caller's buffer) + the target table of its @SQ
    lines (``bkid_host_sam_open`` / ``bkid_host_sam_parse``, breakid_b200/host/bam_reader.h).  ``text`` is a view of the
    alignment lines, which start on file line ``first_line``."""

    def __init__(self, path: Optional[str] = None, buf: Optional[bytes] = None):
        self.lib = host_lib()
        err = C.create_string_buffer(256)
        self._buf = None
        if buf is not None:
            self._buf = C.create_string_buffer(bytes(buf), len(buf))
            self.h = self.lib.bkid_host_sam_parse(C.cast(self._buf, C.c_void_p), len(buf), err, 256)
        else:
            self.h = self.lib.bkid_host_sam_open(path.encode(), err, 256)
        if not self.h:
            raise IOError("SAM header: " + err.value.decode())
        hd = C.cast(self.lib.bkid_host_sam_header(self.h), C.POINTER(Header)).contents
        self.target_len = [int(hd.target_len[i]) for i in range(hd.n_targets)]
        self.target_names = [hd.target_name[i].decode() for i in range(hd.n_targets)]
        self.data = self.lib.bkid_host_sam_data(self.h)
        self.size = int(self.lib.bkid_host_sam_size(self.h))
        self.first_record = int(self.lib.bkid_host_sam_first_record(self.h))
        self.first_line = int(self.lib.bkid_host_sam_first_line(self.h))

    def text(self) -> bytes:
        return C.string_at(self.data + self.first_record, self.size - self.first_record) if self.size > self.first_record else b""

    def close(self):
        if self.h:
            self.lib.bkid_host_sam_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One device context (``bkid_ctx``)."""

    def __init__(self, target_len: Sequence[int], target_names: Sequence[str], device: int = 0, **params):
        self.lib = cuda_lib()
        self._tl = np.ascontiguousarray(target_len, dtype=np.uint32)
        self._names = (C.c_char_p * len(target_names))(*[s.encode() for s in target_names])
        h = Header(len(target_names), self._tl.ctypes.data_as(C.POINTER(C.c_uint32)), C.cast(self._names, C.POINTER(C.c_char_p)))
        p = Params()
        self.lib.bkid_default_params(C.byref(p))
        for k, v in params.items():
            setattr(p, k, int(v))
        self.params = p
        self.ctx = self.lib.bkid_create(device, C.byref(h), C.byref(p))
        if not self.ctx:
            raise BkidError("bkid_create failed: " + (self.lib.bkid_last_error(None) or b"?").decode())

    def _chk(self, rc):
        if rc != 0:
            raise BkidError("bkid error %d: %s" % (rc, (self.lib.bkid_last_error(self.ctx) or b"").decode()))

    def close(self):
        if self.ctx:
            self.lib.bkid_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reserve(self, n, n_x=0, n_sa=0, n_cig=0, sa_bytes=0, oc_bytes=0):
        self._chk(self.lib.bkid_reserve(self.ctx, n, n_x, n_sa, n_cig, sa_bytes, oc_bytes))

    def push(self, hb: HostBatch, narrow: bool = True):
        b = hb.struct(narrow)
        self._chk(self.lib.bkid_push_batch(self.ctx, C.byref(b)))

    def op_banded_align(self, queries: Sequence[bytes], refs: Sequence[bytes], w: int) -> np.ndarray:
        """banded edit distance of queries[i] against refs[i] (extension, bkid_op_banded_align)"""
        n = len(queries)
        q = np.frombuffer(b"".join(queries) + b"\0", np.uint8).copy()
        r = np.frombuffer(b"".join(refs) + b"\0", np.uint8).copy()
        qo = np.concatenate([[0], np.cumsum([len(x) for x in queries])]).astype(np.uint32)
        ro = np.concatenate([[0], np.cumsum([len(x) for x in refs])]).astype(np.uint32)
        out = np.zeros(max(n, 1), np.int32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        self._chk(self.lib.bkid_op_banded_align(self.ctx, n, p(q), p(qo), p(r), p(ro), int(w), p(out)))
        return out[:n]

    def push_bgzf(self, f: "BgzfFile", data_ptr=None, blocks=None, n_blocks=None, first_record=None) -> int:
        """device BGZF inflate + BAM decode of a whole file (``bkid_push_bgzf``); returns the record count.
        ``data_ptr`` overrides the mapped file with another host copy of the same bytes (e.g. a pinned buffer)."""
        n = C.c_int64()
        self._chk(self.lib.bkid_push_bgzf(self.ctx, C.c_void_p(data_ptr if data_ptr is not None else f.data), f.size,
                                          C.c_void_p(blocks if blocks is not None else f.blocks),
                                          f.n_blocks if n_blocks is None else n_blocks,
                                          f.first_record if first_record is None else first_record, C.byref(n)))
        return int(n.value)

    def push_bgzf_range(self, f: "BgzfFile", first_block: int, end_block: int, data_ptr=None):
        """device decode of the records that start inside blocks [first_block, end_block) (``bkid_push_bgzf_range``);
        returns (n_records, stream offset of the first decoded record, stream offset of the next range's first record)"""
        n, a, b = C.c_int64(), C.c_uint64(), C.c_uint64()
        self._chk(self.lib.bkid_push_bgzf_range(self.ctx, C.c_void_p(data_ptr if data_ptr is not None else f.data), f.size, C.c_void_p(f.blocks), f.n_blocks,
                                                f.first_record, first_block, end_block, C.byref(n), C.byref(a), C.byref(b)))
        return int(n.value), int(a.value), int(b.value)

    def push_sam(self, text, first_line: int = 1, data_ptr=None, size=None) -> int:
        """device parse of SAM alignment lines (``bkid_push_sam``); returns the record count.  ``text`` is bytes (its
        lines start on file line ``first_line``) or a ``SamFile`` (its alignment lines, numbered from the file).
        ``data_ptr`` / ``size`` push that host memory instead (e.g. a pinned copy of the text)."""
        n = C.c_int64()
        if isinstance(text, SamFile):
            ptr, ln, first_line = text.data + text.first_record, text.size - text.first_record, text.first_line
            keep = text
        else:
            keep = C.create_string_buffer(bytes(text), len(text)) if data_ptr is None else None
            ptr, ln = (C.cast(keep, C.c_void_p).value, len(text)) if data_ptr is None else (data_ptr, size)
        self._chk(self.lib.bkid_push_sam(self.ctx, C.c_void_p(ptr), ln, first_line, C.byref(n)))
        del keep
        return int(n.value)

    def decode_stats(self) -> dict:
        s = DecodeStats()
        self._chk(self.lib.bkid_get_decode_stats(self.ctx, C.byref(s)))
        return {k: getattr(s, k) for k, _ in DecodeStats._fields_ if k != "reserved"}

    def fetch_column(self, name: str, dtype) -> np.ndarray:
        nb = C.c_int64()
        self._chk(self.lib.bkid_fetch_column(self.ctx, name.encode(), None, 0, C.byref(nb)))
        out = np.zeros(int(nb.value) // np.dtype(dtype).itemsize, dtype)
        if nb.value:
            self._chk(self.lib.bkid_fetch_column(self.ctx, name.encode(), out.ctypes.data_as(C.c_void_p), int(nb.value), C.byref(nb)))
        return out

    def set_exclude(self, tid, beg, end):
        """exclude intervals [beg, end) on target tid (extension, see include/breakid_b200.h: bkid_set_exclude)"""
        t = np.ascontiguousarray(tid, np.int32); b = np.ascontiguousarray(beg, np.int32); e = np.ascontiguousarray(end, np.int32)
        self._chk(self.lib.bkid_set_exclude(self.ctx, int(t.shape[0]), t.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), e.ctypes.data_as(C.c_void_p)))

    def push_device(self, b: Batch):
        self._chk(self.lib.bkid_push_batch_device(self.ctx, C.byref(b)))

    def reset(self):
        self._chk(self.lib.bkid_reset(self.ctx))

    def sort_records(self) -> bool:
        """coordinate-sort the records pushed so far on the device (``bkid_sort_records``); True when they already were
        in order (nothing moved)"""
        w = C.c_int32()
        self._chk(self.lib.bkid_sort_records(self.ctx, C.byref(w)))
        return bool(w.value)

    def insert_stats(self):
        m, s = C.c_double(), C.c_double()
        self._chk(self.lib.bkid_insert_stats(self.ctx, C.byref(m), C.byref(s)))
        return m.value, s.value

    def scan(self, w: float) -> int:
        n = C.c_int64()
        self._chk(self.lib.bkid_scan(self.ctx, w, C.byref(n)))
        return n.value

    def cluster(self, dist: float, mode: int = 0) -> int:
        n = C.c_int64()
        self._chk(self.lib.bkid_cluster(self.ctx, dist, mode, C.byref(n)))
        return n.value

    def set_nib(self, tid: int, packed: np.ndarray, n_bases: int):
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        self._chk(self.lib.bkid_set_nib(self.ctx, tid, packed.ctypes.data, n_bases))

    def refine(self, dist: float) -> int:
        n = C.c_int64()
        self._chk(self.lib.bkid_refine(self.ctx, dist, C.byref(n)))
        return n.value

    def run(self):
        m, s, d, n = C.c_double(), C.c_double(), C.c_double(), C.c_int64()
        self._chk(self.lib.bkid_run(self.ctx, C.byref(m), C.byref(s), C.byref(d), C.byref(n)))
        return m.value, s.value, d.value, n.value

    def fetch_clusters(self) -> np.ndarray:
        n = C.c_int64()
        self._chk(self.lib.bkid_fetch_clusters(self.ctx, None, 0, C.byref(n)))
        out = np.zeros(max(1, n.value), CLUSTER_DTYPE)
        self._chk(self.lib.bkid_fetch_clusters(self.ctx, out.ctypes.data, out.shape[0], C.byref(n)))
        return out[:n.value]

    def fetch_pairs(self, stage: int) -> np.ndarray:
        n = C.c_int64()
        self._chk(self.lib.bkid_fetch_pairs(self.ctx, stage, None, 0, C.byref(n)))
        out = np.zeros(max(1, n.value), PAIR_DTYPE)
        self._chk(self.lib.bkid_fetch_pairs(self.ctx, stage, out.ctypes.data, out.shape[0], C.byref(n)))
        return out[:n.value]

    def fetch_class(self, n: int) -> np.ndarray:
        out = np.zeros(n, np.uint8)
        self._chk(self.lib.bkid_fetch_class(self.ctx, out.ctypes.data, n))
        return out

    def timings(self) -> dict:
        t = Timings()
        self._chk(self.lib.bkid_get_timings(self.ctx, C.byref(t)))
        return {k: getattr(t, k) for k in TIMING_FIELDS_F + TIMING_FIELDS_I}

    # stand-alone operators
    def op_sort_perm(self, key: np.ndarray) -> np.ndarray:
        key = np.ascontiguousarray(key, np.uint32)
        perm = np.zeros(key.shape[0], np.uint32)
        self._chk(self.lib.bkid_op_sort_perm(self.ctx, key.shape[0], key.ctypes.data, perm.ctypes.data))
        return perm

    def op_remove_isolated(self, p1, p2, w):
        p1 = np.ascontiguousarray(p1, np.uint32); p2 = np.ascontiguousarray(p2, np.uint32)
        out = np.zeros(p1.shape[0] + 2, np.uint32)
        n = C.c_int64()
        self._chk(self.lib.bkid_op_remove_isolated(self.ctx, p1.shape[0], p1.ctypes.data, p2.ctypes.data, w, out.ctypes.data, C.byref(n)))
        return out[:n.value]

    def set_params(self, **kw):
        """replace thresholds for the next stage calls (``bkid_set_params``); unknown names raise"""
        p = Params()
        for k, _ in Params._fields_:
            setattr(p, k, getattr(self.params, k))
        for k, v in kw.items():
            if k not in dict(Params._fields_):
                raise KeyError(k)
            setattr(p, k, int(v))
        self._chk(self.lib.bkid_set_params(self.ctx, C.byref(p)))
        self.params = p

    def op_summarize(self, pairs: np.ndarray, dist: float) -> int:
        """K6 on the pairs of one bucket (PAIR_DTYPE rows grouped by ascending ``cluster``): leaves the summaries in the context,
        ``refine`` + ``fetch_clusters`` then give the bucket's calls (``bkid_op_summarize``)"""
        pairs = np.ascontiguousarray(pairs, PAIR_DTYPE)
        n = C.c_int64()
        self._chk(self.lib.bkid_op_summarize(self.ctx, pairs.shape[0], pairs.ctypes.data, dist, C.byref(n)))
        return n.value

    def op_cluster(self, mode, p1, p2, thr):
        p1 = np.ascontiguousarray(p1, np.uint32); p2 = np.ascontiguousarray(p2, np.uint32)
        oi = np.zeros(p1.shape[0] + 2, np.uint32); oc = np.zeros(p1.shape[0] + 2, np.int32)
        n = C.c_int64(); r = C.c_int32()
        self._chk(self.lib.bkid_op_cluster(self.ctx, mode, p1.shape[0], p1.ctypes.data, p2.ctypes.data, thr,
                                           oi.ctypes.data, oc.ctypes.data, C.byref(n), C.byref(r)))
        return oi[:n.value], oc[:n.value], r.value
