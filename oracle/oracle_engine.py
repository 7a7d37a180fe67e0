"""TEST INFRASTRUCTURE: a per-rank engine for breakid_b200.dist.run_sharded built on the CPU oracle
(oracle/liboracle.so orc_shard_*).  Lets the multi-rank host logic (routing, ordering, partial-count
reductions) run under gloo on CPU and be compared with orc_run on the unsplit input."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

import oracle_py as O
from breakid_b200.api import CLUSTER_DTYPE, PAIR_DTYPE

L, D, I = C.c_long, C.c_double, C.c_int
u8p, u16p, u32p, i32p, u64p = O.u8p, O.u16p, O.u32p, O.i32p, O.u64p
vp = C.c_void_p


def _lib():
    o = O.olib()
    if not hasattr(o, "_shard_ready"):
        o.orc_shard_sd_partial.restype = L
        o.orc_shard_sd_partial.argtypes = [L, u16p, i32p, D, L]
        o.orc_shard_candidates.restype = L
        o.orc_shard_candidates.argtypes = [L, u16p, u8p, i32p, i32p, i32p, i32p, u64p, L, C.c_uint64, C.POINTER(vp)]
        o.orc_shard_join.restype = L
        o.orc_shard_join.argtypes = [L, vp, I, u32p, i32p, D, C.POINTER(vp)]
        o.orc_shard_bucket_clusters.restype = L
        o.orc_shard_bucket_clusters.argtypes = [L, vp, D, I, C.POINTER(vp)]
        o.orc_shard_sa_rows.argtypes = [L, u16p, u8p, i32p, i32p, i32p, u64p, L, u32p, u32p, u32p, u32p, u8p, u32p, u8p, vp]
        o.orc_shard_coverage.argtypes = [L, u16p, u8p, i32p, i32p, i32p, L, vp, D, u32p]
        o.orc_shard_vote.restype = L
        o.orc_shard_vote.argtypes = [L, vp, L, vp, u32p, I, C.POINTER(C.c_char_p), D, u32p]
        o.orc_shard_depth.argtypes = [L, u16p, u8p, i32p, i32p, i32p, L, vp, u32p, u32p]
        o.orc_shard_finish.restype = L
        o.orc_shard_finish.argtypes = [L, vp, u32p, u32p, C.POINTER(vp), C.POINTER(C.c_uint64)]
        o._shard_ready = True
    return o


def _bytes_tensor(ptr, n, row, free):
    out = np.zeros((n, row), np.uint8)
    if n:
        C.memmove(out.ctypes.data, ptr, n * row)
    free(ptr)
    return torch.from_numpy(out)


class OracleEngine:
    device = torch.device("cpu")

    def __init__(self, hb, nibs=None, qual=20, ahc_model=False):
        """ahc_model: cluster() runs the component model of AHC instead of the literal O(N^3) form (see O.ahc_model)"""
        self.hb, self.nibs, self.qual, self.ahc_model = hb, nibs, qual, ahc_model
        self.o = _lib()
        self.rank_table = np.zeros((len(hb.target_names) + 1) ** 2, np.int32)
        self.o.orc_bucket_rank_table(len(hb.target_names), O._names(hb), self.rank_table)

    def _insert_x(self):
        f = self.hb.cols["flag"].astype(np.int64); s = self.hb.cols["isize"].astype(np.int64)
        ok = ((f & 1) != 0) & ((f & 2) != 0) & ((f & (0x4 | 0x100 | 0x200 | 0x400)) == 0)
        return np.abs(s[ok])

    def insert_partial(self):
        x = self._insert_x()
        xu = x.astype(np.uint64)
        return int(x.sum()), int(x.shape[0]), int((xu * xu).sum(dtype=np.uint64)), int(x.max(initial=0))       # uint64 wrap-around like the device

    def sd_fast(self, mean, kub):
        """CPU restatement of the one-pass sd form: sum floor(a) and the number of elements whose fraction could round
        the accumulator up below binade kub (a = (|isize| - mean)^2 in IEEE double, like src/BreakID.cc:1944)"""
        x = self._insert_x().astype(np.float64)
        d = x - mean
        a = d * d
        fl = np.floor(a)
        self._sdf = (int(fl.astype(object).sum()) if x.shape[0] else 0, int(((a - fl) >= 1.0 - 2.0 ** (kub - 53)).sum()) if kub < 51 else 1 << 40)

    def sd_fast_collect(self):
        return self._sdf

    def sd_partial(self, mean, t_in):
        return self.o.orc_shard_sd_partial(self.hb.n, self.hb.cols["flag"], self.hb.cols["isize"], mean, t_in)

    def set_stats(self, mean, sd):
        pass

    def candidates(self, offset):
        c = self.hb.cols
        out = vp()
        n = self.o.orc_shard_candidates(self.hb.n, c["flag"], c["mapq"], c["tid"], c["pos"], c["mtid"], c["mpos"], self.hb.name_hash, self.qual, offset, C.byref(out))
        return _bytes_tensor(out, n, 48, self.o.orc_free)

    def join(self, cands, w):
        a = np.ascontiguousarray(cands.numpy())
        out = vp()
        n = self.o.orc_shard_join(a.shape[0], a.ctypes.data, len(self.hb.target_names), self.hb.target_len, self.rank_table, w, C.byref(out))
        return _bytes_tensor(out, n, 64, self.o.orc_free)

    def set_pairs(self, pairs):
        p = np.ascontiguousarray(pairs.numpy()).view(PAIR_DTYPE).reshape(-1)
        key = (p["bucket"].astype(np.uint64) << np.uint64(40)) | (p["_pad"].astype(np.uint64) << np.uint64(32)) | p["orig"].astype(np.uint64)
        self.pairs = np.ascontiguousarray(p[np.argsort(key, kind="stable")])

    def bucket_ranks(self):
        return torch.from_numpy(np.unique(self.pairs["bucket"]).astype(np.int32))

    def cluster(self, d, mode):
        out = vp()
        self.o.orc_set_ahc_model(1 if self.ahc_model else 0)
        try:
            n = self.o.orc_shard_bucket_clusters(self.pairs.shape[0], self.pairs.ctypes.data, d, mode, C.byref(out))
        finally:
            self.o.orc_set_ahc_model(0)
        self._cl = _bytes_tensor(out, n, 192, self.o.orc_free)

    def clusters(self):
        return self._cl

    def set_clusters(self, t):
        self.cl = np.ascontiguousarray(t.numpy()).copy()

    def sa_rows(self):
        hb = self.hb
        rows = np.zeros((hb.n_sa, 88), np.uint8)
        a = O._recargs(hb)
        self.o.orc_shard_sa_rows(*a, rows.ctypes.data)
        return torch.from_numpy(rows)

    def set_sa_rows(self, t):
        self.rows = np.ascontiguousarray(t.numpy())

    def maxspan(self):
        return int((self.hb.cols["endpos"] - self.hb.cols["pos"]).max(initial=0)) + 1

    def set_maxspan(self, m):
        pass

    def _rec(self):
        c = self.hb.cols
        return [self.hb.n, c["flag"], c["mapq"], c["tid"], c["pos"], c["endpos"]]

    def coverage(self, d):
        self._d = d
        ncl = self.cl.shape[0]
        cov = np.zeros(2 * ncl + 1, np.uint32)
        self.o.orc_shard_coverage(*self._rec(), ncl, self.cl.ctypes.data, d, cov)
        return torch.from_numpy(cov[:2 * ncl].astype(np.int32))

    def commit_coverage(self, t):
        self.cov = np.ascontiguousarray(t.numpy().astype(np.uint32))

    def vote(self):
        ncl = self.cl.shape[0]
        self.valid = np.zeros(ncl + 1, np.uint32)
        rc = self.o.orc_shard_vote(self.rows.shape[0], self.rows.ctypes.data, ncl, self.cl.ctypes.data, np.append(self.cov, 0).astype(np.uint32),
                                   len(self.hb.target_names), O._names(self.hb), self._d, self.valid)
        if rc < 0:
            raise RuntimeError("error cigar")

    def depth(self):
        ncl = self.cl.shape[0]
        dep = np.zeros(2 * ncl + 1, np.uint32)
        self.o.orc_shard_depth(*self._rec(), ncl, self.cl.ctypes.data, self.valid, dep)
        return torch.from_numpy(dep[:2 * ncl].astype(np.int32))

    def commit_depth(self, t):
        self.dep = np.append(t.numpy().astype(np.uint32), 0).astype(np.uint32)

    def finish(self):
        nt = len(self.hb.target_names)
        if self.nibs is not None:
            keep = [np.ascontiguousarray(p, np.uint8) for p, _ in self.nibs]
            ptrs = (vp * nt)(*[k.ctypes.data for k in keep])
            lens = (C.c_uint64 * nt)(*[int(l) for _, l in self.nibs])
            m = self.o.orc_shard_finish(self.cl.shape[0], self.cl.ctypes.data, self.valid, self.dep, C.cast(ptrs, C.POINTER(vp)), C.cast(lens, C.POINTER(C.c_uint64)))
        else:
            m = self.o.orc_shard_finish(self.cl.shape[0], self.cl.ctypes.data, self.valid, self.dep, None, None)
        return self.cl[:m].copy().view(CLUSTER_DTYPE).reshape(-1)
