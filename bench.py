#!/usr/bin/env python
"""bench.py -- throughput of the BreakID hot path on B200 (BASELINE.json metric: read pairs/s classified + clustered
+ refined; decode excluded AND included, both stated).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--scale S] [--impl reference] [--dump-outputs DIR]

One JSON line.  Every throughput below (value, e2e, e2e_host_soa, legs) is measured over exactly K timed steps; the
per-kernel and per-stage breakdowns come from two extra steps of their own.  With the same arguments the inputs are the
same from run to run (seeded generators), so DIR (see dump_outputs) lets two builds be compared output for output.
What the keys mean here:

  value     BASELINE.json configs[1] (hg19-shaped 3.1 Gb genome, 30x 2x150 bp, 2000 planted SVs, 1 % chimeric noise;
            --scale shrinks it), records RESIDENT in HBM when the timed region starts, decode EXCLUDED.  A step is one
            pass of the whole hot path: classify + insert statistics, mate join, bucket grouping, isolated-pair mask,
            AHC clustering, split-read refinement.  The inputs (9.3 GB at scale 1) are larger than L2: no flush needed.
  e2e       decode INCLUDED, through the C ABI with HOST buffers: the bytes of a real BGZF-compressed BAM in pinned host
            memory -> bkid_push_bgzf (H2D of the compressed bytes, device inflate, record decode) -> bkid_run ->
            bkid_fetch_clusters (D2H).  The BAM is the bounded sample of configs[1] that `--impl reference` times the
            unmodified reference CPU binary on (the reference has no decode-excluded entry): same file, same metric --
            this pair is the like-for-like comparison; `same_sample` repeats it with the parity check of that run.
  e2e_host_soa   decode excluded but host buffers: pinned struct-of-arrays batch of the FULL workload -> bkid_push_batch
            -> bkid_run -> bkid_fetch_clusters.
  roofline  the dominant kernel by measured time, plus `kernels` (every kernel >= 3 % of the step, CUDA events on the
            launching stream via bkid_profile_kernels) and `whole_step` (the bytes the step must read once / step time).
  parity_checked   outside the timed region: the same path on configs[1] x min(scale, 1/16) compared with the CPU oracle,
            byte for byte; the bench exits non-zero when that fails.
  legs      configs[2] (exclude intervals + -q 20 -s 15), configs[3] (100x tumour, 500 translocations), configs[4]
            (split-read stress) and the banded-alignment kernel, each as a short resident measurement.

N > 1 (torchrun): WEAK scaling by coverage -- the job holds ONE coordinate-sorted record stream of N x 30x coverage
(N samples of the same genome merged), cut into N genomic bins of equal genome length; rank r holds bin r (about as many
records as the single-GPU workload).  A small sharded parity check against the oracle runs before the timed region.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from breakid_b200 import api, synth  # noqa: E402

METRIC = "read_pairs_per_sec_classified_clustered_refined"
UNIT = "read pairs/s"
DTYPE = "u32/i64 integer + f64 (AHC distances)"
N_FULL = 619243482                      # records of configs[1] at scale 1
REF_SEC_PER_RECORD = 1.95e-6            # reference CPU binary incl. htslib decode on this pool's hosts (BENCH_r01: 4.65 s / 2.42 M records)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def sample_scale(steps, warmup):
    """the bounded sample BOTH arms use for the decode-included comparison: the largest power-of-two fraction of configs[1]
    that keeps `steps + warmup` runs of the single-threaded reference binary within about four minutes"""
    budget = 240.0 / max(1, steps + warmup)
    s = 1.0 / 32
    while s > 1.0 / 2048 and N_FULL * s * REF_SEC_PER_RECORD > budget:
        s /= 2
    return s


def workload_cfg(scale):
    return synth.config2(scale=scale)


def config_block(args):
    """identical in both arms (the driver compares it)"""
    s = sample_scale(args.steps, args.warmup)
    return {"workload": "BASELINE.json configs[1]: synthetic hg19-shaped 3.1 Gb genome, 30x 2x150bp, 2000 planted SVs, 1% chimeric noise, AHC mode"
                        + ("" if args.scale == 1.0 else " x scale %g" % args.scale),
            "value_is": "decode excluded, records resident in HBM, whole workload",
            "e2e_is": "decode included, BAM bytes in host memory, bounded sample configs[1] x 1/%d (the file both arms run on)" % round(1 / s),
            "sample_scale": s, "scale": args.scale, "l2": "inputs larger than L2, no flush"}


class ClockSampler:
    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
                 "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# batches
# ------------------------------------------------------------------------------------------------------------------
def device_batch(d: synth.SynthData):
    """SynthData (cuda tensors) -> (api.Batch with device pointers, keep-alive dict).  The insert-size and span columns are
    handed over in their narrow forms (isize16 / span16, include/breakid_b200.h) whenever the whole batch fits them -- what
    a decoder does -- and stay narrow in HBM; tid stays wide (resident)."""
    keep = {}
    c = d.cols
    keep["flag"] = c["flag"].contiguous()
    keep["mapq"] = c["mapq"].contiguous()
    for k in ("tid", "pos"):
        keep[k] = c[k].contiguous()
    n = d.n
    flag = c["flag"].to(torch.int32)
    span = c["endpos"].to(torch.int64) - c["pos"].to(torch.int64)
    if n and int(span.min()) >= 0 and int(span.max()) <= 65535:
        keep["span16"] = span.to(torch.int16).contiguous()          # two's-complement wrap: same 16 bits as uint16
    else:
        keep["endpos"] = c["endpos"].contiguous()
    read = ((flag & 1) != 0) & ((flag & 2) != 0) & ((flag & (0x4 | 0x100 | 0x200 | 0x400)) == 0)
    iz = c["isize"][read]
    if n and (iz.numel() == 0 or (int(iz.min()) >= -32768 and int(iz.max()) <= 32767)):
        keep["isize16"] = c["isize"].clamp(-32768, 32767).to(torch.int16).contiguous()
    else:
        keep["isize"] = c["isize"].contiguous()
    del span, read, iz
    # sparse mate/name table: records that are not proper pairs or carry an SA tag (what a host decoder lists)
    in_x = (flag & 2) == 0
    in_x[d.sa_rec] = True
    del flag
    xr = torch.nonzero(in_x).flatten()
    keep["x_rec"] = xr.to(torch.int32).contiguous()
    keep["x_mtid"] = c["mtid"][xr].contiguous()
    keep["x_mpos"] = c["mpos"][xr].contiguous()
    keep["x_name_hash"] = synth.name_hash_ids(c["name_id"][xr]).contiguous()
    keep["sa_rec"] = d.sa_rec.to(torch.int32).contiguous()
    keep["cig_off"] = d.cig_off.to(torch.int32).contiguous()
    keep["cig_ops"] = d.cig_ops.to(torch.int32).contiguous()
    keep["sa_off"] = d.sa_off.to(torch.int32).contiguous()
    keep["sa_txt"] = d.sa_txt.contiguous()
    keep["oc_off"] = torch.zeros(d.sa_rec.numel() + 1, dtype=torch.int32, device=d.sa_rec.device)
    keep["oc_txt"] = torch.zeros(16, dtype=torch.uint8, device=d.sa_rec.device)
    b = api.Batch()
    b.n = d.n
    b.n_x = int(xr.numel())
    b.n_sa = int(d.sa_rec.numel())
    for k, v in keep.items():
        setattr(b, k, v.data_ptr())
    return b, keep


def host_batch_pinned(keep, n, n_sa, n_x):
    """pinned host copies of the device columns -> (api.Batch with host pointers, keep-alive, bytes).  Same column forms as
    the resident batch, plus tid as one run per target (records are coordinate sorted): 11 B/record instead of 19."""
    hk = {}
    nbytes = 0
    src = dict(keep)
    tid = keep["tid"]
    if n:
        start = torch.nonzero(torch.cat([torch.ones(1, dtype=torch.bool, device=tid.device), tid[1:] != tid[:-1]])).flatten()
        if start.numel() <= 65536:
            src["tid_run_start"] = start.to(torch.int32)
            src["tid_run_tid"] = tid[start].contiguous()
            del src["tid"]
    for k, v in src.items():
        h = torch.empty(v.shape, dtype=v.dtype, pin_memory=True)
        h.copy_(v)
        hk[k] = h
        nbytes += h.numel() * h.element_size()
    b = api.Batch()
    b.n = n
    b.n_sa = n_sa
    b.n_x = n_x
    for k, v in hk.items():
        setattr(b, k, v.data_ptr())
    if "tid_run_start" in hk:
        b.n_tid_runs = int(hk["tid_run_start"].numel())
    return b, hk, nbytes


def _segment_gather(off, data, order):
    """variable-length segments data[off[i]:off[i+1]] re-ordered by `order` -> (new offsets, new data)"""
    ln = (off[1:] - off[:-1])[order]
    new_off = torch.zeros(order.numel() + 1, dtype=off.dtype, device=off.device)
    new_off[1:] = torch.cumsum(ln, 0)
    total = int(new_off[-1])
    if total == 0:
        return new_off, data[:0].clone()
    seg = torch.repeat_interleave(torch.arange(order.numel(), device=off.device), ln)
    src = off[:-1][order][seg] + (torch.arange(total, device=off.device) - new_off[:-1][seg])
    return new_off, data[src]


def rank_slice(cfg, rank, world, dev):
    """bin `rank` of ONE coordinate-sorted stream of world x 30x coverage: sample s of the same genome is generated with its
    own seed and read names, only its records inside the bin are kept, and the kept records of all samples are merged in
    coordinate order (stable: ties keep sample order, like a samtools merge).  Bins have equal genome length."""
    lens = torch.tensor(cfg.chrom_lens, dtype=torch.int64, device=dev)
    cum = torch.zeros(len(cfg.chrom_lens) + 1, dtype=torch.int64, device=dev)
    cum[1:] = torch.cumsum(lens, 0)
    G = int(cum[-1])
    lo, hi = G * rank // world, G * (rank + 1) // world
    parts = []
    for s in range(world):
        c2 = synth.SynthConfig(**{**cfg.__dict__, "seed": cfg.seed + 1000 * s})
        d = synth.generate(c2, device=str(dev))
        tid = d.cols["tid"].to(torch.int64)
        g = torch.where(tid >= 0, cum[tid.clamp(min=0)] + d.cols["pos"].to(torch.int64), torch.full_like(tid, G))    # unplaced records: last bin
        keep = (g >= lo) & ((g < hi) | (rank == world - 1))
        idx = torch.nonzero(keep).flatten()
        cols = {k: v[idx] for k, v in d.cols.items()}
        cols["name_id"] = cols["name_id"] + s * 1_000_000_000
        newpos = torch.full((d.n,), -1, dtype=torch.int64, device=dev)
        newpos[idx] = torch.arange(idx.numel(), device=dev)
        sa_keep = torch.nonzero(newpos[d.sa_rec] >= 0).flatten()
        cig_off, cig_ops = _segment_gather(d.cig_off, d.cig_ops, sa_keep)
        sa_off, sa_txt = _segment_gather(d.sa_off, d.sa_txt, sa_keep)
        parts.append((cols, g[idx], newpos[d.sa_rec][sa_keep], cig_off, cig_ops, sa_off, sa_txt))
        del d, tid, g, keep, idx, newpos
        torch.cuda.empty_cache()
    base = np.cumsum([0] + [int(p[1].numel()) for p in parts])
    key = torch.cat([p[1] for p in parts])
    order = torch.sort(key, stable=True).indices
    inv = torch.empty_like(order)
    inv[order] = torch.arange(order.numel(), device=dev)
    cols = {k: torch.cat([p[0][k] for p in parts])[order] for k in parts[0][0]}
    sa_rec = inv[torch.cat([p[2] + int(base[i]) for i, p in enumerate(parts)])]
    cig_off = torch.zeros(sa_rec.numel() + 1, dtype=torch.int64, device=dev)
    cig_off[1:] = torch.cumsum(torch.cat([p[3][1:] - p[3][:-1] for p in parts]), 0)
    cig_ops = torch.cat([p[4] for p in parts])
    sa_off = torch.zeros(sa_rec.numel() + 1, dtype=torch.int64, device=dev)
    sa_off[1:] = torch.cumsum(torch.cat([p[5][1:] - p[5][:-1] for p in parts]), 0)
    sa_txt = torch.cat([p[6] for p in parts])
    so = torch.sort(sa_rec).indices                                  # the SA side table is kept in ascending record order
    cig_off2, cig_ops2 = _segment_gather(cig_off, cig_ops, so)
    sa_off2, sa_txt2 = _segment_gather(sa_off, sa_txt, so)
    return synth.SynthData(cfg=cfg, cols=cols, sa_rec=sa_rec[so], cig_off=cig_off2, cig_ops=cig_ops2, sa_off=sa_off2, sa_txt=sa_txt2, truth={})


# ------------------------------------------------------------------------------------------------------------------
# the bounded sample both arms share (decode included)
# ------------------------------------------------------------------------------------------------------------------
def sample_dataset(scale, index=False):
    """BAM + nib + refGene of configs[1] x scale in a cache directory under the system temporary directory (whichever arm
    runs first writes it).  index=True adds the .bai index, which only the reference binary reads; it is built with
    oracle/_ref/bamindex, so only where the reference is built."""
    import oracle_py as O
    from breakid_b200 import bamio
    d = os.path.join(tempfile.gettempdir(), "bkid_sample_1_%d" % round(1 / scale))
    done = os.path.join(d, ".done")
    paths = {"bam": os.path.join(d, "reads.bam"), "nib": os.path.join(d, "nib"), "refgene": os.path.join(d, "ref_files", "refGene.txt")}
    if not os.path.exists(done):
        os.makedirs(d, exist_ok=True)
        data = synth.generate(workload_cfg(scale))
        t0 = time.time()
        bamio.write_dataset(d, data, random_qual=True)
        with open(done, "w") as f:
            f.write("%d %.1f\n" % (data.n, time.time() - t0))
    if index and not os.path.exists(paths["bam"] + ".bai"):
        O.ref_index(paths["bam"])
    n = int(open(done).read().split()[0])
    return paths, n


def decode_included(local, steps, warmup, scale, check=True):
    """E2E: compressed BAM bytes in pinned host memory -> bkid_push_bgzf -> bkid_run -> bkid_fetch_clusters, all inside the
    timed region; afterwards (untimed) the calls of that very run are compared with the CPU oracle on the host-decoded file."""
    paths, n_expect = sample_dataset(scale)
    bam = paths["bam"]
    f = api.BgzfFile(bam)
    raw = torch.from_numpy(np.fromfile(bam, dtype=np.uint8)).pin_memory()
    ctx = api.Context(f.target_len, f.target_names, device=local)
    ts = []
    out = None
    for i in range(warmup + steps):
        ctx.reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = ctx.push_bgzf(f, data_ptr=raw.data_ptr())
        res = ctx.run()
        out = ctx.fetch_clusters()
        dt = time.perf_counter() - t0
        if i >= warmup:
            ts.append(dt)
    st = ctx.decode_stats()
    tm = ctx.timings()
    ctx.close()
    f.close()
    ms = float(np.mean(ts)) * 1e3
    r = {"value": n / 2.0 / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "h2d_bytes_per_step": int(st["compressed_bytes"]),
         "d2h_bytes_per_step": int(out.nbytes), "records": int(n), "calls": int(len(out)),
         "sample": "configs[1] x 1/%d: %d records, %d-byte BAM (%d BGZF blocks, %d bytes uncompressed)" % (round(1 / scale), n, raw.numel(), st["n_blocks"], st["uncompressed_bytes"]),
         "decode_ms": st["total_ms"], "inflate_ms": st["inflate_ms"], "boundaries_ms": st["boundaries_ms"], "extract_ms": st["extract_ms"], "hot_path_ms": tm["total"],
         "inflate_GBps_uncompressed": st["uncompressed_bytes"] / (st["inflate_ms"] * 1e-3) / 1e9 if st["inflate_ms"] > 0 else None,
         "note": "compressed BAM bytes in pinned host memory -> bkid_push_bgzf -> bkid_run -> bkid_fetch_clusters"}
    if check:
        import oracle_py as O
        hb = api.HostBatch.from_bam(bam, threads=os.cpu_count() or 8)
        om, osd, od, exp = O.run(hb, None, mode=0)
        r["identical_to_oracle"] = bool((res[0], res[1], res[2]) == (om, osd, od) and out.tobytes() == exp.tobytes() and hb.n == n)
    return r


def decode_included_sharded(rank, world, local, dev, steps, warmup, scale):
    """E2E at N GPUs on the SAME file the reference arm runs on: every rank holds the compressed BAM bytes in pinned host memory,
    inflates and decodes its own BGZF block range (bkid_push_bgzf_range), and the ranks finish the step with the in-library
    exchanges (bkid_dist_run, NCCL).  All inside the timed region; max over ranks.  Afterwards (untimed) the ranges must
    stitch and rank 0 compares the calls of the last step with the CPU oracle on the host-decoded file."""
    import torch.distributed as dist
    from breakid_b200.dist import LibraryDist
    if rank == 0:
        paths, _ = sample_dataset(scale)
    dist.barrier()
    if rank != 0:
        paths, _ = sample_dataset(scale)
    bam = paths["bam"]
    f = api.BgzfFile(bam)
    raw = torch.from_numpy(np.fromfile(bam, dtype=np.uint8)).pin_memory()
    cuts = [f.n_blocks * i // world for i in range(world + 1)]
    ctx = api.Context(f.target_len, f.target_names, device=local)
    ld = LibraryDist(ctx, dev)
    ts = []
    out = None
    for i in range(warmup + steps):
        ctx.reset()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n, a, b = ctx.push_bgzf_range(f, cuts[rank], cuts[rank + 1], data_ptr=raw.data_ptr())
        res = ld.run(0)
        out = ctx.fetch_clusters()
        torch.cuda.synchronize()
        dist.barrier()
        dt = time.perf_counter() - t0
        if i >= warmup:
            ts.append(dt)
    st = ctx.decode_stats()
    marks = torch.tensor([n, a, b, int(st["compressed_bytes"])], dtype=torch.int64, device=dev)
    allm = [torch.zeros_like(marks) for _ in range(world)]
    dist.all_gather(allm, marks)
    allm = [m.tolist() for m in allm]
    t = torch.tensor([float(np.mean(ts)) * 1e3], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    n_total = sum(m[0] for m in allm)
    stitch = all(allm[r][2] == allm[r + 1][1] for r in range(world - 1))
    r = {"value": n_total / 2.0 / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "h2d_bytes_per_step": int(sum(m[3] for m in allm)),
         "d2h_bytes_per_step": int(out.nbytes) * world, "records": int(n_total), "calls": int(len(out)), "n_gpus_used": world, "ranges_stitch": bool(stitch),
         "sample": "configs[1] x 1/%d: %d records, %d-byte BAM" % (round(1 / scale), n_total, raw.numel()),
         "decode_ms_rank0": st["total_ms"], "inflate_ms_rank0": st["inflate_ms"],
         "note": "every rank: its BGZF block range of the compressed BAM (pinned host memory) -> bkid_push_bgzf_range -> bkid_dist_run (NCCL) -> bkid_fetch_clusters"}
    if rank == 0:
        import oracle_py as O
        hb = api.HostBatch.from_bam(bam, threads=os.cpu_count() or 8)
        om, osd, od, exp = O.run(hb, None, mode=0)
        r["identical_to_oracle"] = bool(stitch and (res[0], res[1], res[2]) == (om, osd, od) and out.tobytes() == exp.tobytes() and hb.n == n_total)
    ld.close()
    ctx.close()
    f.close()
    return r


# ------------------------------------------------------------------------------------------------------------------
# legs
# ------------------------------------------------------------------------------------------------------------------
def resident_leg(local, dev, cfg, steps, label, ctx_kw=None, exclude=None):
    """a short resident measurement of another BASELINE.json config: whole-step ms and stage times"""
    d = synth.generate(cfg, device=str(dev))
    names = [synth.chrom_name(t) for t in range(len(cfg.chrom_lens))]
    b_dev, keep = device_batch(d)
    n, n_sa = d.n, int(d.sa_rec.numel())
    del d
    torch.cuda.empty_cache()
    ctx = api.Context(cfg.chrom_lens, names, device=local, **(ctx_kw or {}))
    tot = 0.0
    st = {}
    for i in range(3 + steps):
        ctx.reset()
        ctx.push_device(b_dev)
        if exclude is not None:
            ctx.set_exclude(*exclude)
        res = ctx.run()
        tm = ctx.timings()
        if i >= 3:
            tot += tm["total"]
            for k in api.TIMING_FIELDS_F:
                st[k] = st.get(k, 0.0) + tm[k] / steps
    ctx.close()
    del keep
    torch.cuda.empty_cache()
    ms = tot / steps
    return {"workload": label, "records": n, "n_sa": n_sa, "calls": int(res[3]), "ms_per_step": ms, "value": n / 2.0 / (ms * 1e-3), "unit": UNIT,
            "stage_ms": st, "counts": {k: tm[k] for k in api.TIMING_FIELDS_I}, "steps": steps}


def exclude_intervals(cfg, frac=0.05, seed=3):
    """centromere / telomere shaped exclude intervals covering ~frac of every chromosome (configs[2])"""
    rng = np.random.RandomState(seed)
    t, b, e = [], [], []
    for k, l in enumerate(cfg.chrom_lens):
        w = int(l * frac / 3)
        mid = int(l * (0.35 + 0.1 * rng.rand()))
        for lo in (0, mid, l - w):
            t.append(k); b.append(lo); e.append(lo + w)
    return np.array(t, np.int32), np.array(b, np.int32), np.array(e, np.int32)


def align_leg(local, steps, n_pairs=1 << 20):
    """north_star kernel 4 (banded alignment; extension, default off): clipped reads of length U(20,130) against their
    reference window, band 12.  pairs/s and cell updates/s of the kernel alone (host arrays in, device timing inside)."""
    rng = np.random.RandomState(5)
    ln = rng.randint(20, 131, n_pairs)
    off = np.concatenate([[0], np.cumsum(ln)]).astype(np.uint32)
    q = rng.randint(0, 4, int(off[-1])).astype(np.uint8)
    q = np.frombuffer(b"ACGT", np.uint8)[q]
    r = q.copy()
    mut = rng.rand(r.shape[0]) < 0.03
    r[mut] = np.frombuffer(b"ACGT", np.uint8)[rng.randint(0, 4, int(mut.sum()))]
    ctx = api.Context([1000], ["chr1"], device=local)
    out = np.zeros(n_pairs, np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    ts = []
    api.profile_kernels(True)
    api.profile_report()
    for i in range(steps):
        t0 = time.perf_counter()
        ctx._chk(ctx.lib.bkid_op_banded_align(ctx.ctx, n_pairs, p(q), p(off), p(r), p(off), 12, p(out)))
        ts.append(time.perf_counter() - t0)
    rep = api.profile_report()
    api.profile_kernels(False)
    ctx.close()
    kms = [v[1] / v[0] for k, v in rep.items() if "align" in k]
    kernel_ms = float(min(kms)) if kms else None
    cells = float((ln.astype(np.int64) * 25).sum())                  # band 12: 25 cells per query position
    return {"workload": "%d (clip, window) pairs, clip length U(20,130), band 12, 3%% substitutions" % n_pairs, "kernel_ms": kernel_ms,
            "pairs_per_s": n_pairs / (kernel_ms * 1e-3) if kernel_ms else None, "cell_updates_per_s": cells / (kernel_ms * 1e-3) if kernel_ms else None,
            "host_call_ms": float(min(ts)) * 1e3, "mean_distance": float(out.mean()),
            "note": "issue utilisation of this kernel: profiles/ (ncu smsp__issue_active); it is integer-issue bound, not HBM bound"}


# algorithmic bytes per unit of the kernels that matter (DESIGN.md section 3); unit counts are taken from the run
NCU_TRAFFIC = os.path.join(ROOT, "profiles", "r02h_ncu_front_kernels.json")


def ncu_traffic(kernel, n):
    """DRAM bytes per launch of `kernel` for n records: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full`
    capture (profiles/r02h_ncu_front_kernels.{md,json}, same kernel body, 619 243 482 records), scaled per record; None when the
    kernel is not in that capture"""
    try:
        prof = json.load(open(NCU_TRAFFIC))
    except OSError:
        return None
    base = kernel.split("<")[0]
    k = prof["kernels"].get(base)
    return k["dram_bytes_per_record"] * n if k else None


def kernel_bytes(name, cnt, n):
    nc, npair = cnt["n_candidates"], cnt["n_pairs"]
    if name.startswith("k1_classify"):
        return 8.0 * n, "8 B/record: flag 2 + mapq 1 + isize16 2 + span16 2 read, class 1 written"
    if name.startswith("sd_fast"):
        return 3.0 * n, "3 B/record: class 1 + isize16 2 read"
    if name.startswith("kx_count"):
        return 5.0 * cnt.get("n_x", nc), "x_rec 4 + class byte 1 per sparse-table entry"
    if name.startswith("kx_write"):
        return (28.0 + 11.0 + 60.0) * nc, "per candidate: sparse entry 28 + flag/mapq/tid/pos 11 read, row 48 + sort pair 12 written"
    if name.startswith("k2_join"):
        return (12.0 + 2 * 48.0 + 4.0) * nc, "per candidate: sort pair 12 + its row and its neighbour's row 96 read, mate 4 written"
    if name.startswith("k2_build_pairs"):
        return 4.0 * nc + (2 * 48.0 + 64.0) * npair, "mate 4 per candidate; two rows read + one pair written per pair"
    return None, None


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirpath, res, calls):
    """what one step of the timed path hands its caller, as float64 arrays: insert_mean, insert_sd, cluster_dist and n_called
    from bkid_run, and call_<field> for every field of the call records of bkid_fetch_clusters (the 41-mer fields as
    [n, 44] byte codes).  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of the calls is written, and call_index
    holds their positions."""
    os.makedirs(dirpath, exist_ok=True)
    arrays = {k: np.array([v], np.float64) for k, v in zip(("insert_mean", "insert_sd", "cluster_dist", "n_called"), res)}
    fields = {}
    for k in calls.dtype.names:
        a = np.ascontiguousarray(calls[k])
        fields["call_" + k] = a.view(np.uint8).reshape(len(a), a.dtype.itemsize) if a.dtype.kind == "S" else a
    row_bytes = 8 * (1 + sum(dt.itemsize if dt.kind == "S" else 1 for dt, _ in calls.dtype.fields.values()))     # + call_index
    keep = (DUMP_LIMIT_BYTES - (1 << 16)) // row_bytes          # 64 KiB left for the scalars and the .npy headers
    if len(calls) > keep:
        idx = np.sort(np.random.RandomState(0).choice(len(calls), keep, replace=False))
        fields = {k: a[idx] for k, a in fields.items()}
        arrays["call_index"] = idx.astype(np.float64)
    for k, a in fields.items():
        arrays[k] = a.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(dirpath, k + ".npy"), a)


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    cfg = workload_cfg(args.scale)

    # ---- N > 1: sharded parity pre-step (untimed) ----
    pre = None
    if world > 1:
        pre = sharded_parity(rank, world, local, dev)

    t0 = time.time()
    if world == 1:
        d = synth.generate(cfg, device=str(dev))
    else:
        d = rank_slice(cfg, rank, world, dev)
    torch.cuda.synchronize()
    gen_s = time.time() - t0
    names = [synth.chrom_name(t) for t in range(len(cfg.chrom_lens))]
    b_dev, keep = device_batch(d)
    n, n_sa, n_x = d.n, int(d.sa_rec.numel()), int(b_dev.n_x)
    del d
    torch.cuda.empty_cache()
    ctx = api.Context(cfg.chrom_lens, names, device=local)
    if args.nib:
        for t, l in enumerate(cfg.chrom_lens):
            ctx.set_nib(t, synth.random_nib_bytes(l, cfg.seed * 1000 + t, device=str(dev)).cpu().numpy(), l)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            torch.cuda.synchronize()

    engine = None
    libdist = None
    shard_timing = {}
    timing_on = [False]
    if world > 1:
        from breakid_b200.dist import GpuEngine, LibraryDist, DIST_STAGES, run_sharded
        if args.py_dist:
            engine = GpuEngine(ctx, dev)              # the Python-orchestrated exchanges (torch.distributed), kept for A/B
        else:
            libdist = LibraryDist(ctx, dev)           # the exchanges inside the library: NCCL calls from C++

    def run_path():
        if world == 1:
            return ctx.run()
        if libdist is not None:
            mean, sd, dd, nc, tms = libdist.run(0)
            if timing_on[0]:
                for k, v in zip(DIST_STAGES, tms):
                    shard_timing[k] = shard_timing.get(k, 0.0) + v
            return mean, sd, dd, nc
        mean, sd, dd, out = run_sharded(engine, n, mode=0, timing=shard_timing if timing_on[0] else None)
        return mean, sd, dd, len(out)

    def step_resident():
        ctx.reset()
        ctx.push_device(b_dev)
        return run_path()

    # ---- value: inputs resident in HBM ----
    for _ in range(args.warmup):
        step_resident()
    ref_out = ctx.fetch_clusters() if world == 1 else None
    barrier()
    stage = {k: 0.0 for k in api.TIMING_FIELDS_F}
    launches = 0
    with ClockSampler(local) as clk:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record()
        dev_ms = 0.0
        for _ in range(args.steps):
            res = step_resident()
            tm = ctx.timings()
            dev_ms += tm["total"]
            for k in stage:
                stage[k] += tm[k]
            launches += tm["kernel_launches"]
        barrier()
        ev1.record()
        ev1.synchronize()
        wall = time.perf_counter() - t0
        if world > 1:
            dev_ms = ev0.elapsed_time(ev1)           # every library call is host-synchronous, so device span == wall span
    counts = {k: tm[k] for k in api.TIMING_FIELDS_I}
    counts["n_x"] = n_x
    ms_step = max(dev_ms, wall * 1e3) / args.steps       # device events and the wall clock must agree; report the slower
    ncall = res[3]
    deterministic = None
    if world == 1:
        last_out = ctx.fetch_clusters()
        deterministic = bool(last_out.tobytes() == ref_out.tobytes())
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, res, last_out)
    # ---- N > 1: per-stage / per-collective wall times of the sharded step (extra untimed steps with a sync after every stage) ----
    if world > 1:
        timing_on[0] = True
        for _ in range(2):
            step_resident()
        timing_on[0] = False
        barrier()
    # ---- per-kernel device times (CUDA events on the launching stream): two extra steps with the library's profiling on ----
    kern = {}
    if world == 1:
        api.profile_kernels(True)
        api.profile_report()
        for _ in range(2):
            step_resident()
        kern = {k: (v[0] / 2.0, v[1] / 2.0) for k, v in api.profile_report().items()}
        api.profile_kernels(False)

    # ---- e2e_host_soa: host buffers, H2D + D2H inside the timed region, decode excluded ----
    b_host, hkeep, h2d_bytes = host_batch_pinned(keep, n, n_sa, n_x)

    def step_e2e():
        ctx.reset()
        ctx.lib.bkid_push_batch(ctx.ctx, C.byref(b_host))
        r = run_path()
        out = ctx.fetch_clusters() if (world == 1 or libdist is not None) else None
        return r, out
    input_bytes = sum(v.numel() * v.element_size() for v in keep.values())
    del keep
    ctx.reset()
    torch.cuda.empty_cache()
    ctx.reserve(n, n_x, n_sa, 2 * n_sa + 16, int(hkeep["sa_txt"].numel()) + 16, 16)
    for _ in range(max(1, min(args.warmup, 2))):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r, out = step_e2e()
    barrier()
    soa_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    d2h_bytes = int(out.nbytes) if out is not None else 192 * int(r[3])

    # max over ranks
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms_step, soa_ms, float(n)], device=dev, dtype=torch.float64)
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_step, soa_ms = float(tmax[0]), float(tmax[1])
        n_total = float(tsum[2])
    else:
        n_total = float(n)
    pairs = n_total / 2.0
    peak, peak_src = peaks()

    # ---- roofline ----
    step_kernel_ms = sum(v[1] for v in kern.values()) or None
    klist = []
    for name, (nl, ms) in sorted(kern.items(), key=lambda kv: -kv[1][1]):
        if step_kernel_ms and ms / step_kernel_ms < 0.03:
            continue
        by, what = kernel_bytes(name, counts, n)
        ach = by / (ms * 1e-3) / 1e9 if by and ms > 0 else None
        klist.append({"kernel": name, "launches_per_step": nl, "ms_per_step": ms, "share_of_kernel_time": ms / step_kernel_ms if step_kernel_ms else None,
                      "algorithmic_bytes": by, "bytes_are": what, "achieved_GBps": ach, "frac": (ach / peak) if ach else None})
    dom = next((k for k in klist if k["algorithmic_bytes"]), None)
    if dom is None:                                       # N > 1: no per-kernel pass; K1 from the stage timers
        k1_ms = stage["classify"] / args.steps
        dom = {"kernel": "k1_classify", "ms_per_step": k1_ms, "algorithmic_bytes": 8.0 * n, "achieved_GBps": 8.0 * n / (k1_ms * 1e-3) / 1e9 if k1_ms > 0 else None}
        dom["frac"] = dom["achieved_GBps"] / peak if dom["achieved_GBps"] else None
    whole_bytes = 11.0 * n                                # K1 8 + sd pass 3 B/record: what the step must read once
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved_GBps"], "peak": peak, "unit": "GB/s", "frac": dom["frac"],
                "traffic": ncu_traffic(dom["kernel"], n), "peak_source": peak_src, "algorithmic_bytes_per_launch": dom["algorithmic_bytes"],
                "note": "dominant kernel by measured time (CUDA events around every launch on its own stream, two extra untimed steps); traffic = DRAM bytes per launch from one ncu --set full capture (profiles/r02h_ncu_front_kernels.md), scaled per record",
                "kernels": klist,
                "whole_step": {"algorithmic_bytes": whole_bytes, "bytes_are": "11 B/record must be read once (K1 8 + insert-sd pass 3); everything after K1 works on the 1 % candidates",
                               "ms_per_step": ms_step, "achieved_GBps": whole_bytes * (1 if world == 1 else 1) / (ms_step * 1e-3) / 1e9,
                               "frac": whole_bytes / (ms_step * 1e-3) / 1e9 / peak}}

    line = {
        "metric": METRIC, "value": pairs / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
        "data": "synthetic (device-generated hg19-shaped genome, 2x150bp, planted TRA/INV/DUP/DEL, 1% chimeric noise)",
        "config": config_block(args),
        "gpu_launches": int(launches),
        "workload": {"records_per_gpu": n, "records_total": int(n_total), "n_sa_per_gpu": n_sa, "input_bytes_per_gpu": int(input_bytes), "calls": int(ncall),
                     "parallelism": ("single GPU" if world == 1 else "weak scaling by coverage: one coordinate-sorted stream of %dx30x coverage cut into %d genomic bins of equal genome length, "
                                     "rank r holds bin r; candidates all-to-all by name hash, pairs all-to-all by bucket owner, clusters / evidence rows all-gather, "
                                     "coverage / depth / insert statistics all-reduce (NCCL)" % (world, world))},
        "e2e_host_soa": {"value": pairs / (soa_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": d2h_bytes, "ms_per_step": soa_ms,
                         "note": "decode excluded, whole workload: pinned host SoA batch (isize16 / span16 / tid runs) -> bkid_push_batch -> bkid_run -> bkid_fetch_clusters"},
        "stage_ms_per_step": ({k: v / args.steps for k, v in stage.items()} if world == 1 else {k: v / 2.0 for k, v in shard_timing.items()}),
        "counts": counts,
        "roofline": roofline,
        "deterministic_across_steps": deterministic,
        "clocks": clk.summary(),
        "gen_seconds": gen_s,
    }
    if world > 1:
        from breakid_b200 import dist as _d
        import torch.distributed as dist
        # every rank's own stage walls (a stage that ends in a collective includes the wait for the slowest rank) and its
        # device-side mask / cluster times: where the step's critical path is
        mine = torch.tensor([shard_timing.get(k, 0.0) / 2.0 for k in DIST_STAGES] + [tm["mask"], tm["cluster"], float(tm["n_pairs"]), float(tm["n_masked"])],
                            device=dev, dtype=torch.float64)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        line["stage_ms_per_rank"] = {"columns": list(DIST_STAGES) + ["mask (device)", "cluster (device)", "pairs owned", "pairs after mask"],
                                     "rows": [[round(float(x), 3) for x in r.tolist()] for r in allr]}
        line["exchanges"] = ("inside the library: NCCL all-reduce / grouped send-recv issued from C++ (bkid_dist_run)" if libdist is not None
                             else "Python-orchestrated (torch.distributed), --py-dist")
        line["sharded_parity"] = pre
        if libdist is not None:
            libdist.close()
    ctx.close()
    del hkeep, b_host
    torch.cuda.empty_cache()

    failed = False
    # ---- e2e: decode included, on the file the reference arm runs on ----
    s_scale = min(sample_scale(args.steps, args.warmup), args.scale)
    if world > 1 and not args.no_decode:
        e = decode_included_sharded(rank, world, local, dev, args.steps, 2, s_scale)
        if rank == 0:
            line["e2e"] = {"value": e["value"], "unit": UNIT, "h2d_bytes_per_step": e["h2d_bytes_per_step"], "d2h_bytes_per_step": e["d2h_bytes_per_step"],
                           "ms_per_step": e["ms_per_step"], "n_gpus_used": world, "sample": e["sample"], "note": e["note"]}
            line["same_sample"] = {"ours": e, "reference": "bench.py --impl reference --steps %d --warmup %d on the same file (%s)" % (args.steps, args.warmup, e["sample"]),
                                   "ratio": "ours.value / the reference arm's value: computed by the driver from the two lines"}
            failed |= e.get("identical_to_oracle") is False
    elif rank == 0 and not args.no_decode:
        e = decode_included(local, args.steps, 2, s_scale)
        line["e2e"] = {"value": e["value"], "unit": UNIT, "h2d_bytes_per_step": e["h2d_bytes_per_step"], "d2h_bytes_per_step": e["d2h_bytes_per_step"],
                       "ms_per_step": e["ms_per_step"], "n_gpus_used": 1, "sample": e["sample"], "note": e["note"]}
        line["same_sample"] = {"ours": e, "reference": "bench.py --impl reference --steps %d --warmup %d on the same file (%s)" % (args.steps, args.warmup, e["sample"]),
                               "ratio": "ours.value / the reference arm's value: computed by the driver from the two lines"}
        failed |= e.get("identical_to_oracle") is False
    elif args.no_decode:
        line["e2e"] = {"value": pairs / (soa_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": d2h_bytes,
                       "note": "decode-included leg skipped (--no-decode): this is e2e_host_soa"}
    # ---- parity on the benchmarked workload ----
    if rank == 0 and not args.no_parity:
        line["parity_checked"] = parity_check(local, dev, min(args.scale, 1.0 / 16))
        failed |= not line["parity_checked"]["identical"]
    if rank == 0 and not args.no_legs:
        legs = {}
        c2 = workload_cfg(args.scale)
        legs["configs[2]"] = resident_leg(local, dev, c2, args.steps, "BASELINE.json configs[2] on one GPU: configs[1] + exclude intervals (~5 %% of every chromosome) + -q 20 -s 15"
                                          + ("" if args.scale == 1.0 else " x scale %g" % args.scale), ctx_kw={"qual": 20, "sd_mult": 15}, exclude=exclude_intervals(c2))
        s4 = args.scale * 0.5                     # 100x at half the genome: 1.0e9 records, fits next to nothing else on one GPU
        legs["configs[3]"] = resident_leg(local, dev, synth.config4(scale=s4), args.steps, "BASELINE.json configs[3]: tumour-shaped 100x, planted translocations, x scale %g" % s4)
        sr = resident_leg(local, dev, synth.config5(scale=args.stress_scale), args.steps, "BASELINE.json configs[4] x scale %g: split-read refinement stress" % args.stress_scale)
        sr_ms = sr["stage_ms"]["evidence"] + sr["stage_ms"]["refine"]
        sr["split_reads_refined_per_s"] = sr["n_sa"] / (sr_ms * 1e-3) if sr_ms > 0 else None
        legs["configs[4]"] = sr
        legs["banded_alignment"] = align_leg(local, args.steps)
        line["legs"] = legs
        line["split_reads"] = {"value": sr["split_reads_refined_per_s"], "unit": "split reads refined/s", "note": "configs[4]: SA-tagged records / (evidence + refine stage time)"}
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_port(args)
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if failed:
        sys.exit(3)


def parity_check(local, dev, scale):
    """the benchmarked path on configs[1] x scale against the CPU oracle, byte for byte (untimed)"""
    import oracle_py as O
    cfg = workload_cfg(scale)
    d = synth.generate(cfg, device=str(dev))
    names = [synth.chrom_name(t) for t in range(len(cfg.chrom_lens))]
    b_dev, keep = device_batch(d)
    ctx = api.Context(cfg.chrom_lens, names, device=local)
    ctx.push_device(b_dev)
    res = ctx.run()
    got = ctx.fetch_clusters()
    ctx.close()
    del keep
    t0 = time.perf_counter()
    d_cpu = synth.SynthData(cfg=d.cfg, cols={k: v.cpu() for k, v in d.cols.items()}, sa_rec=d.sa_rec.cpu(), cig_off=d.cig_off.cpu(), cig_ops=d.cig_ops.cpu(),
                            sa_off=d.sa_off.cpu(), sa_txt=d.sa_txt.cpu(), truth={})
    n = d.n
    del d
    torch.cuda.empty_cache()
    hb = api.HostBatch.from_synth(d_cpu)
    om, osd, od, exp = O.run(hb, None, mode=0)
    same = bool((res[0], res[1], res[2]) == (om, osd, od) and got.tobytes() == exp.tobytes())
    return {"scale": scale, "records": n, "calls": int(len(exp)), "identical": same, "oracle": "oracle/liboracle.so orc_run (AHC mode), insert mean / sd / dist and every call record compared byte for byte",
            "oracle_seconds": time.perf_counter() - t0, "sha256_of_calls": hashlib.sha256(got.tobytes()).hexdigest()[:16]}


def sharded_parity(rank, world, local, dev):
    """a small dist_check-style run before the timed region: every rank takes a slice of one small dataset, the sharded
    result must be byte-identical to the oracle on the unsplit input (modes AHC and -fast, plus exclude + -q 20 -s 15)"""
    import torch.distributed as dist
    from breakid_b200.dist import GpuEngine, run_sharded
    from test_multi_gloo import _slice
    import oracle_py as O
    cfg = synth.SynthConfig(chrom_lens=[400000, 300000, 250000, 200000], n_tra=6, n_inv=3, n_dup=3, n_del=3, seed=41, sv_jitter=1)
    d = synth.generate(cfg)
    hb = api.HostBatch.from_synth(d)
    cuts = [hb.n * i // world for i in range(world + 1)]
    part = _slice(hb, cuts[rank], cuts[rank + 1])
    res = {}
    from breakid_b200.dist import LibraryDist
    for label, mode, kw, sdm in (("ahc", 0, {}, 3), ("fast", 1, {"fast": 1}, 3), ("q20_s15", 0, {"qual": 20, "sd_mult": 15}, 15)):
        ctx = api.Context(hb.target_len, hb.target_names, device=local, **kw)
        ctx.push(part)
        ld = LibraryDist(ctx, dev)
        mean, sd, dd, ncall, _ = ld.run(mode)
        out = ctx.fetch_clusters()
        ld.close()
        ok = True
        if rank == 0:
            m, s, d0, exp = O.run(hb, None, mode=mode, sd_mult=sdm)
            ok = bool((mean, sd, dd) == (m, s, d0) and out.tobytes() == exp.tobytes() and len(exp) >= 8)
        res[label] = ok
        ctx.close()
    flag = torch.tensor([1 if all(res.values()) else 0], device=dev)
    dist.broadcast(flag, src=0)
    if int(flag[0]) != 1:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "error": "sharded parity pre-step failed", "sharded_parity": res}), flush=True)
        sys.exit(3)
    return {"world": world, "records": hb.n, "identical_to_oracle": res}


def cpu_baseline_port(args):
    """CPU baseline on the host cores of this box, on the bounded sample the e2e leg ran on: ONE run of the reference CPU
    binary (oracle/_ref/BreakID_ref, single-threaded, BAM decode included -- 10-30 s of CPU work at the default sample) when it
    is built, with the oracle port (decode excluded) on the same records beside it; the port alone otherwise."""
    import oracle_py as O
    scale = min(sample_scale(args.steps, args.warmup), args.scale)
    cores = os.cpu_count()
    if os.path.exists(O.REF_BIN):
        paths, n = sample_dataset(scale, index=True)
        O.ref_install_refgene(paths["refgene"])
        tmp = tempfile.mkdtemp(prefix="bkid_cpu_")
        t0 = time.perf_counter()
        r = O.ref_run_binary(paths["bam"], os.path.join(tmp, "ref"), paths["nib"])
        dt = time.perf_counter() - t0
        if r.returncode == 0:
            hb = api.HostBatch.from_bam(paths["bam"], threads=cores or 8)
            t0 = time.perf_counter()
            O.run(hb, None, mode=0)
            dp = time.perf_counter() - t0
            return {"value": n / 2.0 / dt, "unit": UNIT, "cores": 1, "kind": "reference", "seconds": dt,
                    "sample": "configs[1] x 1/%d: %d records, %d-byte BAM, decode included, one run of oracle/_ref/BreakID_ref (single-threaded program, host has %d cores)"
                              % (round(1 / scale), n, os.path.getsize(paths["bam"]), cores),
                    "port": {"value": hb.n / 2.0 / dp, "unit": UNIT, "cores": 1, "seconds": dp, "what": "oracle/liboracle.so orc_run on the same records, decode excluded"}}
    cfg = workload_cfg(min(args.scale, 1.0 / 4))
    d = synth.generate(cfg)
    hb = api.HostBatch.from_synth(d)
    t0 = time.perf_counter()
    O.run(hb, None, mode=0)
    dt = time.perf_counter() - t0
    return {"value": hb.n / 2.0 / dt, "unit": UNIT, "cores": 1, "kind": "port", "seconds": dt,
            "sample": "configs[1] x 1/4: %d records, oracle/liboracle.so orc_run (AHC mode, decode excluded), host has %d cores" % (hb.n, cores)}


def run_reference(args):
    """the unmodified reference CPU binary (oracle/_ref/BreakID_ref) on the bounded sample both arms share (rank 0 only)"""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import oracle_py as O
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    scale = min(sample_scale(args.steps, args.warmup), args.scale)
    if not os.path.exists(O.REF_BIN):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/BreakID_ref is not built (run __graft_entry__.build() where /root/reference exists)"}), flush=True)
        return
    paths, n = sample_dataset(scale, index=True)
    O.ref_install_refgene(paths["refgene"])
    tmp = tempfile.mkdtemp(prefix="bkid_ref_")
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = O.ref_run_binary(paths["bam"], os.path.join(tmp, "ref"), paths["nib"])
        dt = time.perf_counter() - t0
        if r.returncode != 0:
            print(json.dumps({"impl": "reference", "unavailable": "BreakID_ref exited %d: %s" % (r.returncode, r.stderr[-200:])}), flush=True)
            return
        if i >= args.warmup:
            times.append(dt)
    ms = float(np.mean(times)) * 1e3
    val = n / 2.0 / (ms * 1e-3)
    calls = max(0, len(open(os.path.join(tmp, "ref_fusion_all.txt")).read().splitlines()) - 1) if os.path.exists(os.path.join(tmp, "ref_fusion_all.txt")) else None
    sample = "configs[1] x 1/%d: %d records, %d-byte BAM, BAM decode included (the reference has no other entry); oracle/_ref/BreakID_ref, single-threaded program " \
             "(host has %d cores), default AHC mode, whole process wall clock" % (round(1 / scale), n, os.path.getsize(paths["bam"]), os.cpu_count())
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
            "data": "synthetic (device-generated hg19-shaped genome, 2x150bp, planted TRA/INV/DUP/DEL, 1% chimeric noise)",
            "config": config_block(args),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": "reference", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "calls": calls}
    print(json.dumps(line), flush=True)


def _positive(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive, default=5, help="timed steps of every measurement")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the hg19-shaped 30x workload per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nib", action="store_true", help="also upload a random 4-bit genome so 41-mers are produced")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-legs", "--no-stress", dest="no_legs", action="store_true", help="skip the configs[2] / [3] / [4] / alignment legs")
    ap.add_argument("--no-decode", action="store_true", help="skip the decode-included e2e (BAM file -> device inflate -> hot path)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison on configs[1] x 1/16")
    ap.add_argument("--stress-scale", type=float, default=1.0, help="fraction of the 1e7-SA-record stress workload")
    ap.add_argument("--py-dist", action="store_true", help="N > 1: use the Python-orchestrated exchanges instead of the library's NCCL path")
    ap.add_argument("--dump-outputs", metavar="DIR", help="single GPU: write what the last timed step returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
