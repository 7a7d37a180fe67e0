"""sort_bench.py -- cost of bkid_sort_records (BreakID -sort) on BASELINE.json configs[1] at full size.

Per input order (coordinate = the cost of the order check alone, name-grouped as `bwa mem | samblaster` writes it, random):
the bkid_sort_records time after a warm-up call (the columns are re-pushed before every timed call), records/s, the bytes
per record the algorithm moves (counted from the kernels in breakid_b200/csrc/bkid_sort.cuh), device memory from
cudaMemGetInfo before the push, after the push and after the sort (the context keeps its sort scratch), and a check of
tid / pos / flag against torch.sort(stable=True) of the same key.  Then end to end: the 1/64 sample BAM written
name-grouped and run with `BreakID -sort`, against the coordinate-sorted BAM run without it.

    python tools/sort_bench.py [--scale 1.0] [--steps 3] [--out DIR]
Prints one JSON object (and writes it to DIR/sort_bench.json when --out is given)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import bench  # noqa: E402
from breakid_b200 import api, bamio, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def key_bits(n_targets, max_pos1):
    return int(n_targets).bit_length() + int(max_pos1).bit_length() + 1


def bytes_per_record(kbits, row_bytes, n_x, n_sa, n):
    """HBM bytes per record the kernels of bkid_sort.cuh read + write (a random 4- or 8-byte access counted as one 32-byte
    sector); sparse / SA rows amortised over all records"""
    npass = (kbits + 7) // 8
    b = 8                                   # sort_check: tid + pos
    b += 10 + 12                            # sort_keys: tid, pos, flag -> key + index
    b += 8 + npass * 24                     # onesweep: histogram read + per pass key/value in and out
    b += 7 + row_bytes                      # pack: flag, mapq, isize16, span16 -> row
    b += 12 + 32 + 15                       # unpack: key + index, one random row sector, the columns written
    if n_x or n_sa:
        b += 8 + 4 + 32 + 2                 # slot maps cleared, new order: index + random slot sector, two flags
        b += 2 * (1 + 4 + 1 + 4)            # two scans of the flags + emit reading flags / offsets
    b += (n_x * (4 + 32 + 4 * 2 + 32 + 28 * 2) + n_sa * 200) / max(n, 1)
    return b


def timed_sorts(d, steps, label):
    dev = d.cols["flag"].device
    out = {"order": label}
    free0, total = torch.cuda.mem_get_info()
    b, keep = bench.device_batch(d)
    tl = d.cfg.chrom_lens
    ctx = api.Context(tl, [synth.chrom_name(t) for t in range(len(tl))], device=0)
    ms, was = [], None
    for it in range(steps + 1):
        if it:
            ctx.reset()
        ctx.push_device(b)
        torch.cuda.synchronize()
        free1 = torch.cuda.mem_get_info()[0]
        t0 = time.perf_counter()
        was = ctx.sort_records()
        t1 = time.perf_counter()
        if it:
            ms.append((t1 - t0) * 1e3)
    free2 = torch.cuda.mem_get_info()[0]
    n = d.n
    tid, pos, flag = d.cols["tid"], d.cols["pos"], d.cols["flag"]
    rank = torch.where(tid < 0, torch.full_like(tid, len(tl)), tid).to(torch.int64)
    key = (rank << 33) | ((pos.to(torch.int64) + 1) << 1) | ((flag.to(torch.int64) >> 4) & 1)
    del rank
    # already sorted: nothing moves (the file's tie order is kept); otherwise torch.sort(stable=True) of the same key
    perm = torch.arange(n, device=dev) if was else torch.sort(key, stable=True)[1]
    del key
    ok = True
    for k, col, dt in (("tid", tid, np.int32), ("pos", pos, np.int32), ("flag", flag, np.uint16)):
        got = torch.from_numpy(ctx.fetch_column(k, dt).view(np.int16 if dt == np.uint16 else dt)).to(dev)
        ok &= bool(torch.equal(got, col[perm]))
        del got
    del perm
    max_p1 = int(pos.max()) + 1
    kb = key_bits(len(tl), max_p1)
    row = 8 if ("isize16" in keep and "span16" in keep) else 16
    med = float(np.median(ms))
    out.update({"records": n, "was_sorted": bool(was), "sort_ms": [round(x, 3) for x in ms], "sort_ms_median": round(med, 3),
                "records_per_s": n / (med / 1e3), "key_bits": kb,
                "bytes_per_record": None if was else round(bytes_per_record(kb, row, b.n_x, b.n_sa, n), 1),
                "device_free_gb": {"before_push": free0 / 1e9, "after_push": free1 / 1e9, "after_sort": free2 / 1e9, "total": total / 1e9},
                "matches_torch_sort_stable": ok})
    if not was:
        out["achieved_gbs"] = round(out["bytes_per_record"] * n / (med / 1e3) / 1e9, 1)
    ctx.close()
    del keep, b
    torch.cuda.empty_cache()
    return out


def end_to_end(scale):
    paths, n = bench.sample_dataset(scale)
    if not os.path.exists(paths["bam"] + ".bai"):
        open(paths["bam"] + ".bai", "wb").close()          # the driver only checks that an index exists
    gdir = tempfile.mkdtemp(prefix="bkid_sort_grouped_")
    d = synth.generate(bench.workload_cfg(scale))
    order = torch.argsort(d.cols["name_id"], stable=True)
    pg = bamio.write_dataset(gdir, synth.permute(d, order), sort_order="queryname")
    drv = os.path.join(ROOT, "breakid_b200", "host", "BreakID")
    res = {}
    for tag, p, extra in (("sorted_bam", paths, []), ("name_grouped_bam_sort", pg, ["-sort"])):
        o = os.path.join(gdir, "out_" + tag)
        cmd = [drv, "-i", p["bam"], "-o", o, "-n", p["nib"], "-r", p["refgene"]] + extra
        subprocess.run(cmd, capture_output=True, text=True)                       # warm-up (page cache, module load)
        t0 = time.perf_counter()
        r = subprocess.run(cmd, capture_output=True, text=True)
        wall = time.perf_counter() - t0
        assert r.returncode == 0, r.stderr[-500:]
        tm = dict(ln.split("\t") for ln in open(o + "_b200_timings.txt").read().splitlines())
        res[tag] = {"wall_s": round(wall, 3), "sort_ms": float(tm.get("sort_ms", 0)), "records": int(tm["records"])}
    same = all(open(os.path.join(gdir, "out_sorted_bam") + s).read() == open(os.path.join(gdir, "out_name_grouped_bam_sort") + s).read()
               for s in ("_fusion.txt",))
    res["same_fusion_txt"] = same
    res["sort_share_of_wall"] = round(res["name_grouped_bam_sort"]["sort_ms"] / 1e3 / res["name_grouped_bam_sort"]["wall_s"], 4)
    res["sample"] = "configs[1] x 1/%d, %d records" % (round(1 / scale), n)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of configs[1] for the sort timings")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--e2e-scale", type=float, default=1.0 / 64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.init()
    res = {"card": card(), "workload": "BASELINE.json configs[1] x %g, built on the device (bench.device_batch), AHC" % a.scale, "orders": []}
    d = synth.generate(bench.workload_cfg(a.scale), device="cuda")
    n = d.n
    for label in ("coordinate", "name_grouped", "random"):
        if label == "coordinate":
            dd = d
        elif label == "name_grouped":
            dd = synth.permute(d, torch.argsort(d.cols["name_id"], stable=True))
        else:
            g = torch.Generator(device="cuda"); g.manual_seed(5)
            dd = synth.permute(d, torch.randperm(n, device="cuda", generator=g))
        res["orders"].append(timed_sorts(dd, a.steps, label))
        del dd
        torch.cuda.empty_cache()
    del d
    torch.cuda.empty_cache()
    res["end_to_end"] = end_to_end(a.e2e_scale)
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        open(os.path.join(a.out, "sort_bench.json"), "w").write(s)


if __name__ == "__main__":
    main()
