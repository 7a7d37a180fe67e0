"""sam_bench.py -- cost of SAM input (bkid_push_sam, BreakID -i reads.sam) on BASELINE.json configs[1] x 1/64.

The sample's records are written as SAM text (bamio.write_sam, the records bench.sample_dataset writes as BAM) and
measured four ways, median of --steps timed calls after one warm-up call each:
  push_sam      the whole call from a pinned host copy of the text (copy + line split + parse, chunks overlapped)
  device_parse  the device time of line split + parse alone (decode stats: from the moment each chunk's copy has landed)
  push_bgzf     the BAM holding the same records, also from a pinned host copy
  driver        BreakID end to end on reads.sam against reads.bam (wall time, same flags)
Every timed push is checked to leave the same columns as push_bgzf.  The card's name and power limit are read in the same
run.

    python tools/sam_bench.py [--scale 0.015625] [--steps 3] [--out DIR]
Prints one JSON object (and writes it to DIR/sam_bench.json when --out is given)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import bench  # noqa: E402
from breakid_b200 import api, bamio, synth  # noqa: E402

COLS = (("flag", np.uint16), ("pos", np.int32), ("endpos", np.int32), ("x_name_hash", np.uint64), ("cig_ops", np.uint32), ("sa_txt", np.uint8), ("seq4", np.uint8))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def pinned_copy(path, offset=0):
    size = os.path.getsize(path) - offset
    buf = torch.empty(size, dtype=torch.uint8, pin_memory=True)
    with open(path, "rb") as f:
        f.seek(offset)
        f.readinto(memoryview(buf.numpy()))
    return buf


def timed(push, steps):
    ms, stats, ctx = [], None, None
    for it in range(steps + 1):
        if ctx is not None:
            ctx.close()
        ctx = push.ctx()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        push(ctx)
        t1 = time.perf_counter()
        if it:
            ms.append((t1 - t0) * 1e3)
            stats = ctx.decode_stats()
    return ms, stats, ctx


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0 / 64)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.init()
    paths, n = bench.sample_dataset(a.scale)
    if not os.path.exists(paths["bam"] + ".bai"):
        open(paths["bam"] + ".bai", "wb").close()               # the driver only checks that an index exists
    sam = os.path.join(os.path.dirname(paths["bam"]), "reads.sam")
    if not os.path.exists(sam):
        t0 = time.time()
        bamio.write_sam(sam + ".tmp", synth.generate(bench.workload_cfg(a.scale)))
        os.replace(sam + ".tmp", sam)
        print("wrote %s in %.1f s" % (sam, time.time() - t0), file=sys.stderr)
    sf = api.SamFile(sam)
    bf = api.BgzfFile(paths["bam"])
    text = pinned_copy(sam, sf.first_record)
    bam = pinned_copy(paths["bam"])
    names = (bf.target_len, bf.target_names)

    class Push:
        def __init__(self, fn):
            self.fn = fn

        def ctx(self):
            return api.Context(*names, device=0)

        def __call__(self, c):
            return self.fn(c)

    res = {"card": card(), "sample": "configs[1] x 1/%d, %d records" % (round(1 / a.scale), n),
           "sam_text_bytes": int(text.numel()), "bam_bytes": int(bam.numel()), "steps": a.steps}
    ms_s, st_s, cs = timed(Push(lambda c: c.push_sam(b"", sf.first_line, data_ptr=text.data_ptr(), size=text.numel())), a.steps)
    ms_b, st_b, cb = timed(Push(lambda c: c.push_bgzf(bf, data_ptr=bam.data_ptr())), a.steps)
    same = all(np.array_equal(cs.fetch_column(k, dt), cb.fetch_column(k, dt)) for k, dt in COLS)
    nrec = st_s["n_records"]
    med = float(np.median(ms_s))
    dev = st_s["boundaries_ms"] + st_s["extract_ms"]
    res["push_sam"] = {"ms": [round(x, 2) for x in ms_s], "ms_median": round(med, 2), "text_gbs": round(text.numel() / med / 1e6, 2),
                       "records_per_s": round(nrec / med * 1e3), "n_chunks": st_s["n_chunks"], "records": nrec}
    res["device_parse"] = {"lines_ms": round(st_s["boundaries_ms"], 2), "parse_ms": round(st_s["extract_ms"], 2), "ms": round(dev, 2),
                           "text_gbs": round(text.numel() / dev / 1e6, 2), "records_per_s": round(nrec / dev * 1e3)}
    res["push_bgzf"] = {"ms": [round(x, 2) for x in ms_b], "ms_median": round(float(np.median(ms_b)), 2), "inflate_ms": round(st_b["inflate_ms"], 2),
                        "boundaries_ms": round(st_b["boundaries_ms"], 2), "extract_ms": round(st_b["extract_ms"], 2)}
    res["columns_equal_push_bgzf"] = bool(same) and st_s["n_records"] == st_b["n_records"]
    cs.close(); cb.close()
    del text, bam
    torch.cuda.empty_cache()
    # pinned H2D rate of the text's size, measured here: is the ingest copy-bound?
    h = torch.empty(res["sam_text_bytes"], dtype=torch.uint8, pin_memory=True)
    g = torch.empty_like(h, device="cuda")
    h2d = []
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.copy_(h, non_blocking=True); e1.record(); torch.cuda.synchronize()
        h2d.append(e0.elapsed_time(e1))
    h2d_ms = float(np.median(h2d[1:]))
    res["h2d_of_text"] = {"ms": round(h2d_ms, 2), "gbs": round(res["sam_text_bytes"] / h2d_ms / 1e6, 2)}
    res["device_parse_faster_than_copy"] = dev < h2d_ms
    del h, g
    torch.cuda.empty_cache()
    drv = os.path.join(ROOT, "breakid_b200", "host", "BreakID")
    res["driver"] = {}
    outs = {}
    for tag, inp in (("bam", paths["bam"]), ("sam", sam)):
        o = os.path.join(os.path.dirname(paths["bam"]), "out_sambench_" + tag)
        cmd = [drv, "-i", inp, "-o", o, "-n", paths["nib"], "-r", paths["refgene"]]
        subprocess.run(cmd, capture_output=True, text=True)                       # warm-up (page cache, module load)
        walls = []
        for _ in range(a.steps):
            t0 = time.perf_counter()
            r = subprocess.run(cmd, capture_output=True, text=True)
            walls.append(time.perf_counter() - t0)
            assert r.returncode == 0, r.stderr[-500:]
        tm = dict(ln.split("\t") for ln in open(o + "_b200_timings.txt").read().splitlines())
        res["driver"][tag] = {"wall_s": [round(x, 3) for x in walls], "wall_s_median": round(float(np.median(walls)), 3),
                              "push_s": float(tm["push_s"]), "open_s": float(tm["open_s"]), "records": int(tm["records"])}
        outs[tag] = open(o + "_fusion.txt").read()
    res["driver"]["same_fusion_txt"] = outs["bam"] == outs["sam"]
    sf.close(); bf.close()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        open(os.path.join(a.out, "sam_bench.json"), "w").write(s)


if __name__ == "__main__":
    main()
