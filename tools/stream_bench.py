"""stream_bench.py -- cost of BAM on a pipe (bkid_push_bgzf_stream, BreakID -i -) on BASELINE.json configs[1] x 1/64.

Library: the sample BAM in a pinned host buffer is pushed as a stream of pieces of --pieces MiB (whole BGZF blocks each,
the way the driver cuts what it has read) and, alternating with it, as one file with push_bgzf; median of --steps timed
calls after one warm-up each.  A timed stream call is begin + every push + end.  Every stream must leave the columns
push_bgzf leaves.
Driver: wall time of `cat reads.bam | BreakID -i -` and of a level-0 (stored) copy of the same BAM on stdin against
`BreakID -i reads.bam`, same flags; the call files must agree.  The card's name and power limit are read in the same run.

    python tools/stream_bench.py [--scale 0.015625] [--steps 3] [--pieces 64,256,1024] [--out DIR]
Prints one JSON object (and writes it to DIR/stream_bench.json when --out is given)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import bench  # noqa: E402
from breakid_b200 import api, bamio  # noqa: E402
from sam_bench import COLS, card, pinned_copy  # noqa: E402


def piece_tables(table, piece_bytes):
    """cut the block table into pieces of whole blocks spanning at most piece_bytes: [(start, size, table rel. to start)]"""
    start = table["payload_off"].astype(np.int64) - 18            # every block of these files has XLEN 6
    end = (table["payload_off"] + table["payload_len"] + 8).astype(np.int64)
    out, b0 = [], 0
    while b0 < len(table):
        b1 = int(np.searchsorted(end, start[b0] + piece_bytes, side="right"))
        b1 = max(b1, b0 + 1)
        t = table[b0:b1].copy()
        t["payload_off"] -= np.uint64(start[b0])
        out.append((int(start[b0]), int(end[b1 - 1] - start[b0]), t))
        b0 = b1
    return out


def stored_copy(src, dst):
    """the same BAM with level-0 (stored) deflate blocks, as samtools view -u writes it"""
    f = api.BgzfFile(src)
    raw = open(src, "rb").read()
    with open(dst, "wb") as o:
        for b in f.block_table():
            u = zlib.decompress(raw[int(b["payload_off"]):int(b["payload_off"]) + int(b["payload_len"])], -15)
            if u:
                o.write(bamio._bgzf_block(u, 0))
        o.write(bamio._BGZF_EOF)
    f.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0 / 64)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--pieces", default="64,256,1024")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.init()
    paths, n = bench.sample_dataset(a.scale)
    if not os.path.exists(paths["bam"] + ".bai"):
        open(paths["bam"] + ".bai", "wb").close()               # the driver only checks that an index exists
    bf = api.BgzfFile(paths["bam"])
    bam = pinned_copy(paths["bam"])
    table = bf.block_table()
    names = (bf.target_len, bf.target_names)
    res = {"card": card(), "sample": "configs[1] x 1/%d, %d records" % (round(1 / a.scale), n), "bam_bytes": int(bam.numel()),
           "blocks": int(len(table)), "steps": a.steps}
    ref = api.Context(*names, device=0)
    ref.push_bgzf(bf, data_ptr=bam.data_ptr())
    want = {k: ref.fetch_column(k, dt) for k, dt in COLS}
    ref.close()

    def file_push(c):
        c.push_bgzf(bf, data_ptr=bam.data_ptr())

    def stream_push(pieces):
        def run(c):
            c.bgzf_stream_begin(bf.first_record)
            for s, size, t in pieces:
                c.push_bgzf_stream(size, t, data_ptr=bam.data_ptr() + s)
            c.bgzf_stream_end()
        return run

    sizes = [int(x) for x in a.pieces.split(",")]
    forms = {"push_bgzf": file_push}
    counts = {}
    for mb in sizes:
        pcs = piece_tables(table, mb << 20)
        forms["stream_%dMiB" % mb] = stream_push(pcs)
        counts["stream_%dMiB" % mb] = len(pcs)
    ms = {k: [] for k in forms}
    same = {}
    for it in range(a.steps + 1):                               # alternate the forms; iteration 0 warms each up
        for k, fn in forms.items():
            c = api.Context(*names, device=0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn(c)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if it:
                ms[k].append((t1 - t0) * 1e3)
            else:
                same[k] = all(np.array_equal(c.fetch_column(kk, dt), want[kk]) for kk, dt in COLS)
            c.close()
    res["library_ms"] = {k: {"ms": [round(x, 2) for x in v], "ms_median": round(float(np.median(v)), 2), "pieces": counts.get(k, 1)} for k, v in ms.items()}
    res["columns_equal_push_bgzf"] = same
    del bam
    torch.cuda.empty_cache()
    drv = os.path.join(ROOT, "breakid_b200", "host", "BreakID")
    stored = os.path.join(os.path.dirname(paths["bam"]), "reads_stored.bam")
    if not os.path.exists(stored):
        stored_copy(paths["bam"], stored + ".tmp")
        os.replace(stored + ".tmp", stored)
    res["stored_bam_bytes"] = os.path.getsize(stored)
    flags = ["-o", "{o}", "-n", paths["nib"], "-r", paths["refgene"]]
    runs = {"file": [drv, "-i", paths["bam"]] + flags, "stdin": "cat %s | %s -i - %s" % (paths["bam"], drv, " ".join(flags)),
            "stdin_stored": "cat %s | %s -i - %s" % (stored, drv, " ".join(flags))}
    res["driver"] = {}
    outs = {}
    for tag, cmd in runs.items():
        o = os.path.join(os.path.dirname(paths["bam"]), "out_streambench_" + tag)
        cmd = [x.replace("{o}", o) for x in cmd] if isinstance(cmd, list) else cmd.replace("{o}", o)
        shell = isinstance(cmd, str)
        subprocess.run(cmd, capture_output=True, text=True, shell=shell)          # warm-up (page cache, module load)
        walls = []
        for _ in range(a.steps):
            t0 = time.perf_counter()
            r = subprocess.run(cmd, capture_output=True, text=True, shell=shell)
            walls.append(time.perf_counter() - t0)
            assert r.returncode == 0, r.stderr[-500:]
        tm = dict(ln.split("\t") for ln in open(o + "_b200_timings.txt").read().splitlines())
        res["driver"][tag] = {"wall_s": [round(x, 3) for x in walls], "wall_s_median": round(float(np.median(walls)), 3),
                              "push_s": float(tm["push_s"]), "open_s": float(tm["open_s"]), "records": int(tm["records"]),
                              "pieces": int(tm.get("pieces", 0))}
        outs[tag] = open(o + "_fusion.txt").read()
    res["driver"]["same_fusion_txt"] = outs["stdin"] == outs["file"] == outs["stdin_stored"]
    bf.close()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        open(os.path.join(a.out, "stream_bench.json"), "w").write(s)


if __name__ == "__main__":
    main()
