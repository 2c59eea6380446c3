"""Device encoder (phase B of the compaction) alone: integer columns already in HBM -> PAX micro-blocks + column checksums.
--shape picks the columns (oceanbase_b200.synth.make_encode_columns: cfg5, lineitem, eventlog; generated on the device from a
seed), --encoding raw writes every column RAW (obgpu_encode_columns), auto lets every column's codec be chosen per micro-block
(obgpu_encode_columns_with + OBGPU_ENC_AUTO). Prints one JSON line: event-timed ms (median of the steps after warm-up), rows/s,
image bytes and their ratio to the RAW image of the same rows, algorithmic GB/s (input columns read once + image written once),
the card's name and power limit read in the same run, and with --host-threads N the host writer's encode_table rows/s over the
same rows with the same encodings."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:   # the measurement still stands; say what could not be read
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=64_000_000)
    ap.add_argument("--rows-per-block", type=int, default=500)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shape", choices=["cfg5", "lineitem", "eventlog"], default="cfg5")
    ap.add_argument("--encoding", choices=["raw", "auto"], default="raw")
    ap.add_argument("--host-threads", type=int, default=0, help="also time the host writer over the same rows (0: skip)")
    ap.add_argument("--seed", type=int, default=5)
    a = ap.parse_args()
    import torch
    import oceanbase_b200 as ob
    from oceanbase_b200 import capi, compaction
    from oceanbase_b200.synth import make_encode_columns
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = ob.ScanContext(0, stream=stream.cuda_stream)   # CUDA events below time the stream the kernels run on
    n = a.rows
    dcols = make_encode_columns(a.shape, n, seed=a.seed)
    cols = [(v.data_ptr(), None if nl is None else nl.data_ptr(), t, False) for (t, v, nl) in dcols]
    encodings = None if a.encoding == "raw" else [capi.ENC_AUTO] * len(cols)
    in_bytes = sum(n * 8 + (n if nl is not None else 0) for (_t, _v, nl) in dcols)
    torch.cuda.synchronize()

    def encode(enc):
        if enc is None:   # the entry point every existing caller uses
            return compaction.encode_columns(ctx, cols, n, a.rows_per_block, rowkey_cnt=1)
        return compaction.encode_columns(ctx, cols, n, a.rows_per_block, rowkey_cnt=1, encodings=enc)

    ms, img_bytes, nb, host_blocks = [], 0, 0, 0
    for it in range(a.warmup + a.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        enc = encode(encodings)
        e1.record()
        torch.cuda.synchronize()
        info = enc.info()
        img_bytes, nb, host_blocks = info.image_size, info.n_blocks, info.n_host_blocks
        enc.free()
        if it >= a.warmup:
            ms.append(e0.elapsed_time(e1))
    raw = encode(None)
    raw_bytes = raw.info().image_size
    raw.free()
    t = float(np.median(ms))
    name, power = card()
    out = {"workload": f"device encoder, {a.shape} columns, {a.encoding}", "rows": n, "rows_per_block": a.rows_per_block, "n_blocks": nb,
           "n_host_blocks": host_blocks, "ms": round(t, 3), "ms_min": round(float(np.min(ms)), 3), "ms_max": round(float(np.max(ms)), 3),
           "rows_per_s": n / t * 1e3, "in_bytes": in_bytes, "image_bytes": img_bytes, "raw_image_bytes": raw_bytes,
           "image_vs_raw": round(img_bytes / raw_bytes, 4), "alg_gbps": round((in_bytes + img_bytes) / t / 1e6, 1),
           "gpu": name, "power_limit": power,
           "note": "event-timed around one encode call (includes its allocation); median of the steps after warm-up"}
    if a.host_threads > 0:
        from oceanbase_b200.sstable import Column, encode_table
        hcols = [Column(tt, capi.ENC_RAW if encodings is None else capi.ENC_AUTO, v.cpu().numpy(),
                        nulls=None if nl is None else nl.cpu().numpy()) for (tt, v, nl) in dcols]
        t0 = time.perf_counter()
        table = encode_table(hcols, a.rows_per_block, rowkey_cnt=1, n_threads=a.host_threads)
        dt = time.perf_counter() - t0
        out.update({"host_threads": a.host_threads, "host_rows_per_s": n / dt, "host_image_bytes": int(table.image.size),
                    "host_note": "obgpu_writer_encode_table wall time, same rows and encodings, one run"})
    print(json.dumps(out))


if __name__ == "__main__":
    main()
