#!/usr/bin/env python
"""bench.py -- columnar-scan hot path benchmark (contract: task statement section 4, SURVEY.md 8d).

    python bench.py --gpus N --steps K --warmup W            # our B200 path
    python bench.py --impl reference --gpus N --steps K ...   # the reference CPU algorithm (oracle port)

Headline workload = BASELINE.json configs[2] ("cfg3", the north-star target): a 1-billion-row, 16-column
dictionary-encoded SSTable (8 INT64 DICT + 8 VARCHAR DICT, Zipf(1.1) over per-column dictionaries), micro-blocks
cut at the reference's 16 KiB target, 3-predicate AND filter (~10 %), 4 INT64 + 2 VARCHAR columns projected.
A "step" is one pass of the hot path (skip nothing: filter -> selection -> projection) over the whole table.
The 1 B rows are split over the ranks (strong scaling: every rank scans 1 B / N rows, no data-path collective).
A rank generates ONE seeded segment of its shard on the host (SplitMix64 columns, ~2 GB encoded) and tiles it in
HBM (`config.tiles` physically distinct copies): generating 125 GB of blocks on the box's 16-CPU quota would take
an hour, and every tile (2 GB) is far larger than L2 (126 MB), so timed iterations never see a warm cache.
`secondary.cfg2` repeats the measurement on BASELINE.json configs[1] (100 M rows x 8 INT64 per GPU, weak).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # a benchmark run leaves the tree as it found it

import numpy as np  # noqa: E402

METRIC = "decoded+filtered rows/sec"
UNIT = "rows/s"
BATCH_ROWS = 256  # _rowsets_max_rows default (src/share/parameter/ob_parameter_seed.ipp:418)
CFG3_NAME = ("cfg3: 1 B rows x 16 dict-encoded columns (8 INT64 DICT + 8 VARCHAR DICT), 16 KiB micro-blocks, "
             "3-predicate AND ~10 %, 4 INT64 + 2 VARCHAR projected")


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def host_cpus():
    """Host threads this process can actually run: min(affinity mask, cgroup cpu.max quota). The GPU
    boxes expose 128 logical CPUs but cap the container at a 16-CPU quota; running more threads than
    the quota only gets them throttled."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    n = min(n, max(1, int(int(parts[0]) / int(parts[1]) + 0.5)))
            else:
                quota = int(parts[0])
                if quota > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                        n = min(n, max(1, int(quota / int(f.read()) + 0.5)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def gpu_numa_node(local):
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            return int(f.read().strip())
    except Exception:
        return None


def bind_to_gpu_numa_node(local):
    """Pin this process (and the threads / first-touched pages it creates from now on) to the CPUs of the
    NUMA node the GPU hangs off, so that the pinned host image and result buffers sit next to the PCIe root
    the copies go through. Returns the node number or None when it cannot be determined."""
    try:
        node = gpu_numa_node(local)
        if node is None or node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def build_workload(rows, row_start, seed, chunk_rows=4_000_000, pinned=False, n_threads=0, maker=None,
                   rows_per_block=1400, align_chunks=False):
    """Table of `rows` rows (config 2, or `maker`'s) generated in chunks (bounded host memory), packed
    into one image (optionally pinned host memory = the host-side block cache)."""
    from concurrent.futures import ThreadPoolExecutor
    from oceanbase_b200.synth import make_config2_like
    from oceanbase_b200.sstable import TableImage
    maker = maker or make_config2_like

    if align_chunks:   # chunks end on block boundaries: no ragged block inside the table
        chunk_rows = max(rows_per_block, chunk_rows // rows_per_block * rows_per_block)
    starts = list(range(0, rows, chunk_rows))
    ncpu = host_cpus()
    workers = max(1, min(8, ncpu // 4, len(starts)))
    per = max(1, (n_threads or ncpu) // workers)

    def gen(s):
        n = min(chunk_rows, rows - s)
        return maker(rows=n, rows_per_block=rows_per_block, seed=seed, row_start=row_start + s, n_threads=per)

    with ThreadPoolExecutor(workers) as ex:
        parts = list(ex.map(gen, starts))
        w0 = parts[0]
        sizes = [len(p.table.image) for p in parts]
        total = sum(sizes)
        if pinned:
            import torch
            buf = torch.empty(total, dtype=torch.uint8, pin_memory=True)
            image = buf.numpy()
        else:
            buf = None
            image = np.empty(total, dtype=np.uint8)
        pos = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)

        def place(i):  # parallel first touch: pages spread over the NUMA nodes of the copying threads
            image[pos[i]:pos[i + 1]] = parts[i].table.image
            return parts[i].table.offsets + pos[i]

        offs = list(ex.map(place, range(len(parts))))
    table = TableImage(image, np.concatenate(offs), np.concatenate([p.table.sizes for p in parts]),
                       sum(p.table.total_rows for p in parts), w0.table.n_cols)
    w0.table = table
    return w0, buf


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(name, rows):
    """DRAM bytes per scan from the committed ncu capture (profiles/<name>), scaled by rows when the capture was
    taken on a smaller tiling of the same segment (traffic per row is a property of the blocks); null if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", name)) as f:
            t = json.load(f)
        return int(round(float(t["total"]) * float(rows) / float(t["rows"])))
    except Exception:
        return None


def cpu_reference_leg(w, steps, warmup, n_threads, sample_blocks):
    """Times the oracle port of the reference CPU path (tests/oracle_binding.py) on a bounded
    sample of the workload: first `sample_blocks` micro-blocks, all host threads."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as ora
    rates, rows, sel = [], 0, 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        rows, sel, _ = ora.scan_table_mt(w.table, w.filter, w.proj, batch_size=BATCH_ROWS, n_threads=n_threads,
                                         block_limit=sample_blocks)
        dt = time.perf_counter() - t0
        if i >= warmup:
            rates.append((rows / dt, dt))
    return rates, rows, sel


# ---- workloads -----------------------------------------------------------------------------------------------
def cfg3_shape(args, world):
    """(rows per GPU, tiles, segment rows): rows per GPU = total / world, cut into `tiles` copies of one segment."""
    per_gpu = args.rows // max(world, 1)
    # the host threads are shared by the ranks (cgroup quota / world each): generate a smaller segment per rank on wide jobs so that
    # the untimed set-up stays around half a minute (a tile is still several hundred MB, far beyond L2)
    seg_cap = max(2_000_000, args.segment_rows // max(1, world // 2))
    tiles = max(1, -(-per_gpu // seg_cap))
    seg = per_gpu // tiles
    return seg * tiles, tiles, seg


def cfg3_config(args, world, rpb, seg_rows, tiles, seg_table=None, selectivity=None, extra=None):
    cfg = {"workload": CFG3_NAME, "rows": int(seg_rows) * tiles * world, "columns": 16,
           "micro_block_target_bytes": 16384, "rows_per_block": int(rpb), "segment_rows": int(seg_rows),
           "tiles_per_gpu": int(tiles), "seed": args.seed}
    if seg_table is not None:
        cfg["encoded_bytes_per_row"] = round(float(seg_table.sizes.sum()) / seg_table.total_rows, 3)
        cfg["mean_block_bytes"] = round(float(seg_table.sizes.mean()), 1)
    if selectivity is not None:
        cfg["selectivity"] = selectivity
    if extra:
        cfg.update(extra)
    return cfg


def make_cfg3_segment(args, rank, world, pinned):
    from oceanbase_b200.synth import make_config3_like, rows_per_block_for_target
    rpb = args.rows_per_block or rows_per_block_for_target(make_config3_like, seed=args.seed)
    rows_gpu, tiles, seg_rows = cfg3_shape(args, world)
    w, buf = build_workload(seg_rows, rank * rows_gpu, args.seed, chunk_rows=1_000_000, pinned=pinned,
                            maker=make_config3_like, rows_per_block=rpb, align_chunks=True,
                            n_threads=max(1, host_cpus() // max(1, min(world, 8))))
    return w, buf, rpb, tiles, seg_rows


def run_reference(args):
    rank = env_int("RANK", 0)
    world = env_int("WORLD_SIZE", 1)
    if rank != 0:
        return 0
    import __graft_entry__ as g
    g.build_cpu_side()
    ncpu = host_cpus()
    if args.workload == "cfg3":
        # the same table definition as our arm; one step = one pass over a bounded sample (the first ref_rows rows of
        # rank 0's segment) with every host thread
        rows_gpu, tiles, seg_rows = cfg3_shape(args, world)
        a2 = argparse.Namespace(**vars(args))
        w, _, rpb, _, _ = make_cfg3_segment(a2, 0, world, pinned=False)
        sample_blocks = max(1, min(w.table.n_blocks, args.ref_rows // rpb))
        config = cfg3_config(args, world, rpb, seg_rows, tiles, w.table)
        what = "the cfg3 table"
    else:
        w, _ = build_workload(args.ref_rows, 0, args.seed)
        sample_blocks = None
        config = {"workload": w.name, "rows_per_gpu": args.cfg2_rows, "columns": 8}
        what = "the config-2 table"
    rates, rows, sel = cpu_reference_leg(w, args.steps, args.warmup, ncpu, sample_blocks)
    best = max(r for r, _ in rates)
    mean_dt = float(np.mean([d for _, d in rates]))
    value = rows / mean_dt
    config["selectivity"] = sel / max(rows, 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": mean_dt * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.workload == "cfg3" else "weak", "vs_baseline": None, "dtype": "int64/bytes", "data": "synthetic",
        "config": config,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ncpu, "kind": "port",
                         "sample": f"{rows} rows ({sample_blocks or w.table.n_blocks} micro-blocks) of {what} per step "
                                   f"(rate metric: the table is a repetition of such segments), "
                                   f"oracle port of the reference scan (batch {BATCH_ROWS}), {ncpu} threads (cgroup cpu quota of the box; "
                                   f"{os.cpu_count()} logical CPUs visible), 32-block granules claimed dynamically",
                         "best": best},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


class DeviceRun:
    """Device-resident measurement of one workload: K timed scans of one page batch."""

    def __init__(self, ctx, stream, batch, w, cap, world, dist):
        self.ctx, self.stream, self.batch, self.w, self.cap, self.world, self.dist = ctx, stream, batch, w, cap, world, dist

    def barrier(self):
        import torch
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def run(self, steps, warmup, local, rank, dump=None):
        """dump: called with the last timed step's result (after the timed region) before it is freed."""
        import torch
        batch, w, cap, ctx = self.batch, self.w, self.cap, self.ctx
        for _ in range(warmup):
            r = batch.scan(w.filter, w.proj, max_selected_rows=cap)
            r.info()
            r.free()
        sampler = ClockSampler(local)
        self.barrier()
        if rank == 0:
            sampler.start()
            time.sleep(0.3)
        launches0 = ctx.launch_count
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        ev0.record(self.stream)
        last = None
        for _ in range(steps):
            if last is not None:
                last.free()
            last = batch.scan(w.filter, w.proj, max_selected_rows=cap)
        ev1.record(self.stream)
        self.barrier()
        clocks = sampler.stop() if rank == 0 else None
        launches = ctx.launch_count - launches0
        step_ms = ev0.elapsed_time(ev1) / steps
        info = last.info()  # raises on overflow / unsupported
        kern_ms = float(np.mean(ctx.kernel_times_ms(min(steps, 256))))
        if dump is not None:
            dump(last)
        last.free()
        return step_ms, kern_ms, int(info.selected_rows), int(launches), clocks


DUMP_WINDOWS = 32          # --dump-outputs: seeded windows of consecutive result rows ...
DUMP_WINDOW_ROWS = 2048    # ... of this many rows each (every row when fewer are selected)
DUMP_LIMIT_BYTES = 32 << 20  # per workload: the headline and its cfg2 secondary stay within 64 MB together


def dump_scan_result(res, w, out_dir, prefix):
    """Writes what a caller of the timed scan receives, as float arrays two builds can compare exactly, into
    out_dir/<prefix><name>.npy: selected_rows [1]; rows, the result row indices of the sample; per projected column i
    proj<i>_null (0 / 1) and either proj<i> [rows, 2] float64 (high and low 32 bits of the value) or, for strings,
    proj<i>_len and proj<i>_bytes (the sampled strings concatenated, one float32 per byte). A string cell comes back as an
    address into the image, which differs from run to run, so the bytes it points at are written instead."""
    n = int(res.selected_rows)
    if n <= DUMP_WINDOWS * DUMP_WINDOW_ROWS:
        windows = [(0, n)]
    else:
        picked = np.random.default_rng(0).choice(n // DUMP_WINDOW_ROWS, DUMP_WINDOWS, replace=False)
        windows = [(int(s) * DUMP_WINDOW_ROWS, DUMP_WINDOW_ROWS) for s in np.sort(picked)]
    out = {"selected_rows": np.array([n], dtype=np.float64),
           "rows": np.concatenate([np.arange(s, s + k, dtype=np.float64) for s, k in windows])}
    for i in range(len(w.proj)):
        vals, nulls, lens, heaps = [], [], [], []
        for s, k in windows:
            data, aux, words = res.fetch_col(i, s, k)
            r = np.arange(k)
            nulls.append(((words[r // 64] >> (r % 64).astype(np.uint64)) & np.uint64(1)).astype(np.float32))
            if w.proj_is_string[i]:
                lens.append(aux.astype(np.float32))
                heaps.append(res.fetch_strings(i, s, k)[0].astype(np.float32))
            else:
                v = data.astype(np.uint64)
                vals.append(np.stack([(v >> np.uint64(32)).astype(np.float64), (v & np.uint64(0xffffffff)).astype(np.float64)], axis=1))
        out[f"proj{i}_null"] = np.concatenate(nulls)
        if w.proj_is_string[i]:
            out[f"proj{i}_len"] = np.concatenate(lens)
            out[f"proj{i}_bytes"] = np.concatenate(heaps)
        else:
            out[f"proj{i}"] = np.concatenate(vals)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes for {prefix} exceed {DUMP_LIMIT_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), a)


def e2e_run(local, table, w, rows_per_block, sel_hint, args, repeats, barrier, zero_copy=False):
    """Host buffers in, host vectors out through the library's host-buffer entry (include/obgpu_pipeline.h:
    obgpu_pipeline_scan, n streams overlapping H2D / kernels / D2H); `repeats` passes over the host table per step (the
    tiled table: every pass is a real H2D of the segment and a real D2H of its results into pinned output buffers)."""
    import torch
    from oceanbase_b200.pipeline import HostScanPipeline, HostOutputs
    bpb = max(1, table.n_blocks // args.e2e_batches)
    pipe = HostScanPipeline(local, n_workers=args.e2e_workers)
    n_parts, cap = pipe.plan(table, w.filter, w.proj, bpb, sel_hint, ramp=args.e2e_ramp)
    outputs = HostOutputs.allocate(int(cap * 1.1) + 65536, w.proj_is_string, w.proj_elem_len, pinned=True)
    stats = {"d2h": 0, "h2d": 0, "launches": 0}

    def one_pass():
        out = pipe.scan(table, w.filter, w.proj, bpb, sel_hint, outputs=outputs, ramp=args.e2e_ramp,
                        string_base=table.image.ctypes.data, zero_copy=zero_copy)
        stats["d2h"] += out.d2h_bytes
        stats["h2d"] += out.h2d_bytes
        stats["launches"] += out.kernel_launches
        return out.selected_rows

    one_pass()   # warm-up: contexts, pools, page faults of the output buffers
    steps = max(1, args.e2e_steps)
    barrier()
    stats = {"d2h": 0, "h2d": 0, "launches": 0}
    t0 = time.perf_counter()
    n = 0
    for _ in range(steps):
        n = sum(one_pass() for _ in range(repeats))
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps   # wall clock: every worker stream is drained by each call
    barrier()
    pipe.close()
    return ms, n, stats["h2d"] // steps, stats["d2h"] // steps, n_parts, steps, stats["launches"]


def run_ours(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0 and os.access(ROOT, os.W_OK):   # a read-only tree is run as build() left it
        g.build()
    if world > 1:
        dist.barrier()
    import oceanbase_b200 as ob
    from oceanbase_b200.sstable import TableImage
    from oceanbase_b200.synth import referenced_bytes, filter_columns

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_node = None if args.no_numa_bind else bind_to_gpu_numa_node(local)
    if numa_node is None:
        numa_node = gpu_numa_node(local)
    stream = torch.cuda.Stream(device=dev)   # a dedicated (non-default) torch stream: the ctx launches on it
    torch.cuda.set_stream(stream)
    ctx = ob.ScanContext(local, stream=stream.cuda_stream)
    ctx.set_profiling(True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        if world == 1:
            return list(vals)
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    def allsum(vals):
        if world == 1:
            return list(vals)
        t = torch.tensor(list(vals), device=dev, dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.tolist()

    def dumper(name, w):
        if not args.dump_outputs or rank != 0:
            return None
        return lambda res: dump_scan_result(res, w, args.dump_outputs, name + "_")

    # every rank pins its host buffers next to ITS GPU: report all of them, not rank 0's
    numa_all = [numa_node if numa_node is not None else -1]
    if world > 1:
        t = torch.full((world,), -2, device=dev, dtype=torch.int64)
        t[rank] = numa_all[0]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        numa_all = t.tolist()

    peak, peak_src = measured_peak_gbs()
    line = None
    if args.workload == "cfg3":
        t_gen = time.perf_counter()
        w, pinned_buf, rpb, tiles, seg_rows = make_cfg3_segment(args, rank, world, pinned=True)
        t_gen = time.perf_counter() - t_gen
        seg = w.table
        stride = (seg.image.size + 127) // 128 * 128
        d_image = torch.empty(stride * tiles + 64, dtype=torch.uint8, device=dev)
        d_image[stride * tiles:].zero_()
        d_image[:seg.image.size].copy_(pinned_buf, non_blocking=True)
        if stride > seg.image.size:
            d_image[seg.image.size:stride].zero_()
        for k in range(1, tiles):                       # physically distinct copies of the segment in HBM
            d_image[k * stride:(k + 1) * stride].copy_(d_image[:stride], non_blocking=True)
        torch.cuda.synchronize()
        offs = (seg.offsets[None, :] + (np.arange(tiles, dtype=np.int64) * stride)[:, None]).reshape(-1)
        table = TableImage(None, offs, np.tile(seg.sizes, tiles), seg.total_rows * tiles, seg.n_cols)
        batch = ctx.open_batch(table, device_image_ptr=d_image.data_ptr(), host_view=False, image_size=stride * tiles)
        cap = int(table.total_rows * 0.13)
        run = DeviceRun(ctx, stream, batch, w, cap, world, dist)
        step_ms, kern_ms, selected, launches, clocks = run.run(args.steps, args.warmup, local, rank, dump=dumper("cfg3", w))
        batch.close()
        del d_image
        torch.cuda.empty_cache()
        # e2e: the host segment goes through the host-buffer API `tiles` times per step (every pass a real H2D / D2H)
        e2e_tiles = tiles if not args.e2e_one_tile else 1
        e2e_ms, n_e2e, h2d, d2h, n_parts, e2e_steps, e2e_launches = e2e_run(local, seg, w, rpb, 0.14, args, e2e_tiles, barrier)
        # zero copy: the pinned host segment is opened in place and the kernels pull the referenced regions over PCIe themselves
        zc_ms, zc_d2h = None, 0
        if args.e2e_mode != "staged":
            zc_ms, _, _, zc_d2h, _, _, _ = e2e_run(local, seg, w, rpb, 0.14, args, e2e_tiles, barrier, zero_copy=True)
        e2e_rows = seg.total_rows * e2e_tiles
        step_ms, e2e_ms, kern_ms = allmax([step_ms, e2e_ms, kern_ms])
        if zc_ms is not None:
            zc_ms = allmax([zc_ms])[0]
        rows_all, sel_all, e2e_rows_all = allsum([table.total_rows, selected, e2e_rows])
        if rank == 0:
            used = sorted(set(w.proj) | set(filter_columns(w.filter)))
            out_per_row = sum(12 if s else l for s, l in zip(w.proj_is_string, w.proj_elem_len))
            b_in = referenced_bytes(seg, used) * tiles
            alg = b_in + selected * out_per_row + (table.total_rows + 7) // 8
            achieved = alg / (kern_ms * 1e-3) / 1e9
            line = {
                "metric": METRIC, "value": rows_all / (step_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "int64/bytes", "data": "synthetic",
                "config": cfg3_config(args, world, rpb, seg_rows, tiles, seg, sel_all / rows_all, {
                    "rows_per_gpu": table.total_rows, "micro_blocks_per_gpu": table.n_blocks,
                    "encoded_bytes_per_gpu": int(seg.sizes.sum()) * tiles, "parallelism": f"shard{world}",
                    "tiling": f"one seeded {seg.total_rows}-row segment per rank, generated on the host and copied {tiles}x into "
                              f"HBM (physically distinct tiles, one page batch of {table.n_blocks} micro-blocks)",
                    "l2_policy": "every tile (~2 GB) is larger than L2 (126 MB); no flush needed",
                    "gen_seconds": round(t_gen, 1), "host_numa_node": numa_node, "host_numa_nodes": numa_all}),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": measured_traffic("r2_traffic_cfg3.json", table.total_rows), "peak_source": peak_src,
                             "alg_bytes_per_launch": int(alg), "alg_bytes_in": int(b_in), "alg_bytes_out": int(selected * out_per_row),
                             "alg_rule": "SURVEY 8d with staged regions: per block header + column headers + regions of the referenced "
                                         "columns (3 filter + 6 projected) + selected x (4 x 8 B + 2 x 12 B) + bitmap",
                             "kernel_ms": kern_ms,
                             "kernel": "one scan = count + prefix + project kernels, CUDA events on the launching stream"},
                "e2e": {"value": e2e_rows_all / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "ms_per_step": e2e_ms, "steps": e2e_steps, "rows_per_step": int(e2e_rows_all), "page_batches": n_parts,
                        "streams": args.e2e_workers,
                        "timing": f"host wall clock around obgpu_pipeline_scan ({args.e2e_workers} streams); the pinned host "
                                  f"segment is scanned {tiles if not args.e2e_one_tile else 1}x per step, every pass a real H2D + D2H"},
                "gpu_launches": int(launches),
                "clocks": clocks,
                "gbs_decoded_equiv": rows_all * 16 * 8 / (step_ms * 1e-3) / 1e9,
            }
            line["e2e"]["mode"] = "staged: every byte of every micro-block is copied to HBM first"
            if zc_ms is not None:
                ref_in = referenced_bytes(seg, used) * e2e_tiles * world
                zc = {"value": e2e_rows_all / (zc_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(ref_in), "d2h_bytes_per_step": int(zc_d2h),
                      "ms_per_step": zc_ms, "steps": e2e_steps, "rows_per_step": int(e2e_rows_all), "page_batches": n_parts,
                      "streams": args.e2e_workers,
                      "mode": "zero copy (obgpu_host_scan_spec.zero_copy): the pinned host image is opened in place; the kernels read the "
                              "headers and the referenced columns' regions from host memory over PCIe inside the timed region, results "
                              "are copied back to pinned host vectors; h2d_bytes_per_step = the referenced bytes (roofline.alg_bytes_in "
                              "rule), not a copy the library makes"}
                # the headline e2e is the faster of the two ways the same public entry moves the same host-resident input
                if zc["value"] > line["e2e"]["value"]:
                    line["e2e_staged"] = line["e2e"]
                    line["e2e"] = zc
                else:
                    line["e2e_zero_copy"] = zc
            if world == 1 and not args.no_cpu_baseline:
                ncpu = host_cpus()
                sample_blocks = max(1, min(seg.n_blocks, args.cpu_sample_rows // rpb))
                passes = 6
                rates, crow, csel = cpu_reference_leg(w, passes, 1, ncpu, sample_blocks)
                mean_dt = float(np.mean([d for _, d in rates]))
                line["cpu_baseline"] = {
                    "value": crow / mean_dt, "unit": UNIT, "cores": ncpu, "kind": "port",
                    "sample": f"first {crow} rows ({sample_blocks} micro-blocks) of the segment, {passes} timed passes "
                              f"({sum(d for _, d in rates) * ncpu:.0f} CPU-seconds), oracle port of the reference scan "
                              f"(batch {BATCH_ROWS}), {ncpu} threads = cgroup cpu quota ({os.cpu_count()} logical CPUs visible)"}
        del w, pinned_buf, seg
    # ---- configs[1] (cfg2): 100 M rows x 8 INT64 per GPU, weak scaling ----------------------------------------------
    if args.workload == "cfg2" or not args.no_secondary:
        rows = args.cfg2_rows
        t_gen = time.perf_counter()
        w, pinned_buf = build_workload(rows, rank * rows, 2, pinned=True, n_threads=max(1, host_cpus() // max(world, 1)))
        t_gen = time.perf_counter() - t_gen
        table = w.table
        d_image = torch.empty(table.image.size + 64, dtype=torch.uint8, device=dev)
        d_image[:table.image.size].copy_(pinned_buf, non_blocking=True)
        d_image[table.image.size:].zero_()
        torch.cuda.synchronize()
        batch = ctx.open_batch(table, device_image_ptr=d_image.data_ptr())
        run = DeviceRun(ctx, stream, batch, w, int(table.total_rows * 0.30), world, dist)
        step_ms, kern_ms, selected, launches, clocks = run.run(args.steps, args.warmup, local, rank, dump=dumper("cfg2", w))
        batch.close()
        e2e_ms, n_e2e, h2d, d2h, n_parts, e2e_steps, e2e_launches = e2e_run(local, table, w, 1400, 0.30, args, 1, barrier)
        assert n_e2e == selected
        step_ms, e2e_ms, kern_ms = allmax([step_ms, e2e_ms, kern_ms])
        rows_all, sel_all = allsum([table.total_rows, selected])
        if rank == 0:
            alg = w.alg_bytes(selected)
            achieved = alg / (kern_ms * 1e-3) / 1e9
            c2 = {
                "metric": METRIC, "value": rows_all / (step_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                "config": {"workload": w.name, "rows_per_gpu": table.total_rows, "columns": 8,
                           "micro_blocks_per_gpu": table.n_blocks, "encoded_bytes_per_gpu": int(table.sizes.sum()),
                           "selectivity": selected / table.total_rows, "parallelism": f"shard{world}",
                           "l2_policy": "input image (1.2 GB) larger than L2 (126 MB); no flush needed",
                           "gen_seconds": round(t_gen, 1), "host_numa_node": numa_node, "host_numa_nodes": numa_all},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": measured_traffic("r1_traffic.json", table.total_rows), "peak_source": peak_src,
                             "alg_bytes_per_launch": alg, "kernel_ms": kern_ms,
                             "alg_rule": "whole blocks are staged: full block bytes + selected x 64 B + bitmap"},
                "e2e": {"value": rows_all / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "ms_per_step": e2e_ms, "steps": e2e_steps, "page_batches": n_parts, "streams": args.e2e_workers,
                        "timing": f"host wall clock around obgpu_pipeline_scan ({args.e2e_workers} streams)"},
                "gpu_launches": int(launches), "clocks": clocks,
                "gbs_decoded_equiv": rows_all * 8 * 8 / (step_ms * 1e-3) / 1e9,
            }
            if world == 1 and not args.no_cpu_baseline and (args.workload == "cfg2"):
                ncpu = host_cpus()
                sample_blocks = min(table.n_blocks, max(64, int(args.cpu_sample_rows // 1400)))
                rates, crow, csel = cpu_reference_leg(w, 4, 1, ncpu, sample_blocks)
                mean_dt = float(np.mean([d for _, d in rates]))
                c2["cpu_baseline"] = {"value": crow / mean_dt, "unit": UNIT, "cores": ncpu, "kind": "port",
                                      "sample": f"first {crow} rows ({sample_blocks} micro-blocks) of the same table, 4 timed passes, "
                                                f"oracle port of the reference scan (batch {BATCH_ROWS}), {ncpu} threads"}
            if line is None:
                line = c2
            else:
                line["secondary"] = {"cfg2": c2}
    if rank == 0:
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg2", "compaction"])
    ap.add_argument("--compaction-window", type=int, default=4_000_000, help="compaction: rowkey indexes covered by one of the 8 runs")
    ap.add_argument("--verify", action="store_true", help="compaction: compare the merged stream with the oracle (small sizes)")
    ap.add_argument("--stream-ranges", type=int, default=0, help="compaction: N > 0 merges host-resident runs range by range (runs larger than HBM)")
    ap.add_argument("--rows", type=int, default=1_000_000_000, help="cfg3: rows of the whole table (split over the GPUs)")
    ap.add_argument("--segment-rows", type=int, default=15_625_000, help="cfg3: rows of the generated segment (upper bound)")
    ap.add_argument("--rows-per-block", type=int, default=0, help="cfg3: 0 = cut micro-blocks at the 16 KiB target")
    ap.add_argument("--cfg2-rows", type=int, default=100_000_000, help="cfg2: rows per GPU (BASELINE configs[1]: 100 M)")
    ap.add_argument("--ref-rows", type=int, default=16_000_000, help="rows per step of the reference arm's sample")
    ap.add_argument("--cpu-sample-rows", type=int, default=16_000_000,
                    help="rows of the workload the cpu_baseline leg scans per pass")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-mode", default="both", choices=["both", "staged"], help="cfg3 e2e: also measure the zero-copy mode of the host entry")
    ap.add_argument("--e2e-one-tile", action="store_true", help="cfg3 e2e: one pass over the host segment per step instead of `tiles`")
    ap.add_argument("--e2e-batches", type=int, default=12, help="page batches per e2e pass (pipeline depth)")
    ap.add_argument("--e2e-ramp", type=int, default=2, help="the first N page batches are 1/2^N .. 1/2 of a full one")
    ap.add_argument("--e2e-workers", type=int, default=3, help="host worker threads = CUDA streams of the e2e pipeline")
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the cfg2 measurement")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed scan's results (rank 0's shard) to DIR/<workload>_<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "compaction"):
        ap.error("--dump-outputs applies to the scan workloads of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.workload == "compaction":
        # BASELINE.json configs[4] (stand-in size): K-way major-compaction merge, range-partitioned over the GPUs
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_compaction
        return bench_compaction.run(argparse.Namespace(runs=8, window=args.compaction_window, steps=args.steps, warmup=args.warmup,
                                                      verify=args.verify, python_exchange=False, stream_ranges=args.stream_ranges))
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
