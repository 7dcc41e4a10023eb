#!/usr/bin/env python
"""bench.py -- rows scanned/sec for Pinot's filter -> project -> GROUP BY aggregate path on B200 (BASELINE.json metric:
"rows scanned/sec per box, filter+groupby on 100M-row segments, 1/2/4/8 GPU").

Table (per GPU): 8 segments x 100 M rows, 8 dict-encoded fixed-bit INT columns c0..c7 (cardinalities 10 .. 1 000 000 ->
4,7,10,14,16,17,20,20 bits), synthetic, resident in HBM in Pinot's index formats.

  headline (the metric: filter + GROUP BY, BASELINE configs[2]/[3] shape on the configs[1] table)
      SELECT SUM(c5), COUNT(*) FROM benchTable WHERE c6 > K GROUP BY c3          -- 10 % of the rows, 10 000 groups
  a "step" = ONE pass of that query over all of the rank's segments through the reference-facing plugin call
  (B200PlanMaker.execute_segments -> pb200h_execute -> one persistent scan kernel), delivered as the server-level results
  block: the rank's segments are combined on the device (GroupByCombineOperator's job), with N > 1 GPUs the per-GPU group
  tables are reduced ONCE to rank 0 (NCCL over NVLink), rank 0 extracts the groups.

  c2 (BASELINE configs[1], the aggregation-only scan of round 1, reported beside the headline)
      SELECT SUM(c5), COUNT(*) FROM benchTable WHERE c3 BETWEEN lo AND hi AND c6 > K    -- 2-predicate range filter, 25 %

    value        rows/s with the segments resident in HBM (Pinot loads a segment once, then serves queries from it)
    roofline     algorithmic bytes of the scan kernel (sum of bitsPerElement/8 of the touched columns x rows: both queries
                 touch c3, c5, c6 = 51 bits/row) / its CUDA-event duration, against MEASURED_PEAKS.json's HBM bandwidth
    e2e          the headline through the same call with HOST-resident index buffers: every step uploads the touched
                 columns from pinned host memory (H2D inside the timed region), scans, reads the result block back
    cpu_baseline the CPU oracle (C++ restatement of the Java operator chain, kind "port") on the SAME full-size table,
                 generated independently on the CPU; its per-segment group tables are compared with the device's
    --impl reference   the CPU restatement alone (no device library loaded), all host threads; there is no JVM in the
                 image (SURVEY.md section 0), so the reference's own Java path cannot run here

Multi-GPU (torchrun, one rank per GPU): segments shard whole per GPU, no data-path collective; weak scaling:
value = total rows of all ranks / max-over-ranks time.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time


ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CARDS = [10, 100, 1_000, 10_000, 65_536, 100_000, 1_000_000, 1_000_000]  # c0..c7 -> 4,7,10,14,16,17,20,20 bits
VALUE_STEP = [1, 1, 1, 3, 1, 7, 2, 2]
VALUE_BASE = [0, 0, 0, 5, 0, 11, 1, 1]
TOUCHED = ["c3", "c5", "c6"]   # both queries
METRIC = "rows scanned/sec per box, filter+groupby on 100M-row segments, 1/2/4/8 GPU"


def bits_of(card: int) -> int:
    return 1 if card <= 2 else int(card - 1).bit_length()


def column_specs(rank: int, seg: int, names=None):
    return [{"name": f"c{c}", "cardinality": CARDS[c], "value_base": VALUE_BASE[c], "value_step": VALUE_STEP[c],
             "seed": 1000 + 104729 * rank + 131 * seg + c} for c in range(8) if names is None or f"c{c}" in names]


def groupby_query_text(selectivity: float) -> str:
    k_id = int(round(CARDS[6] * (1 - selectivity))) - 1   # c6 > value(k_id): the upper `selectivity` of the dictionary
    return (f"SELECT SUM(c5), COUNT(*) FROM benchTable WHERE c6 > {VALUE_BASE[6] + VALUE_STEP[6] * k_id} "
            f"GROUP BY c3 LIMIT 100000")


def c2_query_text(selectivity: float) -> str:
    # each predicate keeps sqrt(selectivity) of the dictionary (uniform dictIds): c3 a centred range, c6 the upper tail
    f = selectivity ** 0.5
    n3 = CARDS[3]
    lo_id = int(n3 * (1 - f) / 2)
    hi_id = lo_id + int(round(n3 * f)) - 1
    k_id = int(round(CARDS[6] * (1 - f))) - 1
    lo, hi = VALUE_BASE[3] + VALUE_STEP[3] * lo_id, VALUE_BASE[3] + VALUE_STEP[3] * hi_id
    k = VALUE_BASE[6] + VALUE_STEP[6] * k_id
    return f"SELECT SUM(c5), COUNT(*) FROM benchTable WHERE c3 BETWEEN {lo} AND {hi} AND c6 > {k}"


def bytes_per_row() -> float:
    return sum(bits_of(CARDS[int(c[1:])]) for c in TOUCHED) / 8.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []  # (t, sm, max, power, reasons[4])
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            p = [x.strip() for x in line.split(",")]
            try:
                self.samples.append((time.time(), float(p[1]), float(p[2]), float(p[3]), p[4:8]))
            except (ValueError, IndexError):
                pass

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-5:]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in inside for n, v in zip(names, s[4]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(s[1] for s in inside), "sm_max_mhz": max(s[2] for s in inside),
                "power_w_max": max(s[3] for s in inside), "samples": len(inside), "reasons": reasons}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ------------------------------------------------------------------------------------------------ CPU arm (oracle only)
class CpuTable:
    """The benchmark table's touched columns, generated on the CPU by the oracle's twin of the device generator
    (byte-identical: tests/test_gpu_synth.py), split into row ranges so that the single-threaded operator chain of the
    oracle runs on every host core.  Nothing here touches libpinot_b200.so."""

    def __init__(self, segments: int, rows: int, rank: int = 0, threads: int = 0):
        from oracle.pinot_oracle import oracle as get_oracle
        self.o = get_oracle()
        self.threads = threads or (os.cpu_count() or 1)
        t0 = time.perf_counter()
        self.segments = [self.o.synth_segment(f"r{rank}s{s}", rows, column_specs(rank, s, TOUCHED), self.threads)
                         for s in range(segments)]
        self.generation_s = time.perf_counter() - t0
        parts = max(1, (self.threads + segments - 1) // segments)
        self.work = [(s, part) for s, seg in enumerate(self.segments) for part in self.o.row_ranges(seg, parts)]
        self.rows = segments * rows

    def run(self, q):
        """One pass of `q` over the whole table.  Returns (seconds, [per-segment {dictId key: [sum, count]}])."""
        import numpy as np
        results = [None] * len(self.work)
        nxt = [0]
        lock = threading.Lock()

        def worker():
            while True:
                with lock:
                    i = nxt[0]
                    nxt[0] += 1
                if i >= len(self.work):
                    return
                results[i] = self.o.execute(self.work[i][1], q)   # ctypes releases the GIL

        ts = [threading.Thread(target=worker) for _ in range(min(self.threads, len(self.work)))]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        sec = time.perf_counter() - t0
        # merge the row ranges of a segment (same dictionaries: by dictId) -- outside the timed region, as the
        # reference's combine is outside its per-segment operators
        tables = [dict() for _ in self.segments]
        for (s, _), r in zip(self.work, results):
            t = tables[s]
            if r.num_groups < 0:
                cur = t.setdefault((), [0.0, 0])
                cur[0] += float(r.doubles[0][0]); cur[1] += int(r.longs[1][0])
                continue
            keys = r.keys[:, 0].astype(np.int64)
            for k, sm, c in zip(keys.tolist(), r.doubles[0].tolist(), r.longs[1].tolist()):
                cur = t.get(k)
                if cur is None:
                    t[k] = [sm, c]
                else:
                    cur[0] += sm; cur[1] += c
        return sec, tables


def block_table(block):
    """{dictId key: [sum, count]} of a device results block of the bench queries (SUM, COUNT)."""
    if block.num_groups < 0:
        return {(): [float(block.doubles[0][0]), int(block.longs[1][0])]}
    return {int(k): [float(s), int(c)] for k, s, c in
            zip(block.keys[:, 0].tolist(), block.doubles[0].tolist(), block.longs[1].tolist())}


def dump_outputs(block, q, out_dir):
    """Writes the headline results block as float64 .npy files: the group keys (dictIds of the GROUP BY column) and one
    array per aggregation, rows ordered by key so that two builds can be compared array for array whatever order their
    extraction emits the groups in."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    order = np.lexsort(block.keys.T[::-1])
    arrays = {"group_keys": block.keys[order]}
    for a, agg in enumerate(q.aggregations):
        col = block.longs[a] if agg.function == "COUNT" else block.doubles[a]
        arrays[f"agg{a}_{agg.function.lower()}" + (f"_{agg.column}" if agg.column else "")] = np.asarray(col)[order]
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(arr, dtype=np.float64))


def assert_same_table(got, want, what):
    assert set(got) == set(want), f"{what}: group keys differ ({len(got)} vs {len(want)})"
    for k, (ws, wc) in want.items():
        gs, gc = got[k]
        assert gc == wc, (what, k, "count", gc, wc)
        assert gs == ws or abs(gs - ws) <= 1e-6 * abs(ws), (what, k, "sum", gs, ws)   # north_star: SUM within 1e-6 relative


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--segments", type=int, default=8)
    ap.add_argument("--rows", type=int, default=100_000_000, help="rows per segment")
    ap.add_argument("--selectivity", type=float, default=0.10, help="headline filter selectivity")
    ap.add_argument("--c2-selectivity", type=float, default=0.25)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-threads", type=int, default=0, help="0 = all host cores")
    ap.add_argument("--reference-seconds", type=float, default=120.0, help="time budget of the --impl reference steps")
    ap.add_argument("--quick", action="store_true", help="tuning runs: skip the c2, e2e and cpu_baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline's results block of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference" and rank != 0:
        return 0  # the CPU arm runs on rank 0 only

    from pinot_b200 import sql   # pure Python (the SQL front end of the tests); loads no native code

    q_gb = sql.parse(groupby_query_text(args.selectivity))
    q_c2 = sql.parse(c2_query_text(args.c2_selectivity))
    bpr = bytes_per_row()
    config = {"workload": f"filter+GROUP BY on the C2 table: {args.segments} segments x {args.rows} rows per GPU, 8 dict-encoded "
                          f"fixed-bit INT columns (bits 4,7,10,14,16,17,20,20); {groupby_query_text(args.selectivity)} "
                          f"(10 000 groups); per-GPU device-side combine, N>1: one reduce of the group tables to rank 0",
              "segments_per_gpu": args.segments, "rows_per_segment": args.rows, "selectivity": args.selectivity,
              "groups": CARDS[3], "touched_bits_per_row": int(bpr * 8),
              "l2_policy": f"inputs larger than L2 (touched columns = {args.segments * args.rows * bpr / 1e9:.2f} GB per step "
                           "per GPU vs 126 MB L2)",
              "parallelism": f"segments sharded {args.segments}/GPU x {world} GPU, group tables reduced once"}

    # ---------------------------------------------------------------------------------------------- reference arm
    if args.impl == "reference":
        cores = args.cpu_threads or (os.cpu_count() or 1)
        table = CpuTable(args.segments, args.rows, 0, cores)
        table.run(q_gb)  # warm-up / page-in
        times = []
        t_start = time.perf_counter()
        while len(times) < max(1, args.steps) and (not times or time.perf_counter() - t_start < args.reference_seconds):
            times.append(table.run(q_gb)[0])
        sec = statistics.mean(times)
        val = table.rows / sec
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "rows/s", "n_gpus": args.gpus,
                "steps": len(times), "warmup": 1, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "rows/s", "cores": cores, "kind": "port", "cpu": cpu_model(),
                                 "nproc": os.cpu_count(),
                                 "sample": f"the whole table every step: {args.segments} segments x {args.rows} rows generated on the "
                                           f"CPU, each segment split into {len(table.work) // args.segments} row ranges "
                                           f"({len(table.work)} work items on {cores} threads); C++ restatement of the Java "
                                           f"operator chain (oracle/), no JVM in the image; generation {table.generation_s:.1f} s"},
                "e2e": {"value": val, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------------------------------------- B200 arm
    import torch
    from pinot_b200.plan_maker import B200Context, B200PlanMaker, IndexSegment

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        from pinot_b200.distributed import execute_and_combine

    ctx = B200Context(local_rank)
    pm = B200PlanMaker(ctx)
    t_gen = time.perf_counter()
    segs = [IndexSegment.synthetic(ctx, f"r{rank}s{s}", args.rows, column_specs(rank, s)) for s in range(args.segments)]
    gen_s = time.perf_counter() - t_gen
    rows_per_step = args.segments * args.rows
    domain = None
    combine_kind = "none (one GPU)"
    if dist is not None:
        # the per-GPU group tables are merged BY VALUE: all ranks' segments share table-wide dictionaries for the group key
        # and the summed column (synthetic dictionaries are identical, so binding re-encodes nothing)
        from pinot_b200.distributed import DeviceBackend, global_domain, init_comm
        combine_backend = DeviceBackend(pm, views=True)
        domain = global_domain(ctx, segs, ["c3", "c5"], dist)
        combine_kind = "torch.distributed reduce of the aliased device tables"
        if os.environ.get("PB200_TORCH_REDUCE", "0") != "1":
            # the reduce of the group tables runs inside libpinot_b200.so (pb200_result_combine); every rank must take the
            # same route, so the outcome of the attempt is agreed on first
            try:
                init_comm(ctx, dist)
                ok = 1
            except Exception as e:  # NCCL not loadable by the library: the torch-driven reduce is the same protocol
                sys.stderr.write(f"in-library combine unavailable ({e}); using torch.distributed\n")
                ok = 0
            flag = torch.tensor([ok], dtype=torch.int32, device=f"cuda:{local_rank}")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 1:
                combine_kind = "in-library NCCL group (pb200_result_combine)"
            else:
                ctx.comm_world = 0

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def gb_step():
        """The headline step: the whole table's results block on rank 0."""
        # views=True: the block's columns alias the pinned host block the device extracted the groups into (what a JVM
        # wraps with NewDirectByteBuffer) instead of being copied once more into numpy arrays
        if dist is not None:
            block = execute_and_combine(combine_backend, segs, q_gb, dist, dst=0, merged_docs_bound=rows_per_step * world)
            return block, (block.device_ms if block is not None else pm.last_device_ms)
        block = pm.execute_segments(segs, q_gb, merge=True, views=True)[0]
        return block, block.device_ms

    def c2_step():
        blocks = pm.execute_segments(segs, q_c2)
        return (sum(float(b.doubles[0][0]) for b in blocks), sum(int(b.longs[1][0]) for b in blocks)), blocks[0].device_ms

    def timed(step, steps):
        # the warm-up keeps the same results alive as the timed loop does (`first`, the previous step's `out` and the
        # step in flight), so that the library's device and pinned result pools reach their final size here: otherwise
        # the second timed step allocates them (cudaMalloc / cudaHostAlloc, up to ~100 ms) inside the timed region
        first = step()
        for _ in range(args.warmup - 1):
            out = step()
        barrier()
        w0 = time.time()
        t0 = time.perf_counter()
        kms = []
        for _ in range(steps):
            out, dms = step()
            kms.append(dms)
        barrier()
        elapsed = time.perf_counter() - t0
        w1 = time.time()
        if dist is not None:
            t = torch.tensor([elapsed], dtype=torch.float64, device=f"cuda:{local_rank}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            elapsed = float(t.item())
        return out, first[0], elapsed, statistics.mean(kms), (w0, w1)

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    gb_out, gb_first, gb_elapsed, gb_kms, (w0, w1) = timed(gb_step, args.steps)
    clocks = sampler.stop(w0, w1)
    peak, peak_src = measured_peak_gbs()
    gb_ms = gb_elapsed / args.steps * 1e3
    value = rows_per_step * world / (gb_elapsed / args.steps)
    gb_achieved = rows_per_step * bpr / (gb_kms * 1e-3) / 1e9
    gb_table = None
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(gb_out, q_gb, args.dump_outputs)
        gb_table = block_table(gb_out)
        assert gb_table == block_table(gb_first), "non-deterministic result across steps"
        matched = sum(c for _, c in gb_table.values())
    gb_out = gb_first = None   # blocks alias native results: dropped before the context closes
    if rank == 0:
        expect = rows_per_step * world * args.selectivity
        assert abs(matched - expect) < 0.02 * expect + 10, (matched, expect)

    if args.quick:
        if rank == 0:
            print(json.dumps({"quick": True, "value": value, "ms_per_step": gb_ms, "kernel_ms": gb_kms,
                              "achieved_gbs": gb_achieved, "frac": gb_achieved / peak, "clocks": clocks,
                              "env": {k: v for k, v in os.environ.items() if k.startswith("PB200_")},
                              "selectivity": args.selectivity, "groups": len(gb_table)}))
        for sgm in segs:
            sgm.destroy()
        ctx.close()
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---- the same query delivered as PER-SEGMENT results blocks (what the per-segment Operator.nextBlock() seam returns) ----
    def gb_blocks_step():
        blocks = pm.execute_segments(segs, q_gb)
        return blocks, blocks[0].device_ms
    seg_blocks, _, sb_elapsed, sb_kms, _ = timed(gb_blocks_step, max(20, args.steps // 10))
    sb_steps = max(20, args.steps // 10)

    # ---- c2: the aggregation-only scan ----
    c2_steps = max(20, args.steps // 3)
    c2_out, c2_first, c2_elapsed, c2_kms, _ = timed(c2_step, c2_steps)
    assert c2_out == c2_first, "non-deterministic c2 result"
    c2_achieved = rows_per_step * bpr / (c2_kms * 1e-3) / 1e9

    # ---- e2e: host-resident index buffers, H2D inside the timed region (rank-local; N>1: max over ranks) ----
    pinned = []
    h2d = 0
    for sgm in segs:
        cols = []
        for cname in TOUCHED:
            info = sgm.column_info(cname)
            fwd = sgm.read_index(cname, "fwd")
            pt = torch.empty(len(fwd), dtype=torch.uint8).pin_memory()
            pt.numpy()[:] = fwd
            dct = sgm.read_index(cname, "dict")
            cols.append((cname, info, pt, dct))
            h2d += len(fwd) + len(dct)
        pinned.append(cols)

    class _Col:  # duck type of IndexSegment.from_columns' column description
        def __init__(self, name, info, fwd, dct):
            self.name, self.data_type, self.has_dictionary = name, 0, True
            self.bits, self.cardinality, self.is_sorted, self.dict_entry_bytes = info["bits"], info["cardinality"], False, 4
            self.fwd, self.dict, self.inv = fwd, dct, None

    d2h = [0]

    def e2e_step():
        loaded = [IndexSegment.from_columns(ctx, f"e2e{i}", args.rows, [_Col(n, inf, pt.numpy(), d) for n, inf, pt, d in cols])
                  for i, cols in enumerate(pinned)]
        block = pm.execute_segments(loaded, q_gb, merge=True)[0]
        d2h[0] = block.keys.nbytes + sum(a.nbytes for a in block.doubles) + sum(a.nbytes for a in block.longs)
        for l in loaded:
            l.destroy()
        return block

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        eb = e2e_step()
    barrier()
    e2e_elapsed = time.perf_counter() - t0
    if world == 1:
        assert block_table(eb) == gb_table, "e2e result differs from the resident result"
    if dist is not None:
        t = torch.tensor([e2e_elapsed], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_elapsed = float(t.item())
    e2e_value = rows_per_step * world / (e2e_elapsed / args.e2e_steps)
    del pinned

    # ---- cpu_baseline + FULL-SIZE parity: the oracle on the same table, generated independently on the CPU ----
    cpu = None
    if rank == 0 and world == 1:
        cores = args.cpu_threads or (os.cpu_count() or 1)
        table = CpuTable(args.segments, args.rows, 0, cores)
        table.run(q_gb)  # page-in
        sec, cpu_tables = table.run(q_gb)
        for s, (blk, want) in enumerate(zip(seg_blocks, cpu_tables)):
            assert_same_table(block_table(blk), want, f"segment {s}: device vs CPU oracle, {args.rows} rows")
        merged = {}
        for t in cpu_tables:
            for k, (sm, c) in t.items():
                cur = merged.setdefault(k, [0.0, 0])
                cur[0] += sm; cur[1] += c
        assert_same_table(gb_table, merged, "device-side combine vs merged CPU oracle tables")
        _, c2_tables = table.run(q_c2)
        want_c2 = (sum(t[()][0] for t in c2_tables), sum(t[()][1] for t in c2_tables))
        assert c2_out[1] == want_c2[1] and abs(c2_out[0] - want_c2[0]) <= 1e-6 * abs(want_c2[0]), ("c2 vs CPU oracle", c2_out, want_c2)
        cpu = {"value": table.rows / sec, "unit": "rows/s", "cores": cores, "kind": "port", "cpu": cpu_model(),
               "sample": f"the whole table, one pass: {args.segments} segments x {args.rows} rows generated on the CPU (same bytes as "
                         f"the device generator), {len(table.work)} row-range work items on {cores} threads; C++ restatement of the "
                         "Java operator chain (oracle/); no JVM in the image",
               "parity": f"per-segment and combined group tables of the device == the oracle's on all {table.rows} rows "
                         "(COUNT exact, SUM within 1e-6 relative); c2 result == oracle"}

    # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the scan kernel, from the committed `ncu --set full`
    # captures of these same workloads (profiles/): only quoted when this run IS that workload
    def traffic_of(name, sel):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            if tj.get("segments") == args.segments and tj.get("rows_per_segment") == args.rows and abs(tj.get("selectivity", -1) - sel) < 1e-9:
                return tj["dram_bytes_per_launch"], tj["source"]
        return None, None
    gb_traffic, gb_traffic_src = traffic_of("r2_gb_traffic.json", args.selectivity)
    c2_traffic, c2_traffic_src = traffic_of("r2_c2_traffic.json", args.c2_selectivity)

    if rank == 0:
        alg = rows_per_step * bpr
        line = {"metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": gb_ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int64", "data": "synthetic", "config": config,
                "roofline": {"bound": "hbm", "achieved": gb_achieved, "peak": peak, "unit": "GB/s",
                             "frac": gb_achieved / peak, "traffic": gb_traffic, "traffic_source": gb_traffic_src,
                             "peak_source": peak_src,
                             "kernel": "pb200::scan_kernel<6,true> (group-by, W=6 warps, 2 CTAs/SM)", "kernel_ms": gb_kms,
                             "algorithmic_bytes_per_launch": alg},
                "cpu_baseline": cpu,
                "e2e": {"value": e2e_value, "unit": "rows/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h[0],
                        "steps": args.e2e_steps,
                        "note": "every step re-uploads the touched columns from pinned host memory (PCIe bound) and reads the "
                                "results block back; `value` is the same plugin call with the segments resident in HBM"},
                "gpu_launches": args.steps * (5 if getattr(gb_out, "count_carrier", False) else 4),
                "gpu_launches_note": "per step: 1 scan_kernel (+ 1 carrier_verify_kernel when the counts ride in the sum) + 3 extraction "
                                     "kernels (count, scan, write); memsets and NCCL not counted",
                "count_carrier": bool(getattr(gb_out, "count_carrier", False)),
                "per_segment_blocks": {"ms_per_step": sb_elapsed / sb_steps * 1e3, "kernel_ms": sb_kms, "steps": sb_steps,
                                       "value": rows_per_step * world / (sb_elapsed / sb_steps),
                                       "note": "same query, one results block per segment (8 x 10 000 groups extracted) "
                                               "instead of the device-side combine"},
                "c2": {"query": c2_query_text(args.c2_selectivity), "value": rows_per_step * world / (c2_elapsed / c2_steps),
                       "ms_per_step": c2_elapsed / c2_steps * 1e3, "steps": c2_steps,
                       "roofline": {"bound": "hbm", "achieved": c2_achieved, "peak": peak, "unit": "GB/s",
                                    "frac": c2_achieved / peak, "traffic": c2_traffic, "traffic_source": c2_traffic_src,
                                    "kernel": "pb200::scan_kernel<6,false> (aggregation only)", "kernel_ms": c2_kms,
                                    "algorithmic_bytes_per_launch": alg},
                       "result": {"sum_c5": c2_out[0], "count": c2_out[1], "scope": "rank 0's segments"}},
                "clocks": clocks, "segment_generation_s": gen_s, "cross_gpu_combine": combine_kind,
                "result": {"groups": len(gb_table), "matched": sum(c for _, c in gb_table.values()),
                           "sum_c5": sum(s for s, _ in gb_table.values()), "scope": "all ranks (reduced to rank 0)"}}
        print(json.dumps(line))
    for sgm in segs:
        sgm.destroy()
    if domain is not None:
        domain.release()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
