#!/usr/bin/env python
"""bench.py — BASELINE.json metric: rows/sec (and HBM GB/s) of the TPC-H Q6 Filter
(shipdate range AND discount range AND quantity) over synthetic lineitem rows.

  python bench.py --gpus N --steps K --warmup W          (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                   (CPU arm on the host cores, see below)

A "step" is one pass of the hot path (Filter::Evaluate -> one fused predicate + ordered
compaction kernel) over one batch of `--rows` lineitem rows per GPU (default 1e9 = configs[1]
of BASELINE.json; at N>1 each rank owns a contiguous row range: weak scaling, configs[4]
shape; `--rows 1250000000` is configs[4]'s stated 10 B rows at N=8), inputs resident in HBM.
Inputs (20 GB) are far larger than L2 (126 MB), so every step streams from HBM; no flush needed.

`value`    = rows/s over all ranks, device-resident (CUDA events, max over ranks).
`e2e`      = same metric through the C-ABI with HOST buffers (gdv_filter_evaluate(GDV_MEM_HOST)):
             H2D of every input column and D2H of the selection vector inside the timed region.
             `e2e.value` is measured on PINNED host buffers; `e2e.pageable` repeats it on plain
             malloc'd (pageable) buffers, the memory an Arrow MemoryPool hands out.
`roofline` = algorithmic bytes (20 B/row in + 4 B per selected row out, SURVEY.md §8d) over the
             kernel's CUDA-event time, against MEASURED_PEAKS.json hbm_gbs.
`configs`  = (N=1 only) the other single-GPU workloads of BASELINE.json, each with rows/s, kernel
             ms, roofline fraction, a full-size check against an independent evaluation and the
             CPU arm's number:  q6_nulls (configs[1] with 1 % nulls per column), q1 (configs[2]:
             eight-output projector, 2 % nulls, ~1e9 rows in chunks), str (configs[3]: string
             filter, 1e8 rows in 2 RecordBatches), ab_1m (configs[0]: a+b over a 1M-row batch).
`cpu_baseline` = the CPU arm on this box's host cores.  Gandiva's LLVM JIT cannot be built in this
             image (no source under /root/reference, no LLVM), so the arm is
             kind "fused-cxx-proxy": oracle/cpu_proxy.cc, the row loop a JIT would emit, hand-fused,
             g++ -O3 -march=native (AVX-512 where present), one pinned thread per hardware thread —
             plus `arrow_compute`: the same predicate through pyarrow.compute (not Gandiva either).
`--impl reference` prints that CPU arm as its own line (same workload, same rows per step).

`--dump-outputs DIR` writes the SelectionVector of the last timed step to DIR as float64 .npy files
(see dump_outputs), so that two builds run with the same arguments can be compared output for output.
The bench writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ALGO_IN_BYTES_PER_ROW = 20.0   # date32 + 2 x float64, no validity buffers in the base run
IDX_BYTES = 4.0                # uint32 selection vector entries
Q1_IN_BYTES = 8 + 3 * 16 + 3 * 8 + 4 + 8 / 8.0      # 8 columns + 8 validity bits
Q1_OUT_BYTES = 2 * 16 + 6 * 8 + 8 / 8.0             # 8 outputs + 8 validity bits
METRIC = "rows/sec (TPC-H Q6 filter over synthetic lineitem)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=int(os.environ.get("GDV_BENCH_ROWS", 0)),
                    help="lineitem rows per GPU per step (default: 1e9 at N=1 = BASELINE.json configs[1]; 1.25e9 at N>1 = "
                         "configs[4]'s 10 B rows over 8 GPUs, the same per-GPU shard at every N>1)")
    ap.add_argument("--e2e-rows", type=int, default=0, help="rows per e2e step (0 = same as --rows)")
    ap.add_argument("--e2e-chunk", type=int, default=32 * 1024 * 1024, help="rows per host RecordBatch")
    ap.add_argument("--cpu-rows", type=int, default=0, help="CPU arm rows per step (0 = same as --rows)")
    ap.add_argument("--rows-per-thread", type=int, default=0)
    ap.add_argument("--block-threads", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` object (N=1)")
    ap.add_argument("--only", default="", help="comma list of configs entries to run (q6_nulls,q1,str,ab_1m)")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--equal-shards", action="store_true",
                    help="N>1, --gather push: keep equal row ranges (default: rank 0's shard is smaller by what absorbing the "
                         "other ranks' runs costs it)")
    ap.add_argument("--gather", default="push", choices=["push", "nccl"],
                    help="N>1: how the SelectionVector reaches rank 0.  push (default): "
                         "gdv_selection_push, device-side NVLink stores into rank 0's vector, no host "
                         "sync; nccl: all-gather of counts + send/recv (host reads the count)")
    ap.add_argument("--no-overlap", action="store_true", help="--gather nccl: gather inside each step, no pipelining")
    ap.add_argument("--no-numa-bind", action="store_true",
                    help="leave the process unbound (default: run on the CPUs of the GPU's NUMA node, restored for the CPU arms)")
    ap.add_argument("--waves", type=int, default=1,
                    help="N>1, --gather push: filter each step's batch in this many row slices (wave-major global row "
                         "order) so that the NVLink push of slice j hides under the filter kernel of slice j+1 and only "
                         "the last slice's push is exposed.  Default 1 (one run per rank: the push of batch i hides under the filter of "
                         "batch i+1, only the LAST batch's push is exposed).  Measured at N=2, 1.25e9 rows/GPU: 4 waves cost "
                         "+0.23 ms per step (four kernel ramps instead of one) and take the last step from +0.28 ms to +0.09 ms "
                         "— worth it for one isolated batch, not for a stream of batches (profiles/r02_multi_gpu.md)")
    ap.add_argument("--push-ctas", type=int, default=8, help="--gather push: CTAs (256 threads) of the push kernel")
    ap.add_argument("--sm-reserve", type=int, default=-1,
                    help="SMs the filter leaves free for the push / NCCL kernels (default with N>1: 2, i.e. twelve "
                         "256-thread CTA slots for the eight push CTAs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the SelectionVector of the last timed step to DIR (float64 .npy, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def q6_filter(gandiva, cases, cfg):
    b = gandiva.TreeExprBuilder()
    return gandiva.make_filter(cases.Q6_SCHEMA, b.make_condition(cases.q6_condition(b)), cfg), b


# =================================================================================================
# CPU arm (no product code: oracle/cpu_proxy.cc + pyarrow.compute; tree via oracle/tree.py)
# =================================================================================================
def _median(xs):
    s = sorted(xs)
    return s[len(s) // 2]


def cpu_rows_that_fit(want: int, bytes_per_row: float) -> int:
    import psutil
    avail = psutil.virtual_memory().available
    fit = int(avail * 0.45 / bytes_per_row)
    return max(min(want, fit) // (1 << 20) * (1 << 20), 1 << 20)


def cpu_q6(rows: int, steps: int, warmup: int, nullp: int = 0, arrow: bool = True) -> dict:
    """Q6 filter on the host cores: fused-cxx-proxy (all threads, pinned) and pyarrow.compute."""
    import numpy as np
    from oracle import cpu_proxy as px
    T = px.threads()
    rows = cpu_rows_that_fit(rows, 28.0)
    cols, vl = [], []
    for kind in (0, 1, 2):
        v, m = px.generate(kind, 42, 0, rows, nullp)
        cols.append(v)
        vl.append(m)
    out = px.Buf(rows, np.uint32)
    bits = px.Buf((rows + 63) // 64 + 1, np.uint64)
    px.lib().proxy_generate(9, 1, 0, rows, out.ptr, None, 0, 0)      # first touch of the output
    times, count = [], 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        count = px.q6_filter(cols[0], cols[1], cols[2], vl[0], vl[1], vl[2], rows, out, bits)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    med = _median(times)      # the box's other tenants make single steps noisy: the median step is reported
    res = {"value": rows / med, "unit": "rows/s", "cores": T, "kind": "fused-cxx-proxy",
           "rows_per_step": rows, "steps": len(times), "ms_per_step": med * 1e3, "statistic": "median step",
           "ms_per_step_min": min(times) * 1e3, "ms_per_step_max": max(times) * 1e3,
           "host_gbs": rows * (20.0 + (3 / 8.0 if nullp else 0)) / med / 1e9,
           "selected": int(count), "simd": px.simd(),
           "sample": "%d rows/step x %d steps of the same synthetic lineitem, oracle/cpu_proxy.cc (hand-fused Q6 row loop + "
                     "bitmap->index pass, g++ -O3 -march=native, %s) on %d pinned threads; NOT Gandiva's LLVM JIT "
                     "(unbuildable here)" % (rows, len(times), px.simd(), T)}
    if arrow:
        try:
            res["arrow_compute"] = cpu_q6_arrow(cols, vl, rows, T)
        except Exception as e:  # noqa: BLE001 - the proxy number stands on its own
            res["arrow_compute"] = {"error": repr(e)}
    for b in cols + [m for m in vl if m is not None] + [out, bits]:
        b.free()
    return res


def cpu_q6_arrow(cols, vl, rows: int, threads: int) -> dict:
    """The same predicate with pyarrow.compute over 1M-row RecordBatches on a thread pool (zero-copy
    views of the proxy's columns): compare -> and_kleene -> fill_null(false) -> indices_nonzero."""
    import concurrent.futures as cf
    import pyarrow as pa
    import pyarrow.compute as pc
    rows = min(rows, 256 << 20)           # bounded: arrow materialises every intermediate
    B = 1 << 20

    def arr(t, buf, vbuf, lo, n, width):
        bufs = [pa.py_buffer(vbuf.array) if vbuf is not None else None,
                pa.py_buffer(buf.array)]
        return pa.Array.from_buffers(t, lo + n, bufs).slice(lo, n)

    def one(lo):
        n = min(B, rows - lo)
        s = arr(pa.int32(), cols[0], vl[0], lo, n, 4)
        d = arr(pa.float64(), cols[1], vl[1], lo, n, 8)
        q = arr(pa.float64(), cols[2], vl[2], lo, n, 8)
        m = pc.and_kleene(pc.and_kleene(pc.greater_equal(s, 8766), pc.less(s, 9131)),
                          pc.and_kleene(pc.and_kleene(pc.greater_equal(d, 0.05), pc.less_equal(d, 0.07)),
                                        pc.less(q, 24.0)))
        return len(pc.indices_nonzero(pc.fill_null(m, False)))

    pa.set_cpu_count(1)                    # parallelism comes from the batch-level pool below
    with cf.ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(one, range(0, min(rows, 8 * B), B)))          # warm-up
        t0 = time.perf_counter()
        sel = sum(ex.map(one, range(0, rows, B)))
        dt = time.perf_counter() - t0
    return {"value": rows / dt, "unit": "rows/s", "cores": threads, "rows": rows, "selected": int(sel),
            "kind": "pyarrow.compute %s, 1M-row batches on %d threads (not Gandiva)" % (pa.__version__, threads)}


def run_reference(args):
    """--impl reference: the reference's CPU path, timed on this box's host cores.  dremio/gandiva
    cannot be built here (no source in /root/reference, no LLVM): the arm is the fused C++ proxy of the
    row loop its JIT emits (oracle/cpu_proxy.cc), all hardware threads, on the SAME workload and the
    same rows per step as the GPU arm (bounded only by host memory)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rows = args.cpu_rows or args.rows or (1_000_000_000 if world == 1 else 1_250_000_000)
    res = cpu_q6(rows, max(args.steps, 1), max(args.warmup, 1))
    rps = res["value"]
    line = {
        "impl": "reference", "metric": METRIC,
        "value": rps, "unit": "rows/s", "n_gpus": args.gpus, "steps": res["steps"],
        "warmup": max(args.warmup, 1), "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "TPC-H Q6 filter (BASELINE.json configs[1]%s)" %
                               ("; configs[4] sharding" if world > 1 else ""),
                   "rows_per_step": res["rows_per_step"],
                   "note": "CPU arm: one host, all cores, whatever --gpus says; rows per step = the GPU arm's rows "
                           "per GPU (bounded by host memory)"},
        "cpu_baseline": res,
        "e2e": {"value": rps, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# =================================================================================================
# `configs` entries (N=1): the other single-GPU workloads of BASELINE.json
# =================================================================================================
def _time_stream(torch, stream, fn, reps, warm=3):
    for _ in range(warm):
        fn()
    stream.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    stream.synchronize()
    return e0.elapsed_time(e1) / reps


def _unpack_bits(torch, words_i32, n):
    """LSB-first validity bitmap (int32 words on the device) -> bool[n]."""
    b = words_i32.view(torch.uint8)
    sh = torch.arange(8, device=b.device, dtype=torch.uint8)
    return ((b.unsqueeze(1) >> sh) & 1).flatten()[:n].bool()


def cfg_q6_nulls(ctx):
    """configs[1] with validity bitmaps (1 % nulls per column) on the resident Q6 columns."""
    torch, gandiva, cases = ctx["torch"], ctx["gandiva"], ctx["cases"]
    dev, stream, st, n = ctx["dev"], ctx["stream"], ctx["st"], ctx["n"]
    ship, disc, qty = ctx["q6_cols"]
    W = (n + 31) // 32
    vl = [torch.empty(W, dtype=torch.int32, device=dev) for _ in range(3)]
    for kind, t, v in ((0, ship, vl[0]), (1, disc, vl[1]), (2, qty, vl[2])):
        gandiva.generate_lineitem(ctx["local_rank"], kind, 42, 0, n, t.data_ptr(), v.data_ptr(), 10, st)
    filt, _ = q6_filter(gandiva, cases, gandiva.Configuration(device=ctx["local_rank"]))
    out, cnt = ctx["out_idx"], ctx["d_count"]
    cols = [(v.data_ptr(), t.data_ptr(), 0, 0) for t, v in zip((ship, disc, qty), vl)]

    def run():
        filt.evaluate_device(n, cols, out.data_ptr(), n, "UINT32", st, cnt.data_ptr(), sync=False)
    ms = _time_stream(torch, stream, run, 5)
    count = filt.sync(st)
    algo = n * (20.0 + 3 / 8.0) + 4.0 * count
    mask = (ship >= 8766) & (ship < 9131) & (disc >= 0.05) & (disc <= 0.07) & (qty < 24)
    for v in vl:
        mask &= _unpack_bits(torch, v, n)
    want = torch.nonzero(mask).flatten()
    got = out[:count].to(torch.int64) & 0xFFFFFFFF
    ok = count == want.numel() and bool(torch.equal(got, want))
    del mask, want, got
    info = filt.kernel_info
    return {"workload": "TPC-H Q6 filter, 1 %% nulls in every column (configs[1] with validity bitmaps), %d rows" % n,
            "rows": n, "rows_per_s": n / ms * 1e3, "kernel_ms": ms, "kernel": info["name"].rsplit("_", 1)[0],
            "regs": info["regs"], "selected": int(count),
            "algorithmic_bytes_per_row": algo / n,
            "full_size_check": "ok: == nonzero(torch mask & validity)" if ok else "FAILED",
            "_algo_bytes": algo}


def cfg_q1(ctx):
    """configs[2]: eight-output Q1 projector, 2 % nulls per column, ~1e9 rows resident, evaluated in chunks."""
    import pyarrow as pa
    torch, gandiva, cases = ctx["torch"], ctx["gandiva"], ctx["cases"]
    dev, stream, st = ctx["dev"], ctx["stream"], ctx["st"]
    chunk = 1 << 26
    free_b, _ = torch.cuda.mem_get_info(dev)
    chunks = int(min(15, (free_b * 0.9 - chunk * Q1_OUT_BYTES) // (chunk * Q1_IN_BYTES)))
    if chunks < 1:
        return {"error": "not enough free HBM for one Q1 chunk"}
    n = chunks * chunk
    W = n // 32
    ins, vls = [], []
    for kind, f in zip(cases.Q1_KINDS, cases.Q1_SCHEMA):
        w = f.type.bit_width // 8
        vals = torch.empty(n * w, dtype=torch.uint8, device=dev)
        vld = torch.empty(W, dtype=torch.int32, device=dev)
        gandiva.generate_lineitem(ctx["local_rank"], kind, 42, 0, n, vals.data_ptr(), vld.data_ptr(), 20, st)
        ins.append((vals, w))
        vls.append(vld)
    b = gandiva.TreeExprBuilder()
    outs_t = cases.q1_outputs(b)
    exprs = [b.make_expression(r, pa.field("o%d" % i, t)) for i, (r, t) in enumerate(outs_t)]
    p = gandiva.make_projector(cases.Q1_SCHEMA, exprs, None, "NONE", gandiva.Configuration(device=ctx["local_rank"]))
    outs = []
    for _, t in outs_t:
        v = torch.empty(chunk * (t.bit_width // 8), dtype=torch.uint8, device=dev)
        vl = torch.empty(chunk // 32, dtype=torch.int32, device=dev)
        outs.append((vl, v))
    optrs = [(vl.data_ptr(), v.data_ptr()) for vl, v in outs]

    def cols_of(c):
        lo = c * chunk
        return [(vls[j].data_ptr() + lo // 8, ins[j][0].data_ptr() + lo * ins[j][1], 0, 0) for j in range(8)]
    col_sets = [cols_of(c) for c in range(chunks)]

    def run():
        for c in range(chunks):
            p.evaluate_device(chunk, col_sets[c], optrs, st)
    ms = _time_stream(torch, stream, run, 3, warm=2)
    p.sync(st)
    info = p.kernel_info

    # full-size check: every chunk re-evaluated and compared with torch arithmetic on the same columns
    bad = []
    i64 = torch.int64

    def col(j, c, dt):
        lo = c * chunk
        w = ins[j][1]
        return ins[j][0][lo * w:(lo + chunk) * w].view(dt)

    def bits(t, c):
        return _unpack_bits(torch, t[c * chunk // 32:(c + 1) * chunk // 32], chunk)
    for c in range(chunks):
        p.evaluate_device(chunk, col_sets[c], optrs, st)
        p.sync(st)
        vq, ve, vd, vt, vef, vdf, vtf, vs = [bits(vls[j], c) for j in range(8)]
        qty = col(0, c, i64)
        ext, disc, tax = [col(j, c, i64).view(-1, 2) for j in (1, 2, 3)]
        extf, discf, taxf = [col(j, c, torch.float64) for j in (4, 5, 6)]
        ship = col(7, c, torch.int32)
        d1 = ext[:, 0] * (100 - disc[:, 0])
        d2 = d1 * (100 + tax[:, 0])
        f1 = extf * (1.0 - discf)
        f2 = f1 * (1.0 + taxf)
        taken = vdf & (discf > 0.05)
        zero = torch.zeros((), dtype=torch.float64, device=dev)
        want = [(d1, ve & vd), (d2, ve & vd & vt), (f1, vef & vdf), (f2, vef & vdf & vtf), (qty + qty, vq),
                (torch.where(taken, extf, zero), torch.where(taken, vef, torch.ones_like(vef))),
                ((vq & (qty < 24)).to(i64), torch.ones_like(vq)), (qty, vs & (ship <= 10471) & vq)]
        for k, (wv, wvalid) in enumerate(want):
            gvalid = _unpack_bits(torch, outs[k][0], chunk)
            if not bool(torch.equal(gvalid, wvalid)):
                bad.append("chunk %d output %d validity" % (c, k))
                continue
            if k < 2:     # decimal128: low word == int64 product, high word == its sign extension
                g = outs[k][1].view(i64).view(-1, 2)
                okv = bool(torch.equal(g[:, 0][wvalid], wv[wvalid])) and bool(torch.equal(g[:, 1][wvalid], (wv >> 63)[wvalid]))
            else:
                g = outs[k][1].view(wv.dtype)
                okv = bool(torch.equal(g[wvalid], wv[wvalid]))      # bit-exact, floats included
            if not okv:
                bad.append("chunk %d output %d values" % (c, k))
        del want
    algo = n * (Q1_IN_BYTES + Q1_OUT_BYTES)
    return {"workload": "TPC-H Q1 eight-output projector (configs[2]): decimal128/float64/int64 arithmetic + CASE, 2 %% nulls "
                        "per column, %d rows resident in HBM, %d launches of %d rows per pass" % (n, chunks, chunk),
            "rows": n, "rows_per_s": n / ms * 1e3, "kernel_ms": ms / chunks, "ms_per_pass": ms,
            "kernel": info["name"].rsplit("_", 1)[0], "regs": info["regs"],
            "loader": "tma-bulk" if info.get("staged") else "ldg", "stages": info.get("stages"),
            "dynamic_smem": info.get("dynamic_smem"), "algorithmic_bytes_per_row": Q1_IN_BYTES + Q1_OUT_BYTES,
            "full_size_check": ("ok: all %d chunks == torch evaluation of the 8 outputs (values bit-exact on valid rows, "
                                "validity bit-exact)" % chunks) if not bad else "FAILED: " + "; ".join(bad[:4]),
            "_algo_bytes": algo}


def _comment_block(cases, seed, block_rows):
    import numpy as np
    hb = cases.comment_batch(block_rows, seed=seed)
    arr = hb.column(0)
    offs = np.frombuffer(arr.buffers()[1], dtype=np.int32)[: block_rows + 1].astype(np.int64)
    data = np.frombuffer(arr.buffers()[2], dtype=np.uint8)[: offs[-1]]
    vbits = np.frombuffer(arr.buffers()[0], dtype=np.uint8)[: block_rows // 8]
    return hb, offs, data, vbits


def cfg_str(ctx):
    """configs[3]: like(upper(substr(l_comment,1,32)), '%SPECIAL%REQUESTS%') over 1e8 rows in 2 RecordBatches."""
    import numpy as np
    import oracle
    from oracle.tree import TreeBuilder
    torch, gandiva, cases = ctx["torch"], ctx["gandiva"], ctx["cases"]
    dev, stream, st = ctx["dev"], ctx["stream"], ctx["st"]
    block_rows, reps = 2_000_000, 25
    n = block_rows * reps
    batches, want_blocks, block_bytes = [], [], []
    for seed in (42, 43):
        hb, offs, data, vbits = _comment_block(cases, seed, block_rows)
        bb = int(offs[-1])
        assert bb * reps < 2 ** 31
        d_block = torch.from_numpy(data.copy()).to(dev)
        o_block = torch.from_numpy(offs.copy()).to(dev)
        v_block = torch.from_numpy(vbits.copy()).to(dev)
        d_bytes = d_block.repeat(reps)
        shifts = (torch.arange(reps, device=dev, dtype=torch.int64) * bb).repeat_interleave(block_rows)
        d_offs = torch.empty(n + 1, dtype=torch.int32, device=dev)
        d_offs[:n] = (o_block[:block_rows].repeat(reps) + shifts).to(torch.int32)
        d_offs[n] = bb * reps
        d_vld = v_block.repeat(reps)
        del shifts
        batches.append((d_vld, d_offs, d_bytes))
        block_bytes.append(bb)
        want_blocks.append(oracle.filter_indices(cases.comment_condition(TreeBuilder()), hb,
                                                 threads=min(oracle.hardware_threads(), 32)))
    b = gandiva.TreeExprBuilder()
    f = gandiva.make_filter(cases.COMMENT_SCHEMA, b.make_condition(cases.comment_condition(b)),
                            gandiva.Configuration(device=ctx["local_rank"]))
    outs = [torch.empty(n, dtype=torch.int32, device=dev) for _ in batches]
    cnts = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in batches]
    colsets = [[(v.data_ptr(), o.data_ptr(), d.data_ptr(), 0)] for v, o, d in batches]

    def run():
        for k in range(len(batches)):
            f.evaluate_device(n, colsets[k], outs[k].data_ptr(), n, "UINT32", st, cnts[k].data_ptr(), sync=False)
    ms = _time_stream(torch, stream, run, 5)
    f.sync(st)
    counts = [int(c.item()) for c in cnts]
    ok = True
    for k in range(len(batches)):       # the oracle's answer for the 2M-row block, tiled over the batch
        w = torch.from_numpy(want_blocks[k].astype(np.int64)).to(dev)
        want = (w.unsqueeze(0) + (torch.arange(reps, device=dev, dtype=torch.int64) * block_rows).unsqueeze(1)).flatten()
        got = outs[k][:counts[k]].to(torch.int64) & 0xFFFFFFFF
        ok = ok and counts[k] == want.numel() and bool(torch.equal(got, want))
    rows = n * len(batches)
    algo = sum(4.0 * (n + 1) + bb * reps + n / 8.0 + 4.0 * c for bb, c in zip(block_bytes, counts))
    info = f.kernel_info
    return {"workload": "string filter like(upper(substr(l_comment,1,32)),'%%SPECIAL%%REQUESTS%%') (configs[3]): %d rows in %d "
                        "RecordBatches of %d rows (int32 offsets), 1 %% nulls" % (rows, len(batches), n),
            "rows": rows, "rows_per_s": rows / ms * 1e3, "kernel_ms": ms / len(batches), "ms_per_pass": ms,
            "kernel": info["name"].rsplit("_", 1)[0], "regs": info["regs"], "dynamic_smem": info.get("dynamic_smem"),
            "block_threads": info["block_threads"], "selected": sum(counts), "algorithmic_bytes_per_row": algo / rows,
            "full_size_check": "ok: both batches == oracle indices of the 2M-row block tiled over the batch" if ok else "FAILED",
            "_algo_bytes": algo}


def cfg_ab_1m(ctx):
    """configs[0]: add(int32, int32) Projector over a 1M-row RecordBatch with 10 % nulls: per-call latency through the
    C-ABI with host buffers (H2D + kernel + D2H, synchronous, as Projector::Evaluate is) and device-resident."""
    import ctypes as C
    import numpy as np
    import pyarrow as pa
    import oracle
    torch, gandiva, cases = ctx["torch"], ctx["gandiva"], ctx["cases"]
    dev, stream, st = ctx["dev"], ctx["stream"], ctx["st"]
    n = 1_000_000
    b = gandiva.TreeExprBuilder()
    schema, outs_t, _ = cases.case_arith("add", pa.int32())(b)
    batch = cases.random_batch(schema, n, seed=1, null_prob=0.1)
    p = gandiva.make_projector(schema, [b.make_expression(outs_t[0][0], pa.field("c", pa.int32()))], None, "NONE",
                               gandiva.Configuration(device=ctx["local_rank"]))
    want, = oracle.project([outs_t[0][0]], [pa.int32()], batch, threads=4)
    got, = p.evaluate(batch)
    ok = got.equals(want)
    # host path, raw C-ABI (no Python array wrapping in the timed loop)
    cb, keep = gandiva._batch_to_c(batch)
    out_v = np.zeros(n, dtype=np.int32)
    out_b = np.zeros((n + 63) // 64 * 8, dtype=np.uint8)
    oc = (gandiva.gdv_out_column_t * 1)()
    oc[0].values = out_v.ctypes.data
    oc[0].validity = out_b.ctypes.data
    sh = gandiva._stream_handle(st)

    def call():
        gandiva._check(gandiva.lib.gdv_projector_evaluate(p._h, C.byref(cb), None, oc, 1, sh, 0))
    for _ in range(5):
        call()
    lat = []
    for _ in range(50):
        t0 = time.perf_counter()
        call()
        lat.append(time.perf_counter() - t0)
    host_ok = np.array_equal(out_v[np.asarray(want.is_valid())], want.drop_null().to_numpy())
    # device-resident
    a_d = torch.from_numpy(np.frombuffer(batch.column(0).buffers()[1], dtype=np.int32)[:n].copy()).to(dev)
    b_d = torch.from_numpy(np.frombuffer(batch.column(1).buffers()[1], dtype=np.int32)[:n].copy()).to(dev)
    va = torch.from_numpy(np.frombuffer(batch.column(0).buffers()[0], dtype=np.uint8)[:(n + 7) // 8].copy()).to(dev)
    vb = torch.from_numpy(np.frombuffer(batch.column(1).buffers()[0], dtype=np.uint8)[:(n + 7) // 8].copy()).to(dev)
    pad = lambda t: torch.cat([t, torch.zeros(8, dtype=torch.uint8, device=dev)])   # noqa: E731
    va, vb = pad(va), pad(vb)
    o_d = torch.empty(n, dtype=torch.int32, device=dev)
    ov = torch.empty((n + 31) // 32, dtype=torch.int32, device=dev)
    cols = [(va.data_ptr(), a_d.data_ptr(), 0, 0), (vb.data_ptr(), b_d.data_ptr(), 0, 0)]

    def run():
        p.evaluate_device(n, cols, [(ov.data_ptr(), o_d.data_ptr())], st)
    ms = _time_stream(torch, stream, run, 200, warm=20)
    p.sync(st)
    algo = n * 12.375
    med = _median(lat)
    info = p.kernel_info
    return {"workload": "add(int32,int32) Projector over one 1M-row RecordBatch, 10 %% nulls per column (configs[0]); per-call "
                        "latency, host buffers through gdv_projector_evaluate(GDV_MEM_HOST)",
            "rows": n, "rows_per_s": n / med, "host_call_us_median": med * 1e6, "host_call_us_min": min(lat) * 1e6,
            "h2d_bytes_per_call": int(n * 8.25), "d2h_bytes_per_call": int(n * 4.125),
            "kernel_ms": ms, "device_resident_rows_per_s": n / ms * 1e3, "kernel": info["name"].rsplit("_", 1)[0],
            "regs": info["regs"], "algorithmic_bytes_per_row": 12.375,
            "note": "1M rows = 12.4 MB: far below the ~100 MB a B200 needs in flight to reach its HBM roofline; the figure that "
                    "matters here is the per-call latency next to the CPU arm's",
            "full_size_check": "ok: == oracle (python mirror and raw C-ABI host call)" if (ok and host_ok) else "FAILED",
            "_algo_bytes": algo}


def cpu_configs(only) -> dict:
    """CPU arm (fused-cxx-proxy, all threads unless stated) for the `configs` entries."""
    import numpy as np
    from oracle import cpu_proxy as px
    import cases
    T = px.threads()
    res = {}

    def timeit(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return _median(ts)
    if "q6_nulls" in only:
        r = cpu_q6(256 << 20, 5, 2, nullp=10, arrow=False)
        res["q6_nulls"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "rows_per_step", "ms_per_step", "host_gbs")}
    if "q1" in only:
        n = cpu_rows_that_fit(64 << 20, Q1_IN_BYTES + Q1_OUT_BYTES + 8)
        ins, vins = [], []
        for kind in cases.Q1_KINDS:
            v, m = px.generate(kind, 42, 0, n, 20)
            ins.append(v)
            vins.append(m)
        outs = [px.Buf(n * w, np.uint8) for w in (16, 16, 8, 8, 8, 8, 8, 8)]
        vouts = [px.Buf((n + 7) // 8 + 8, np.uint8) for _ in range(8)]
        dt = timeit(lambda: px.q1_project(ins, vins, n, outs, vouts))
        res["q1"] = {"value": n / dt, "unit": "rows/s", "cores": T, "kind": "fused-cxx-proxy", "rows_per_step": n,
                     "ms_per_step": dt * 1e3, "host_gbs": n * (Q1_IN_BYTES + Q1_OUT_BYTES) / dt / 1e9,
                     "note": "ONE fused loop for all eight outputs (the reference's JIT runs one loop per output expression)"}
        for x in ins + vins + outs + vouts:
            x.free()
    if "str" in only:
        block_rows, reps = 2_000_000, 8
        hb, offs, data, vbits = _comment_block(cases, 42, block_rows)
        n = block_rows * reps
        bb = int(offs[-1])
        d = px.Buf(bb * reps + 64, np.uint8)
        o = px.Buf(n + 1, np.int32)
        v = px.Buf(n // 8 + 8, np.uint8)
        big_o = (np.tile(offs[:block_rows], reps) + np.repeat(np.arange(reps, dtype=np.int64) * bb, block_rows)).astype(np.int32)
        o.array[:n] = big_o
        o.array[n] = bb * reps
        d.array[:bb * reps] = np.tile(data, reps)
        v.array[:n // 8] = np.tile(vbits, reps)
        out = px.Buf(n, np.uint32)
        bits = px.Buf(n // 64 + 2, np.uint64)
        dt = timeit(lambda: px.comment_filter(o, d, v, n, out, bits))
        res["str"] = {"value": n / dt, "unit": "rows/s", "cores": T, "kind": "fused-cxx-proxy", "rows_per_step": n,
                      "ms_per_step": dt * 1e3, "host_gbs": (4.0 * n + bb * reps + n / 8.0) / dt / 1e9}
        for x in (d, o, v, out, bits):
            x.free()
    if "ab_1m" in only:
        n = 1_000_000
        a, va = px.generate(9, 1, 0, n, 100)
        b, vb = px.generate(10, 1, 0, n, 100)
        out = px.Buf(n, np.int32)
        vo = px.Buf(n // 8 + 16, np.uint8)
        dt1 = timeit(lambda: px.add_i32_inline(a, b, va, vb, n, out, vo), reps=100, warm=10)
        dtp = timeit(lambda: px.add_i32(a, b, va, vb, n, out, vo), reps=100, warm=10)
        res["ab_1m"] = {"value": n / dt1, "unit": "rows/s", "cores": 1, "kind": "fused-cxx-proxy", "call_us_median": dt1 * 1e6,
                        "note": "one 1M-row batch on ONE thread (how the reference evaluates a RecordBatch); 12 MB, cache-resident "
                                "after the first call",
                        "all_threads": {"value": n / dtp, "cores": T, "call_us_median": dtp * 1e6,
                                        "note": "the same batch split over the pinned pool: waking %d threads costs more than the work" % T}}
    return res


def run_configs(ctx, only):
    peak, _ = measured_peak_gbs()
    torch = ctx["torch"]
    table = {"q6_nulls": cfg_q6_nulls, "q1": cfg_q1, "str": cfg_str, "ab_1m": cfg_ab_1m}
    out = {}
    for name in ("q6_nulls", "q1", "str", "ab_1m"):
        if name not in only:
            continue
        if name == "q1":       # the Q1 inputs (84 GB) need the HBM the Q6 columns hold
            for k in ("q6_cols", "out_idx"):
                ctx[k] = None
            ctx["release"]()
            torch.cuda.empty_cache()
        try:
            t0 = time.perf_counter()
            r = table[name](ctx)
            if "kernel_ms" in r and "_algo_bytes" in r:
                ms_total = r.get("ms_per_pass", r["kernel_ms"])
                ach = r.pop("_algo_bytes") / (ms_total * 1e-3) / 1e9
                r["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak}
            r["wall_s"] = time.perf_counter() - t0
            out[name] = r
        except Exception as e:  # noqa: BLE001 - one workload failing must not lose the bench line
            import traceback
            out[name] = {"error": repr(e), "trace": traceback.format_exc()[-600:]}
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    return out


# =================================================================================================
def gpu_numa_cpus(torch, dev):
    """(node, cpus) of the NUMA node the GPU hangs off (sysfs), or (None, None)."""
    try:
        pr = torch.cuda.get_device_properties(dev)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(path).read().strip())
        if node < 0:
            return None, None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        return (node, cpus) if cpus else (None, None)
    except Exception:  # noqa: BLE001 - no sysfs / attribute: run unbound
        return None, None


DUMP_SAMPLE = 3 << 20    # entries kept of a longer SelectionVector: 2 x 24 MB with their positions


def dump_outputs(directory, vec, count):
    """--dump-outputs: the SelectionVector a caller of the timed path receives (`count` row numbers, ascending)
    as float64, exact below 2**53.  selection_count.npy holds the count; selection_vector.npy the vector, or,
    when it is longer than 2 x DUMP_SAMPLE entries, the entries at DUMP_SAMPLE positions drawn with a fixed
    seed, which selection_positions.npy holds.  At most 48 MB in all."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    idx = vec[:count].to(torch.int64)
    if vec.dtype == torch.int32:                  # UINT32 entries live in an int32 tensor
        idx &= 0xFFFFFFFF
    np.save(os.path.join(directory, "selection_count.npy"), np.array([count], dtype=np.float64))
    positions = os.path.join(directory, "selection_positions.npy")
    if idx.numel() > 2 * DUMP_SAMPLE:
        pos = np.sort(np.random.default_rng(0).choice(idx.numel(), DUMP_SAMPLE, replace=False))
        idx = idx[torch.from_numpy(pos).to(idx.device)]
        np.save(positions, pos.astype(np.float64))
    elif os.path.exists(positions):              # left by an earlier, sampled run
        os.remove(positions)
    np.save(os.path.join(directory, "selection_vector.npy"), idx.cpu().numpy().astype(np.float64))


def main():
    sys.dont_write_bytecode = True   # no __pycache__ in the tree, which may be read-only
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import cases
    import gandiva_b200 as gandiva

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    # The process that feeds a GPU runs on the CPUs of the GPU's NUMA node (what a one-process-per-GPU launcher
    # does with numactl / --cpunodebind): host batches are then allocated next to the link.  On the two-socket
    # bench box the pageable e2e path varied 25-47 GB/s with the feeding thread left to float.  Undone before
    # the CPU arms run, which use every core of the box.
    affinity0 = os.sched_getaffinity(0)
    numa_node, numa_cpus = gpu_numa_cpus(torch, dev)
    if numa_cpus and not args.no_numa_bind:
        try:
            os.sched_setaffinity(0, numa_cpus)
        except OSError:       # a container that forbids it: run unbound
            numa_cpus = None
    stream = torch.cuda.Stream(dev)   # a real (non-default) stream: events, kernels and
    torch.cuda.set_stream(stream)     # NCCL ops are all ordered on it
    st = stream.cuda_stream

    n_nominal = args.rows or (1_000_000_000 if world == 1 else 1_250_000_000)
    total_rows = n_nominal * world
    n, first_row = n_nominal, rank * n_nominal
    idx_mode = "UINT32" if (world == 1 and n <= (1 << 32)) else "UINT64"
    idx_dtype = torch.int32 if idx_mode == "UINT32" else torch.int64
    use_push = world > 1 and not args.no_gather and args.gather == "push"
    if args.dump_outputs and world > 1 and not use_push:
        raise SystemExit("--dump-outputs with N>1 needs --gather push (the vector a caller receives is rank 0's)")
    sm_reserve = args.sm_reserve if args.sm_reserve >= 0 else ((2 if use_push else 4) if world > 1 and not args.no_gather else 0)
    cfg = gandiva.Configuration(device=local_rank, rows_per_thread=args.rows_per_thread,
                                block_threads=args.block_threads, sm_reserve=sm_reserve)
    filt, _ = q6_filter(gandiva, cases, cfg)

    # ---- inputs resident in HBM (generated on device; same stream as oracle/lineitem.h) -----
    cap_rows = n_nominal if world == 1 else (int(n_nominal * 1.05) // 64 + 1) * 64
    ship_full = torch.empty(cap_rows, dtype=torch.int32, device=dev)
    disc_full = torch.empty(cap_rows, dtype=torch.float64, device=dev)
    qty_full = torch.empty(cap_rows, dtype=torch.float64, device=dev)

    def generate(first, rows, at=0):
        for kind, t in ((0, ship_full), (1, disc_full), (2, qty_full)):
            gandiva.generate_lineitem(local_rank, kind, 42, first, rows, t.data_ptr() + at * t.element_size(), 0, 0, st)
    generate(first_row, n)
    d_count = torch.zeros(1, dtype=torch.int64, device=dev)
    cols = [(0, ship_full.data_ptr(), 0, 0), (0, disc_full.data_ptr(), 0, 0), (0, qty_full.data_ptr(), 0, 0)]
    torch.cuda.synchronize()

    # ---- N>1 with the SelectionVector reassembled on rank 0: the root's shard is smaller ----------
    # Rank 0 does everything the other ranks do AND absorbs their runs: (N-1) x selectivity x 8 B per row
    # land in its HBM while its own filter streams 20 B per row, and an incoming write costs the memory
    # system about twice what a streamed read does (measured: +0.39 ms per 1.27 GB at N=8, +0.16 ms per
    # 0.54 GB at N=4, profiles/r02_multi_gpu.md).  With equal shards every step waits for rank 0; shards
    # sized so that all ranks finish together keep the same total (N x rows) and the same global order.
    # The selectivity is measured by one calibration pass over the equal shards.
    shard_rows = [n_nominal] * world
    shard_note = None
    if use_push and not args.equal_shards:
        scratch_idx = torch.empty(1 << 20, dtype=idx_dtype, device=dev)
        filt.evaluate_device(n, cols, scratch_idx.data_ptr(), scratch_idx.numel(), idx_mode + "|BOUNDED", st,
                             d_count.data_ptr(), sync=False, index_base=first_row)
        c = torch.tensor([filt.sync(st)], dtype=torch.int64, device=dev)
        dist.all_reduce(c)
        sel = float(c.item()) / total_rows
        write_cost = 2.0
        from gandiva_b200.sharding import shard_rows_with_root
        shard_rows = shard_rows_with_root(total_rows, world, sel, ALGO_IN_BYTES_PER_ROW, 8, write_cost)
        if max(shard_rows) <= cap_rows and min(shard_rows) > 0:
            n = shard_rows[rank]
            first_row = sum(shard_rows[:rank])
            generate(first_row, n)
            shard_note = ("rank 0 also absorbs the other ranks' runs: shards sized so that all ranks finish together "
                          "(selectivity %.4f from a calibration pass, an incoming 8-byte index costed as %.0f B of streaming)"
                          % (sel, write_cost * 8.0))
        else:
            shard_rows = [n_nominal] * world
        del scratch_idx
        torch.cuda.synchronize()
    # ---- waves: the shard is filtered in slices, global row order wave-major -------------------------
    waves = max(1, args.waves) if use_push else 1
    wave_rows, wave_first = None, None
    if waves > 1:
        from gandiva_b200.sharding import wave_layout
        all_rows, all_first = wave_layout(shard_rows, waves)
        wave_rows, wave_first = all_rows[rank], all_first[rank]
        if min(wave_rows) <= 0:
            waves, wave_rows, wave_first = 1, None, None
        else:
            at = 0
            for j in range(waves):
                generate(wave_first[j], wave_rows[j], at)
                at += wave_rows[j]
            torch.cuda.synchronize()
    ship, disc, qty = ship_full[:n], disc_full[:n], qty_full[:n]
    out_idx = None if use_push else torch.empty(n, dtype=idx_dtype, device=dev)

    from gandiva_b200.sharding import gather_selection
    pipelined = world > 1 and not args.no_gather and not args.no_overlap and not use_push
    ps = None
    if use_push:
        from gandiva_b200.sharding import PeerSelection
        ps = PeerSelection(capacity=int(total_rows * 0.03) + 4096,
                           local_rows=cap_rows if waves == 1 else max(wave_rows), mode=idx_mode, device=dev,
                           slots=2, ctas=args.push_ctas, waves=waves)
    gstep = {"i": 0}
    # N>1: the gather of batch i runs on a second stream while the filter kernel of batch i+1
    # runs (double-buffered index buffers).  The filter was built with sm_reserve so that the
    # copy CTAs find free slots next to the persistent filter CTAs.
    comm_stream = torch.cuda.Stream(dev) if world > 1 else None
    if use_push:                       # the kernel-only timing below writes here
        out_idx = ps.local[0] if (rank != 0 and waves == 1) else torch.empty(n, dtype=idx_dtype, device=dev)
    bufs = [out_idx, torch.empty(n, dtype=idx_dtype, device=dev) if pipelined else out_idx]
    cnts = [d_count, torch.zeros(1, dtype=torch.int64, device=dev)]
    host_cnt = [torch.zeros(1, dtype=torch.int64).pin_memory() for _ in range(2)]
    ev_k = [torch.cuda.Event() for _ in range(2)]
    ev_g = [torch.cuda.Event() for _ in range(2)]
    gathered = {"buf": None}

    def launch(i):
        b = i % 2
        filt.evaluate_device(n, cols, bufs[b].data_ptr(), n, idx_mode, st, cnts[b].data_ptr(),
                             sync=False, index_base=first_row)
        if world > 1 and not args.no_gather:
            host_cnt[b].copy_(cnts[b], non_blocking=True)
            ev_k[b].record(stream)

    def gather(i):
        b = i % 2
        ev_k[b].synchronize()              # kernel i and its count copy are done
        cnt = int(host_cnt[b][0])
        with torch.cuda.stream(comm_stream):
            comm_stream.wait_event(ev_k[b])
            out, total = gather_selection(bufs[b], cnt, dst=0, out=gathered["buf"])
            if rank == 0 and (gathered["buf"] is None or out.numel() > gathered["buf"].numel()):
                gathered["buf"] = torch.empty(int(total * 1.1) + 16, dtype=idx_dtype, device=dev)
            ev_g[b].record(comm_stream)
        return total

    def run_steps_push(k, events=None):
        """N>1, --gather push: filter kernel i+1 overlaps the NVLink push of run i; nothing
        touches the host between steps."""
        for i in range(k):
            g = gstep["i"]
            gstep["i"] += 1
            if waves == 1:
                ps.before_filter(g, stream)
                ptr, cap, mode, cnt_ptr = ps.filter_target(g)
                filt.evaluate_device(n, cols, ptr, cap, mode, st, cnt_ptr, sync=False, index_base=first_row)
                # the last run of the job has no filter kernel to hide under: push it with the whole GPU
                ps.after_filter(g, stream, ctas=(2 * 148 if i == k - 1 else 0))
            else:
                at = 0
                for j in range(waves):
                    ps.before_filter(g, stream, wave=j)
                    ptr, cap, mode, cnt_ptr = ps.filter_target(g, wave=j)
                    wcols = [(0, ship_full.data_ptr() + 4 * at, 0, 0), (0, disc_full.data_ptr() + 8 * at, 0, 0),
                             (0, qty_full.data_ptr() + 8 * at, 0, 0)]
                    filt.evaluate_device(wave_rows[j], wcols, ptr, cap, mode, st, cnt_ptr, sync=False,
                                         index_base=wave_first[j])
                    ps.after_filter(g, stream, ctas=(2 * 148 if (i == k - 1 and j == waves - 1) else 0), wave=j)
                    at += wave_rows[j]
            if events is not None and i + 1 < k:
                events[i + 1].record(stream)
        ps.finish(stream)                          # the last step closes after its push landed
        if events is not None:
            events[k].record(stream)
        return None

    def run_steps(k, events=None):
        """k passes of the hot path; with N>1 each pass ends with the SelectionVector on rank 0."""
        if use_push:
            return run_steps_push(k, events)
        total = None
        for i in range(k):
            if pipelined and i >= 2:
                stream.wait_event(ev_g[i % 2])      # buffer i%2 is free again
            launch(i)
            if world > 1 and not args.no_gather:
                if pipelined:
                    if i >= 1:
                        total = gather(i - 1)
                else:
                    total = gather(i)
                    stream.wait_event(ev_g[i % 2])
            if events is not None:
                events[i + 1].record(stream)
        if pipelined and k >= 1:
            total = gather(k - 1)
            stream.wait_event(ev_g[(k - 1) % 2])
            if k >= 2:
                stream.wait_event(ev_g[k % 2])
            if events is not None:
                events[k].record(stream)          # the last event closes after the last gather
        return total

    run_steps(max(args.warmup, 3))
    count = filt.sync(st)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = gandiva.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    torch.cuda.synchronize()
    ev[0].record(stream)
    run_steps(args.steps, ev)
    torch.cuda.synchronize()
    total_ms = ev[0].elapsed_time(ev[args.steps])
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    launches = gandiva.launch_count() - launches0
    count = filt.sync(st)
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        tc = torch.tensor([count], dtype=torch.int64, device=dev)
        dist.all_reduce(tc)
        total_selected = int(tc.item())
    else:
        total_selected = count
    ms_per_step = total_ms / args.steps
    value = total_rows / (ms_per_step * 1e-3)
    gather_check = None
    full_check = None
    if world == 1:
        # outside the timed region, at the full bench size: the SelectionVector of the last step is
        # ascending, its length is the count of an independent torch evaluation of the predicate,
        # and it holds exactly torch.nonzero of that mask
        try:
            torch.cuda.synchronize()
            mask = (ship >= 8766) & (ship < 9131) & (disc >= 0.05) & (disc <= 0.07) & (qty < 24)
            want_n = int(mask.sum().item())
            idx = out_idx[:count].to(torch.int64)
            if idx_mode == "UINT32":
                idx = idx & 0xFFFFFFFF
            ok = (count == want_n)
            if ok and count > 1:
                ok = bool((idx[1:] > idx[:-1]).all().item())
            ok = ok and bool(torch.equal(idx, torch.nonzero(mask).flatten()))
            full_check = ("ok: %d rows == torch mask count, ascending, == nonzero(mask)" % count) if ok else \
                         ("FAILED: count %d, torch %d" % (count, want_n))
            del mask, idx
        except Exception as e:  # noqa: BLE001 - the bench line must still be printed
            full_check = "not run: %r" % (e,)
    if use_push:
        # outside the timed region: the last step's vector on rank 0 is complete and holds EXACTLY the
        # rows an independent torch evaluation of the predicate selects on every rank, in order:
        # every rank computes nonzero(mask) + first_row of its shard, rank 0 gathers them (NCCL, not
        # the push path) and compares element-wise with the pushed vector
        torch.cuda.synchronize()
        dist.barrier()
        mask = (ship >= 8766) & (ship < 9131) & (disc >= 0.05) & (disc <= 0.07) & (qty < 24)
        if waves == 1:
            mine = [torch.nonzero(mask).flatten() + first_row]
        else:                               # wave-major global row order: one run per (wave, rank)
            mine, at = [], 0
            for j in range(waves):
                mine.append(torch.nonzero(mask[at:at + wave_rows[j]]).flatten() + wave_first[j])
                at += wave_rows[j]
        del mask
        sizes = [torch.zeros(waves, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([m.numel() for m in mine], dtype=torch.int64, device=dev))
        sizes = [[int(x) for x in s_.tolist()] for s_ in sizes]
        total_selected = sum(sum(s_) for s_ in sizes)
        ok = True
        if rank == 0:
            vec, total = ps.result(gstep["i"] - 1)
            ok = (total == total_selected) and not ps.overflowed()
            pos = 0
            for j in range(waves):
                for r in range(world):
                    part = mine[j] if r == 0 else torch.empty(sizes[r][j], dtype=torch.int64, device=dev)
                    if r != 0:
                        dist.recv(part, src=r)
                    ok = ok and bool(torch.equal(vec[pos:pos + sizes[r][j]].to(torch.int64), part))
                    pos += sizes[r][j]
            gather_check = ("ok: %d global indices on rank 0 == concat over %s of nonzero(torch mask) + slice base"
                            % (total, "ranks" if waves == 1 else "(wave, rank)")) if ok else "FAILED"
        else:
            for j in range(waves):
                dist.send(mine[j], dst=0)
        del mine
    if args.dump_outputs and rank == 0:             # before the kernel-only timing below reuses out_idx
        vec, total = ps.result(gstep["i"] - 1) if use_push else (out_idx, count)
        dump_outputs(args.dump_outputs, vec, total)

    # ---- roofline of the dominant (only) kernel ----------------------------------------------
    peak, peak_src = measured_peak_gbs()
    # kernel-only duration: time K evaluate calls without the gather
    kev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    kreps = max(3, min(args.steps, 10))
    torch.cuda.synchronize()
    kev[0].record(stream)
    for _ in range(kreps):
        filt.evaluate_device(n, cols, out_idx.data_ptr(), n, idx_mode, st, d_count.data_ptr(),
                             sync=False, index_base=first_row)
    kev[1].record(stream)
    torch.cuda.synchronize()
    count = filt.sync(st)
    algo_bytes = ALGO_IN_BYTES_PER_ROW * n + (IDX_BYTES if idx_mode == "UINT32" else 8.0) * count
    kernel_ms = kev[0].elapsed_time(kev[1]) / kreps
    achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
    info = filt.kernel_info
    traffic = None
    try:  # DRAM bytes per launch from the committed ncu --set full capture of this kernel/config
        tj = json.load(open(os.path.join(ROOT, "profiles", "q6_filter_traffic.json")))
        if int(tj["rows"]) == n and idx_mode == "UINT32":
            traffic = float(tj["traffic_bytes_per_launch"])
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic,
                "traffic_source": "profiles/q6_filter_traffic.json (ncu --set full capture of this kernel at this size, "
                                  "committed; not re-measured in this run)" if traffic else None,
                "peak_source": peak_src,
                "kernel": info["name"].rsplit("_", 1)[0], "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_launch": algo_bytes, "regs": info["regs"],
                "rows_per_thread": info["rows_per_thread"], "block_threads": info["block_threads"]}

    # ---- e2e: host buffers through the C-ABI, copies inside the timed region -----------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, gandiva, cases, torch, np, dev, local_rank, rank, world, n,
                      ship, disc, qty, first_row)

    # ---- the other single-GPU workloads -------------------------------------------------------
    configs = None
    only = [x for x in (args.only.split(",") if args.only else ["q6_nulls", "q1", "str", "ab_1m"]) if x]
    if world == 1 and not args.no_configs:
        holder = {"ship": ship, "disc": disc, "qty": qty}

        def release():
            holder.clear()
        ctx = {"torch": torch, "gandiva": gandiva, "cases": cases, "dev": dev, "stream": stream, "st": st, "n": n,
               "local_rank": local_rank, "q6_cols": (ship, disc, qty), "out_idx": out_idx, "d_count": d_count,
               "release": release}
        del ship, disc, qty, out_idx, bufs, cols
        configs = run_configs(ctx, only)

    for tid in os.listdir("/proc/self/task"):      # threads created while bound inherited the mask
        try:
            os.sched_setaffinity(int(tid), affinity0)
        except OSError:
            pass
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            cpu = cpu_q6(args.cpu_rows or n, 7, 2)
            if configs is not None:
                for name, r in cpu_configs(only).items():
                    if name in configs:
                        configs[name]["cpu"] = r
        except Exception as e:  # noqa: BLE001
            cpu = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value,
            "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "TPC-H Q6 filter (BASELINE.json configs[1]%s)" %
                                   ("; configs[4] sharding" if world > 1 else ""),
                       "rows_per_gpu": n_nominal, "total_rows": total_rows, "selectivity": total_selected / total_rows,
                       "shard_rows": shard_rows if world > 1 else None, "shard_note": shard_note,
                       "selection_vector": idx_mode + ((" reassembled on rank 0 over NVLink" + (", gdv_selection_push: device-side stores into rank 0's vector (CUDA IPC), counts exchanged through a board in rank 0's HBM, no host sync, overlapped with the next batch's kernel (%d SMs reserved)" % sm_reserve if use_push else (", NCCL send/recv, overlapped with the next batch's kernel" if pipelined else ", NCCL send/recv"))) if world > 1 and not args.no_gather else ""),
                       "gather_check": gather_check, "full_size_check": full_check,
                       "l2_policy": "inputs (20 B/row x %d rows) larger than L2; no flush" % n,
                       "host_numa": ("process bound to NUMA node %d, the GPU's (%d CPUs), for the GPU arm" % (numa_node, len(numa_cpus)))
                                    if (numa_cpus and not args.no_numa_bind) else "unbound",
                       "parallelism": "row-range shards, %d" % world},
            "hbm_gbs": achieved, "per_step_ms": per_step,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clocks, "configs": configs,
        }
        print(json.dumps(line))
    if world > 1:
        if ps is not None:
            ps.close()
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(args, gandiva, cases, torch, np, dev, local_rank, rank, world, n, ship, disc, qty,
            first_row):
    """Q6 through gdv_filter_evaluate with HOST buffers: every step copies its input columns H2D,
    runs the fused kernel, and copies the selection vector D2H.  Measured twice: pinned host buffers
    (gdv_host_alloc) and pageable ones (posix_memalign, what an Arrow MemoryPool returns)."""
    import ctypes as C
    import psutil
    rows = args.e2e_rows or n
    if world > 1:   # every rank stages its own host copy: bound the node's total (the per-GPU rate is the PCIe link's)
        rows = min(rows, 512 * 1024 * 1024)
    avail = psutil.virtual_memory().available
    need = rows * 24 + (1 << 30)
    if need * world > avail * 0.5:
        rows = int(avail * 0.5 / world - (1 << 30)) // 24 // 1024 * 1024
    chunk = min(args.e2e_chunk, rows)
    rows = rows // chunk * chunk
    if rows <= 0:
        return None
    libc = C.CDLL(None)
    libc.posix_memalign.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t]
    libc.free.argtypes = [C.c_void_p]

    def pinned(nbytes):
        p = C.c_void_p()
        gandiva._check(gandiva.lib.gdv_host_alloc(nbytes, C.byref(p)))
        return p

    def pageable(nbytes):
        p = C.c_void_p()
        if libc.posix_memalign(C.byref(p), 64, nbytes) != 0:
            raise MemoryError("posix_memalign")
        return p

    def host_view(ptr, count, np_dtype):
        ct = np.ctypeslib.as_ctypes_type(np_dtype)
        return torch.from_numpy(np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(count,)))

    filt, _ = q6_filter(gandiva, cases, gandiva.Configuration(device=local_rank))
    stream = torch.cuda.current_stream()

    def measure(alloc, free, steps):
        h_ship, h_disc, h_qty = alloc(rows * 4), alloc(rows * 8), alloc(rows * 8)
        h_idx = alloc(chunk * 4)
        try:
            host_view(h_ship, rows, np.int32).copy_(ship[:rows])
            host_view(h_disc, rows, np.float64).copy_(disc[:rows])
            host_view(h_qty, rows, np.float64).copy_(qty[:rows])
            torch.cuda.synchronize()

            def one_pass():
                total = 0
                for c0 in range(0, rows, chunk):
                    cols = (gandiva.gdv_column_t * 3)()
                    cols[0].values = h_ship.value + c0 * 4
                    cols[1].values = h_disc.value + c0 * 8
                    cols[2].values = h_qty.value + c0 * 8
                    cb = gandiva.gdv_batch_t(chunk, 3, gandiva.GDV_MEM_HOST, cols)
                    sel = gandiva.gdv_selection_t(h_idx, chunk, 0, gandiva.GDV_SEL_UINT32,
                                                  gandiva.GDV_MEM_HOST, 0)
                    gandiva._check(gandiva.lib.gdv_filter_evaluate(filt._h, C.byref(cb), C.byref(sel),
                                                                   gandiva._stream_handle(stream.cuda_stream), 0, None))
                    total += sel.num_slots
                return total
            one_pass()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            t0 = time.perf_counter()
            sel_total = 0
            for _ in range(steps):
                sel_total = one_pass()
            e1.record(stream)
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) / steps
            ms = e0.elapsed_time(e1) / steps
            return max(wall, ms * 1e-3), sel_total
        finally:
            for p in (h_ship, h_disc, h_qty, h_idx):
                free(p)

    steps = max(1, min(args.steps, 3))
    sec, sel_total = measure(pinned, gandiva.lib.gdv_host_free, steps)
    sec_pg, _ = measure(pageable, libc.free, steps)
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([sec, sec_pg], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec, sec_pg = float(t[0].item()), float(t[1].item())
    h2d = int(rows * 20) * world
    return {"value": rows * world / sec, "unit": "rows/s",
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(sel_total * 4 + 8 * (rows // chunk)) * world,
            "rows_per_step": rows * world, "chunk_rows": chunk, "ms_per_step": sec * 1e3,
            "h2d_gbs": h2d / sec / 1e9,
            "pcie_note": "PCIe Gen5 x16 moves ~55 GB/s per direction per GPU: 20 B/row caps host-resident Q6 at ~2.8e9 "
                         "rows/s per GPU whatever the kernel does",
            "pageable": {"value": rows * world / sec_pg, "unit": "rows/s", "ms_per_step": sec_pg * 1e3,
                         "h2d_gbs": h2d / sec_pg / 1e9,
                         "buffers": "posix_memalign (pageable), staged through the engine's pinned ring"},
            "api": "gdv_filter_evaluate(GDV_MEM_HOST), pinned host buffers (value) / pageable (pageable.value), one call per "
                   "%d-row RecordBatch" % chunk}


if __name__ == "__main__":
    main()
