#!/usr/bin/env python
"""bench.py — update-rows/sec through the TPC-H-Q3-shaped delta join + reduce.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W`
prints ONE JSON line.  A step is one pass of the hot path over one update batch
(~100K update rows per GPU at one new timestamp: arrange x4, three delta paths x
two half_joins, accumulable reduce, compaction).

  value   whole-job update-rows/s with the batch already resident in HBM
  e2e     the same through the public C-ABI harness with HOST (pinned) buffers:
          H2D of the batch and D2H of the output corrections inside the timed region
  roofline  dominant kernel of the step, timed live with CUDA events on the
          launching stream (mzgpu_profile_*), against MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (C++ restatement of the reference algorithms; the
          Rust reference cannot be built here) on the box's host cores

`--impl reference` times that CPU implementation alone on the same config.
`--dump-outputs DIR` writes the output corrections of the last timed step (either arm) as
DIR/<field>.npy; the seeded inputs are the same from run to run, so two builds compare output for output.
Multi-GPU (torchrun, one rank per GPU): key-sharded arrangements, NCCL
all-to-all per exchange point, weak scaling (SF and batch grow with N).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 7
ORDERS_PER_BATCH_PER_GPU = 10_000  # ~100K update rows (2 order rows + ~8 lineitem rows per replaced order)
P2P_LANDING_ROWS = 1 << 19  # capacity of one landing region (rows one worker may send to one peer per buffer and round)


def scale(sf):
    return dict(n_customer=int(150_000 * sf), n_orders=int(1_500_000 * sf), n_part=int(200_000 * sf))


def sf_per_gpu(args, n):
    """BASELINE.json configs[2] is SF=10 on one GPU, configs[4] SF=100 over 8 GPUs: one GPU runs
    SF=10, N > 1 GPUs run SF=12.5 per GPU (25 / 50 / 100 at N = 2 / 4 / 8).  The update batch --
    the unit of work a step processes -- is ~100K rows per GPU at every N (weak scaling)."""
    return args.sf if n <= 1 else args.sf_multi


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []
        self.nvml, self.handle, self.samples, self.thread = None, None, [], None
        self.stop_flag = threading.Event()

    # -- in-process NVML (a query costs microseconds, so even a 10 ms timed region is sampled);
    #    nvidia-smi -lms (below) is the fallback when NVML cannot be loaded
    def _nvml_open(self):
        import pynvml

        pynvml.nvmlInit()
        handle = None
        try:
            import torch

            uuid = str(torch.cuda.get_device_properties(self.device).uuid)
            uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            try:
                handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except TypeError:
                handle = pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            handle = None
        if handle is None:
            handle = pynvml.nvmlDeviceGetHandleByIndex(self.device)
        self.nvml, self.handle = pynvml, handle
        self.sample_now()  # fails here (-> fallback) rather than in the thread

    def sample_now(self):
        """One sample of (SM MHz, max SM MHz, event-reason bits); called from the sampling thread and
        once by the timing loop itself while the GPU still has the timed steps queued."""
        if self.nvml is None:
            return
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        try:
            bits = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            bits = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        self.samples.append((float(sm), float(mx), int(bits)))

    def _poll(self):
        while not self.stop_flag.is_set():
            try:
                self.sample_now()
            except Exception:
                return
            time.sleep(0.004)

    def start(self):
        try:
            self._nvml_open()
            self.samples = []  # the probe sample was taken before the timed region
            if os.environ.get("MZ_CLOCK_SAMPLER", "1") != "0":  # (0: only the sample the timing loop takes itself)
                self.thread = threading.Thread(target=self._poll, daemon=True)
                self.thread.start()
            return
        except Exception:
            self.nvml, self.thread = None, None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL,
                text=True,
            )
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def _stop_nvml(self):
        self.stop_flag.set()
        if self.thread is not None:
            self.thread.join(timeout=1.0)
        n = self.nvml
        names = [
            ("hw_slowdown", getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8)),
            ("hw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
            ("sw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)),
            ("sw_power_cap", getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)),
        ]
        sm = sorted(x[0] for x in self.samples)
        reasons = sorted({nm for _, _, bits in self.samples for nm, bit in names if bits & bit})
        return {
            "sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": max(x[1] for x in self.samples) if self.samples else None,
            "samples": len(sm),
            "reasons": reasons,
            "source": "nvml",
        }

    def stop(self):
        if self.nvml is not None:
            try:
                return self._stop_nvml()
            except Exception as e:  # never let the sampler take the bench line down
                return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": [f"nvml: {e}"]}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {
            "sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


def oracle_workers():
    """Worker threads of the CPU oracle dataflow: every host core (one timely worker per core, as
    the reference deploys), unless MZ_ORACLE_WORKERS says otherwise.  At ~100K-row batches the
    oracle is synchronisation bound well before 128 workers (8 workers on 8 cores already reach
    ~1.2e7 rows/s at SF=1), so a smaller count can be the stronger baseline on a big host."""
    try:
        w = int(os.environ.get("MZ_ORACLE_WORKERS", "0"))
    except ValueError:
        w = 0
    return w if w > 0 else (os.cpu_count() or 1)


def oracle_candidates(sf_total):
    """Worker counts tried for the CPU arm; the best one is reported.  The oracle dataflow is
    synchronisation bound at ~100K-row batches long before it runs out of cores, so fewer workers
    than cores is often the stronger baseline (BASELINE.md section 3)."""
    cores = os.cpu_count() or 1
    if os.environ.get("MZ_ORACLE_WORKERS"):
        return [oracle_workers()]
    cand = [w for w in (8, 16, 32, 64) if w < cores] + [cores]
    if sf_total > 20:  # hydration of a big instance with few workers takes minutes: top two only
        cand = cand[-2:]
    return cand


def run_oracle(B, sf_total, per_batch, workers, n_warm, n_steps, keep_outputs=False):
    """Hydrate the CPU dataflow, run batches 0 .. n_warm + n_steps - 1 in order (timestamps as in
    the GPU arm), time the last n_steps.  Returns (rows/s, rows, seconds, hydration seconds,
    [output corrections per batch] if keep_outputs)."""
    t0 = time.time()
    o = B.Q3(seed=SEED, workers=workers, per_batch=per_batch, **scale(sf_total))
    o.hydrate()
    o.drain()
    hyd = time.time() - t0
    outs, rows, secs = [], 0, 0.0
    for b in range(n_warm + n_steps):
        s_, r_ = o.step(b)
        if b >= n_warm:
            secs += s_
            rows += r_
        if keep_outputs:
            outs.append(o.drain())
    if not keep_outputs:
        o.drain()
    del o
    return rows / secs, rows, secs, hyd, outs


def best_oracle(B, sf_total, per_batch, n_warm, n_steps, keep_outputs_of_first=False):
    """Sweep the worker counts; the first candidate can keep its outputs (they do not depend on
    the worker count) for the parity check."""
    table, best, outs = [], None, []
    for i, w in enumerate(oracle_candidates(sf_total)):
        keep = keep_outputs_of_first and i == 0
        v, rows, secs, hyd, o = run_oracle(B, sf_total, per_batch, w, n_warm, n_steps, keep)
        if keep:
            outs = o
        table.append({"workers": w, "value": v, "hydration_s": round(hyd, 1)})
        if best is None or v > best["value"]:
            best = {"workers": w, "value": v, "rows": rows, "secs": secs, "hyd": hyd}
    return best, table, outs


DUMP_FIELDS = ("key", "count", "sum", "flags", "time", "diff")
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, rows):
    """Write one step's output corrections (ROUT rows) as out_dir/<field>.npy, one float64 array per
    field of DUMP_FIELDS, rows sorted on every field so that two builds compare array for array.
    The 128-bit SUM is rounded to float64 once; the other fields are integers below 2**53 (group
    keys are 45 bits) and are exact.  Beyond DUMP_MAX_BYTES, a seeded sample of the rows is written."""
    import numpy as np

    order = ("key", "count", "sum_hi", "sum_lo", "flags", "time", "diff")
    rows = rows[np.lexsort([rows[f] for f in reversed(order)])]
    n_max = DUMP_MAX_BYTES // (8 * len(DUMP_FIELDS))
    if len(rows) > n_max:
        rows = rows[np.sort(np.random.default_rng(SEED).choice(len(rows), n_max, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for f in DUMP_FIELDS:
        if f == "sum":
            a = np.array([float((int(h) << 64) + int(lo)) for h, lo in zip(rows["sum_hi"], rows["sum_lo"])], dtype=np.float64)
        else:
            a = rows[f].astype(np.float64)
        np.save(os.path.join(out_dir, f + ".npy"), a)


def measured_peak():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# ------------------------------------------------------- the CPU reference
def run_reference(args, rank):
    """The reference's CPU implementation of the path: the C++ oracle dataflow with
    all host threads, on the same config / metric / unit."""
    if rank != 0:
        return
    from oracle import binding as B

    # same workload as our arm at --gpus N (weak scaling: SF and batch grow with N)
    n = max(1, args.gpus)
    sf = sf_per_gpu(args, n) * n
    best, table, outs = best_oracle(B, sf, ORDERS_PER_BATCH_PER_GPU * n, args.warmup, args.steps,
                                    keep_outputs_of_first=bool(args.dump_outputs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs[args.warmup + args.steps - 1])
    cores, value, rows, secs = best["workers"], best["value"], best["rows"], best["secs"]
    sample = (f"SF={sf:g} hydrated in {best['hyd']:.1f}s (untimed), {args.steps} batches of ~{rows // max(1, args.steps)} update rows;"
              f" best of worker counts {[t['workers'] for t in table]} on {os.cpu_count()} host cores")
    line = {
        "impl": "reference",
        "metric": "update_rows_per_sec",
        "value": value,
        "unit": "rows/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1000.0 * secs / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "int64",
        "data": "synthetic",
        "config": workload_config(sf_per_gpu(args, n), n),
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample,
                         "worker_sweep": table},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(sf_per_gpu, n):
    return {
        "workload": f"TPC-H-Q3-shaped 3-way delta join + accumulable reduce, synthetic SF={sf_per_gpu * n:g}"
        f" ({sf_per_gpu:g}/GPU), ~100K-row update batches per GPU"
        + (" = BASELINE.json configs[2]" if n == 1 else f" = BASELINE.json configs[4] (SF=100 at 8 GPUs) at N={n}"),
        "scaling_note": "weak scaling: every GPU processes one ~100K-row update batch per step at every N; the"
        " arrangements hold SF=10 on one GPU and SF=12.5 per GPU beyond (SF=100 at N=8, configs[4])",
        "sf_total": sf_per_gpu * n,
        "orders_replaced_per_batch": ORDERS_PER_BATCH_PER_GPU * n,
        "parallelism": f"key-hash sharded x{n}; exchange rounds over NVLink peer memory (one scatter + one gather kernel,"
        " no host wait), NCCL all-to-all for hydration chunks" if n > 1 else "1 GPU",
        "l2": "inputs_larger_than_l2 (arrangements >= 5 GB/GPU vs 126 MB L2)",
        "plan": "customer>>orders[custkey]>>lineitem[orderkey]; orders>>customer>>lineitem; lineitem>>orders[orderkey]>>customer",
    }


class stdout_to_stderr:
    """fd-level redirect: NCCL prints its version banner to stdout during communicator
    creation; the contract is ONE JSON line on stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


# ------------------------------------------------------------------- ours
def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch

    import materialize_b200 as mz
    from materialize_b200 import harness

    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        # NCCL's debug output (version banner, nranks, transports) goes to stderr, at whatever
        # level the caller asked for: stdout carries ONE JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

        dist = dist_mod
        torch.cuda.set_device(local_rank)
        with stdout_to_stderr():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    ctx = mz.Context(local_rank, rank, world)
    if world > 1:
        # the worker mesh bootstrap stays on the host (timely does its own): rank 0
        # creates the NCCL id, the others receive it
        import ctypes as C

        from materialize_b200 import _ffi as F

        idbuf = (C.c_uint8 * F.COMM_ID_BYTES)()
        if rank == 0:
            ctx.check(F.lib.mzgpu_comm_unique_id(idbuf))
        with stdout_to_stderr():
            t = torch.tensor(list(idbuf), dtype=torch.uint8, device="cuda")
            dist.broadcast(t, 0)
        idbuf = (C.c_uint8 * F.COMM_ID_BYTES)(*t.cpu().tolist())
        with stdout_to_stderr():
            ctx.check(F.lib.mzgpu_comm_init(ctx.h, idbuf))
            # first collectives on both communicators (lazy NCCL initialisation prints here)
            w = torch.zeros(1, device="cuda")
            dist.all_reduce(w)
            torch.cuda.synchronize()

    p2p = False
    if world > 1:
        import ctypes as C

        import numpy as np

        from materialize_b200 import _ffi as F

        with stdout_to_stderr():
            # NCCL connects peers lazily on first use: one small all-to-all now, so that connection
            # setup is not counted as hydration
            warm_in = mz.DeviceRows(ctx, 32).upload(np.zeros(4096, dtype=mz.R32))
            warm_out = mz.DeviceRows(ctx, 32)
            ctx.check(F.lib.mzgpu_exchange(ctx.h, warm_in.h, warm_out.h))
            ctx.sync()
        if os.environ.get("MZGPU_P2P", "1") != "0":
            # update-batch exchange rounds over peer memory: every rank exports its landing zone
            # (CUDA IPC handle), the handles are all-gathered on the host side, every rank maps all
            hnd = mz.p2p_export(ctx, P2P_LANDING_ROWS, 32)
            t = torch.tensor(list(hnd), dtype=torch.uint8, device="cuda")
            ts = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(ts, t)
            mz.p2p_import(ctx, [bytes(x.cpu().tolist()) for x in ts])
            dist.barrier()
            p2p = True

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def allmax(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    sf = sf_per_gpu(args, world) * world
    per_batch = ORDERS_PER_BATCH_PER_GPU * world
    q = harness.Q3Dataflow(ctx, SEED, per_batch=per_batch, worker=rank, peers=world, **scale(sf))
    if p2p:
        q.use_p2p(True)
    barrier()
    t0 = time.time()
    hyd_rows = q.hydrate()
    ctx.sync()
    hyd_s = time.time() - t0
    q.clear_out()

    n_warm, n_timed, n_e2e, n_prof = args.warmup, args.steps, args.steps, max(3, min(args.steps, 10))
    total_batches = n_warm + n_timed + n_warm + n_e2e + n_prof
    # stage every batch up front (generation is not part of a step)
    staged, staged_rows = [], []
    t_first = q.time()
    for b in range(total_batches):
        rows = q.stage_batch(b, t_first + b)
        staged.append([q.staged_copy(a) for a in (1, 2, 3)])
        staged_rows.append(rows)
    ext = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local_rank))

    OUT_ROWS_MAX = 1 << 16  # output corrections of one timestamp (a few hundred) -- checked on the device
    kept = mz.DeviceRows(ctx, 64)

    def run_device_step(b, keep=False):
        for a, d in zip((1, 2, 3), staged[b]):
            q.stage_device(a, d)
        q.step()
        if keep:
            q.keep_out(kept, OUT_ROWS_MAX)
        q.clear_out()

    # ---- device-resident timing
    b = 0
    for _ in range(n_warm):
        run_device_step(b)
        b += 1
    launches0 = ctx.stats()["kernel_launches"]
    clocks = ClockSampler(local_rank)
    barrier()
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    step_ev = [torch.cuda.Event(enable_timing=True) for _ in range(n_timed)]
    first_timed = b
    e0.record(ext)
    rows_timed = 0
    host_t0 = time.perf_counter()
    ht0 = ctx.host_times()
    hp0 = q.host_ns()
    for i in range(n_timed):
        # the output corrections of every timed step are appended (device to device, no read-back)
        # to `kept` and compared with the CPU oracle's after the region
        run_device_step(b, keep=True)
        step_ev[i].record(ext)
        rows_timed += staged_rows[b]
        b += 1
    host_enqueue_ms = 1e3 * (time.perf_counter() - host_t0) / n_timed  # host time per step inside the loop ...
    ht1 = ctx.host_times()
    hp1 = q.host_ns()
    host_phase_ms = {k: round((hp1[k] - hp0[k]) / 1e6 / n_timed, 4) for k in hp1}  # host time inside the harness's step, by phase
    host_alloc_ms = (ht1["alloc_ns"] - ht0["alloc_ns"]) / 1e6 / n_timed if "alloc_ns" in ht1 else None
    host_wait_ms = (ht1["wait_ns"] - ht0["wait_ns"]) / 1e6 / n_timed  # ... of which: waiting for the device
    e1.record(ext)
    try:
        clocks.sample_now()  # the GPU is still working through the queued steps
    except Exception:
        pass
    barrier()
    clk = clocks.stop()
    ms = allmax(e0.elapsed_time(e1))
    # completion-to-completion interval of consecutive steps on this rank's stream
    step_ms = sorted(([e0.elapsed_time(step_ev[0])] + [step_ev[i - 1].elapsed_time(step_ev[i]) for i in range(1, n_timed)]))
    per_step = {"min": step_ms[0], "median": step_ms[len(step_ms) // 2], "max": step_ms[-1]}
    timed_out = kept.download()  # (outside the timed region)
    launches = ctx.stats()["kernel_launches"] - launches0
    total_rows = allsum(rows_timed)
    value = total_rows / (ms / 1000.0)

    # ---- end to end: pinned host inputs, H2D + D2H inside the timed region
    host_batches = []
    for bb in range(b, b + n_warm + n_e2e):
        hb = []
        for d in staged[bb]:
            arr = d.download()
            pin = torch.empty(arr.nbytes, dtype=torch.uint8).pin_memory()
            view = pin.numpy().view(mz.R32)
            view[:] = arr
            hb.append((pin, view))
        host_batches.append(hb)
    out_pin = torch.empty(64 * 4_000_000, dtype=torch.uint8).pin_memory()
    out_view = out_pin.numpy().view(mz.ROUT)

    def stage_host_batch(hb):
        """H2D of one update batch (pinned host memory -> device staging) on the copy stream."""
        for a, (_, view) in zip((1, 2, 3), hb):
            q.stage_host(a, view)
        q.stage_commit()

    def run_host_steps(batches):
        """Each step: the batch's H2D copy, the timestamp, the D2H read of its output
        corrections.  The copy of batch i+1 is issued while timestamp i runs (double-buffered
        staging) and the corrections of timestamp i are copied out (copy stream) while timestamp
        i+1 runs, as a worker between a network source and a sink would; every copy of every
        step is inside the region, the last read-back drains the stream."""
        outs = 0
        stage_host_batch(batches[0])
        for i in range(len(batches)):
            q.step()
            if i + 1 < len(batches):
                stage_host_batch(batches[i + 1])
            outs += len(q.fetch_out(0, out_view))  # timestamp i-1 (nothing for i = 0)
        outs += len(q.fetch_out(1, out_view))  # the last timestamp
        return outs

    q.pipeline_out()
    run_host_steps(host_batches[:n_warm])
    b += n_warm
    barrier()
    s0 = ctx.stats()
    h2d0 = q.h2d_bytes()
    d2h0 = q.d2h_bytes()
    e0.record(ext)
    out_rows = run_host_steps(host_batches[n_warm : n_warm + n_e2e])
    rows_e2e = sum(staged_rows[b : b + n_e2e])
    b += n_e2e
    e1.record(ext)
    barrier()
    ms_e2e = allmax(e0.elapsed_time(e1))
    s1 = ctx.stats()
    e2e_value = allsum(rows_e2e) / (ms_e2e / 1000.0)
    h2d = (q.h2d_bytes() - h2d0) / n_e2e
    d2h = (s1["d2h_bytes"] - s0["d2h_bytes"] + q.d2h_bytes() - d2h0) / n_e2e

    # ---- live per-kernel timing (CUDA events around every launch) for the roofline
    ctx.profile(True)
    ctx.profile_report()
    for _ in range(n_prof):
        run_device_step(b)
        b += 1
    prof = ctx.profile_report()
    ctx.profile(False)
    tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
    ranked = sorted(prof.items(), key=lambda kv: -kv[1]["ms"])
    top_name, top = ranked[0]
    # the roofline record is for the kernel with the largest share of the step among those whose algorithmic
    # bytes are exact under profiling: the fused seal / merge kernel leaves a debug record with its row count,
    # the probe chains read their stream lengths back ahead of the launch (probe.cu), the merge-path tiles have
    # host-known sizes; the stream maps of the multi-GPU path report bytes only for host-known counts
    exact = [kv for kv in ranked if kv[1]["bytes"] > 0 and "map_rows" not in kv[0]]
    with_bytes = exact or [kv for kv in ranked if kv[1]["bytes"] > 0]
    dom_name, dom = with_bytes[0] if with_bytes else ranked[0]
    peak, peak_kind = measured_peak()
    achieved = dom["bytes"] / (dom["ms"] / 1000.0) / 1e9 if dom["ms"] > 0 else 0.0
    # DRAM traffic of the dominant kernel from the committed `ncu --set full` capture
    # (profiles/, same command line): mean of the captured launches, bytes per launch
    traffic = None
    try:
        import csv

        tag = "fused" if "fused" in dom_name else ("probe" if "probe" in dom_name else None)
        cands = [os.path.join(ROOT, "profiles", f"{r}_ncu_full_{tag}_raw.csv") for r in ("r02c", "r02")]
        path = next((c for c in cands if os.path.exists(c)), cands[-1])
        if tag and world == 1 and os.path.exists(path):
            rows = list(csv.reader(open(path)))
            hdr, units = rows[0], rows[1]
            tot = []
            for r in rows[2:]:
                b = 0.0
                for col in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    i = hdr.index(col)
                    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(units[i], 1.0)
                    b += float(r[i].replace(",", "")) * mult
                tot.append(b)
            traffic = sum(tot) / len(tot) if tot else None
    except Exception:
        traffic = None
    roofline = {
        "bound": "hbm",
        "kernel": dom_name,
        "achieved": achieved,
        "peak": peak,
        "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
        "unit": "GB/s",
        "frac": achieved / peak,
        "traffic": traffic,
        "traffic_source": "NOT measured in this run: mean DRAM bytes per launch of the committed ncu --set full capture of"
        f" the same command (profiles/{os.path.basename(path)})" if traffic else None,
        "launches_per_step": dom["launches"] / n_prof,
        "avg_launch_us": 1000.0 * dom["ms"] / max(1, dom["launches"]),
        "algorithmic_bytes_per_launch": dom["bytes"] / max(1, dom["launches"]),
        "share_of_kernel_time": dom["ms"] / tot_ms,
        "kernel_time_per_step_ms": tot_ms / n_prof,
        "top_kernels": [
            {"kernel": k, "share": round(v["ms"] / tot_ms, 4), "launches_per_step": v["launches"] / n_prof,
             "gbps": (v["bytes"] / (v["ms"] / 1000.0) / 1e9) if v["ms"] > 0 and v["bytes"] else None}
            for k, v in ranked[:8]
        ],
    }

    line = {
        "metric": "update_rows_per_sec",
        "value": value,
        "unit": "rows/s",
        "n_gpus": world,
        "steps": n_timed,
        "warmup": n_warm,
        "ms_per_step": ms / n_timed,
        "per_step_ms": per_step,
        "host_ms_per_step": {"loop": host_enqueue_ms, "waiting_for_device": host_wait_ms, "work": host_enqueue_ms - host_wait_ms,
                             "allocations": (ht1["allocs"] - ht0["allocs"]) / n_timed, "in_allocator": host_alloc_ms,
                             "harness_phases": host_phase_ms},
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "int64",
        "data": "synthetic",
        "config": workload_config(sf_per_gpu(args, world), world),
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "rows/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / n_e2e, "out_rows_per_step": out_rows / n_e2e},
        "gpu_launches": launches,
        "roofline": roofline,
        "hydration": {"rows": allsum(hyd_rows), "seconds": allmax(hyd_s)},
        "device_bytes_peak": ctx.stats()["device_bytes_peak"],
    }

    # ---- parity of the TIMED steps: every rank's output corrections of the timed region against
    # the CPU oracle dataflow on the same seeded batches (rank 0 runs the oracle: as the checker,
    # and at N=1 also as the reported CPU baseline -- a bounded sample of the same workload)
    want_oracle = not args.no_cpu_baseline
    gathered = timed_out
    if dist is not None and (want_oracle or args.dump_outputs):
        nn = torch.tensor([len(timed_out)], dtype=torch.int64, device="cuda")
        ns = [torch.zeros_like(nn) for _ in range(world)]
        dist.all_gather(ns, nn)
        mx = max(int(x.item()) for x in ns)
        buf = torch.zeros(max(mx, 1) * 64, dtype=torch.uint8, device="cuda")
        if len(timed_out):
            buf[: len(timed_out) * 64] = torch.from_numpy(timed_out.view(np.uint8).copy()).cuda()
        bufs = [torch.zeros_like(buf) for _ in range(world)]
        dist.all_gather(bufs, buf)
        gathered = np.concatenate([bb_[: int(k.item()) * 64].cpu().numpy().view(mz.ROUT) for bb_, k in zip(bufs, ns)])
    if rank == 0 and want_oracle:
        from oracle import binding as B

        n_cpu = max(args.cpu_batches, n_timed)
        best, table, outs = best_oracle(B, sf, per_batch, n_warm, n_cpu, keep_outputs_of_first=True)
        if world == 1:
            line["cpu_baseline"] = {
                "value": best["value"],
                "unit": "rows/s",
                "cores": best["workers"],
                "kind": "port",
                "worker_sweep": table,
                "sample": f"same workload: SF={sf:g} hydrated ({best['hyd']:.1f}s, untimed), {n_cpu} update batches of ~{best['rows'] // n_cpu} rows;"
                f" best of worker counts {[t['workers'] for t in table]} on {os.cpu_count()} host cores; C++ restatement of the"
                " reference CPU algorithms (Rust toolchain unavailable)",
            }
        ok, compared, bad = True, 0, []
        for i in range(n_timed):
            t = t_first + first_timed + i
            got = B.consolidate(gathered[gathered["time"] == t])
            want = outs[n_warm + i]
            compared += len(want)
            if got.tobytes() != want.tobytes():
                ok = False
                bad.append(int(t))
        line["parity"] = {
            "checked_steps": n_timed,
            "ok": ok,
            "rows_compared": compared,
            "against": f"CPU oracle dataflow, same seeded batches, SF={sf:g}; output corrections of the timed steps"
            f" (all {world} ranks gathered), bit-exact after consolidation",
            "mismatched_times": bad,
        }
    elif rank == 0:
        line["parity"] = None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, gathered[gathered["time"] == t_first + first_timed + n_timed - 1])
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sf", type=float, default=10, help="TPC-H scale factor on one GPU (BASELINE configs[2])")
    ap.add_argument("--sf-multi", type=float, default=12.5, help="scale factor per GPU at N > 1 (SF=100 at N=8, configs[4])")
    ap.add_argument("--cpu-batches", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output corrections of the last timed step to DIR/<field>.npy (float64)")
    args = ap.parse_args()
    args.warmup = max(3, args.warmup)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        print(json.dumps({"error": f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks"}))
        sys.exit(2)
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
