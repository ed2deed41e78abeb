#!/usr/bin/env python3
"""bench.py -- Session.Run samples/sec of the B200 op-kernel layer (BASELINE.json metric:
"Session.Run samples/sec (MLP-1024 & LeNet) at 1/2/4/8 B200 vs Eigen CPU").

    python bench.py --gpus N --steps K --warmup W            # this repo's arm
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port, see below)

ONE JSON line.  Its top level is the MLP record (BASELINE configs[1], the config the metric is
quoted on): 3-layer MLP 1024-1024-1024, batch 4096, fp32 graph, fwd + bwd + SGD, one "step" =
one Session.Run([loss, train_op]) through the C API (TF_SessionRun).  `workloads` carries the
same record for the other configs the metric names, each measured the same way in the same run:
    lenet     BASELINE configs[2]: LeNet-5 conv graph, batch 512, NHWC fp32
    mlp_bf16  BASELINE configs[3] per replica: the MLP with bf16 storage, fp32 accumulate
N>1: one process per GPU (torchrun), one graph replica per rank, weak scaling (per-replica batch
fixed), gradients averaged by ONE all-reduce of the gradient arena per step (B200AllReduceN).

Per record:
  value    samples/s with inputs resident in HBM (x / labels live in device variables).
  e2e      the same step fed from pinned HOST buffers through TF_SessionRun: H2D of x+labels and
           D2H of the loss inside the timed region.
  parity   step-1 loss, gradients and updated weights of THIS full-size graph vs the CPU oracle,
           computed before any timed region (tests/workloads.py::check_parity); N>1: vs the oracle
           on the global batch.
  roofline the tcgen05 GEMM / convolution kernels (dominant), device time per launch measured
           with CUDA events on the session's stream (b200_profile_begin/end) in a separate pass.
  cpu_baseline  the CPU oracle port (FMA build, oracle/_build/liboracle_fast.so) on the box's
           host cores, rank 0.
--impl reference times that same CPU port with all host threads (the reference's own CPU
implementation is unbuildable here: no bazel / protoc / Eigen; DESIGN.md section 3).

--dump-outputs DIR writes, per workload, what the last timed step handed back (the loss it
fetched and the trained variables it left) as DIR/<workload>_<name>.npy in float32.  Inputs and
initial weights are seeded, so two builds run with the same arguments can be compared array by
array.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "Session.Run samples/sec (MLP-1024 & LeNet) at 1/2/4/8 B200 vs Eigen CPU"
ALL_WORKLOADS = ["mlp", "lenet", "mlp_bf16"]
MIN_WARMUP = 20   # steps; the first steps after a cold start run below the sustained clock
DUMP_LIMIT_BYTES = 64 * 10**6   # all arrays of one --dump-outputs run together


# =================================================================================== CPU arm
def _cgroup_cpu_quota():
    """CPUs this container may use per the cgroup bandwidth controller (None = unlimited)."""
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]  # cgroup v2
        if quota != "max":
            return max(1, -(-int(quota) // int(period)))
        return None
    except Exception:
        pass
    try:  # cgroup v1
        quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if quota > 0 and period > 0:
            return max(1, -(-quota // period))
    except Exception:
        pass
    return None


def host_threads():
    """Threads of the CPU arms = the CPUs this process can really use: the schedulable CPUs (what
    the reference's NumSchedulableCPUs returns, platform/posix/port.cc:50-55), capped by the
    physical core count and by the container's cgroup CPU quota.  Measured on the GPU box
    (128 logical / 64 physical CPUs, cpu.max = 16 CPUs): 16 threads 40.2 K samples/s, 64 threads
    21.0 K, 128 threads 2.7 K -- oversubscribing the quota only throttles, and the baseline
    should be the CPU's best.  B200TF_HOST_THREADS overrides."""
    if os.environ.get("B200TF_HOST_THREADS"):
        return max(1, int(os.environ["B200TF_HOST_THREADS"]))
    n = len(os.sched_getaffinity(0))
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys:
            n = min(n, phys)
    except Exception:
        pass
    quota = _cgroup_cpu_quota()
    if quota:
        n = min(n, quota)
    return max(1, n)


def cpu_step_fn(w):
    """One full training step of workload `w` on the CPU port, FMA build (the timed CPU arm; the
    bit-stable -ffp-contract=off build stays the checker)."""
    import oracle_bind as o
    prev = o.select("fast")
    o.set_num_threads(host_threads())
    cores = o.num_threads()
    o.select(prev)
    # bf16 workloads: the reference's CPU device has no bf16 MatMul (types.proto:30 "only for
    # cast ops"), its CPU path for the same graph is fp32 -- that is what this arm times (the
    # bf16 storage rounding of tests/workloads.py is a numpy emulation for the parity check only)
    import workloads as W
    wt = W.MLP("f32", w.batch, w.width, w.layers) if w.dtype == "bf16" else w
    x, labels = wt.data(1234)
    params = wt.init_params()

    def step():
        prev = o.select("fast")
        try:
            return wt.reference_step(o, x, labels, params)
        finally:
            o.select(prev)

    return step, cores


def cpu_baseline(w, max_seconds=10.0, max_steps=200):
    step, cores = cpu_step_fn(w)
    step()  # warm-up (page faults, thread pool)
    t0 = time.perf_counter()
    n = 0
    while n < max_steps and (n == 0 or time.perf_counter() - t0 < max_seconds):
        step()
        n += 1
    dt = time.perf_counter() - t0
    gf = w.flops_per_step * n / dt / 1e9
    return {"value": w.batch * n / dt, "unit": "samples/s", "cores": cores, "kind": "port",
            "gflops": gf, "gflops_per_core": gf / cores,
            "build": "oracle.c -O3 -march=native -ffp-contract=fast (FMA), OpenMP",
            "sample": "%d full training steps (%s) of the CPU oracle port, OpenMP over %d host "
                      "threads; %.2f s" % (n, w.describe.split(";")[0], cores, dt)}


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return  # under torchrun only rank 0 runs the CPU arm
    import workloads as W
    records = {}
    for name in args.workloads:
        w = W.get(name)
        step, cores = cpu_step_fn(w)
        for _ in range(max(1, min(args.warmup, 2))):
            step()
        # each step is a full training step of the workload
        steps, t0 = args.steps, time.perf_counter()
        for _ in range(steps):
            step()
        dt = time.perf_counter() - t0
        value = w.batch * steps / dt
        gf = w.flops_per_step * steps / dt / 1e9
        note = ("CPU restatement of the reference's Eigen path, FMA build (reference unbuildable "
                "offline: needs bazel+protoc+Eigen)")
        if w.dtype == "bf16":
            note += ("; the reference has no bf16 MatMul on CPU (types.proto:30): this arm runs the "
                     "same graph in fp32")
        records[name] = {
            "impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w.describe, "note": note},
            "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port",
                             "gflops": gf, "gflops_per_core": gf / cores,
                             "sample": "%d full training steps, %d OpenMP threads, FMA build"
                                       % (steps, cores)},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
        }
    head = args.workloads[0]
    line = dict(records[head])
    line["workloads"] = {n: r for n, r in records.items() if n != head}
    print(json.dumps(line))


# =================================================================================== GPU arm
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region.

    ONE long-lived `nvidia-smi -lms 100` child, started before the warm-up: forking a process
    that holds a CUDA context costs tens of milliseconds, and a fork per sample inside the timed
    region stalled the launch loop (a 100-step LeNet pass read 1.19 ms/step with a per-sample
    subprocess, 0.60 without).  Only the samples between mark_begin() and mark_end() count."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []          # (wall time, fields)
        self.t_begin = self.t_end = None
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                line = line.strip()
                if line:
                    self.rows.append((time.time(), [c.strip() for c in line.split(",")]))
        except Exception:
            pass

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def summary(self):
        if self.t_end is None:
            self.mark_end()
        time.sleep(0.15)  # let the sample that covers the end of the region arrive
        try:
            if self.proc is not None:
                self.proc.terminate()
        except Exception:
            pass
        self.join(timeout=3)
        lo = (self.t_begin or 0.0) - 0.05
        hi = self.t_end + 0.15
        rows = [r for t, r in self.rows if lo <= t <= hi] or [r for _, r in self.rows[-2:]]
        sm = [float(r[1]) for r in rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for name, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(rows)}


def load_peaks():
    """Roofline denominators.  bf16 / HBM: MEASURED_PEAKS.json (driver-written).  TF32: the file
    has no TF32 figure, so tools/measure_peaks.py measured cuBLAS TF32 with the driver's protocol
    on this pool's B200 (committed: profiles/r02_measured_peaks.json).  Kernels timed per launch
    (this roofline pass) are compared with the BURST figure."""
    peaks, src = {}, {}
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peaks["bf16"] = d.get("bf16_tflops")
        src["bf16"] = "MEASURED_PEAKS.json bf16_tflops (burst, cuBLAS 8192^3)"
        peaks["hbm"] = d.get("hbm_gbs")
    except Exception:
        pass
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_measured_peaks.json")))
        peaks["tf32"] = d.get("tf32_tflops")
        src["tf32"] = ("profiles/r02_measured_peaks.json tf32_tflops (burst; cuBLAS TF32 8192^3, "
                       "tools/measure_peaks.py on this pool's B200; sustained %.0f)"
                       % d.get("tf32_tflops_sustained", 0))
        if not peaks.get("bf16"):
            peaks["bf16"] = d.get("bf16_tflops")
            src["bf16"] = "profiles/r02_measured_peaks.json bf16_tflops (burst)"
    except Exception:
        pass
    if not peaks.get("bf16"):
        peaks["bf16"], src["bf16"] = 1680.0, "fallback burst bf16 1.68 PF (B200_PROFILING.md)"
    if not peaks.get("tf32"):
        peaks["tf32"] = 0.5 * peaks["bf16"]
        src["tf32"] = "0.5 x " + src["bf16"] + " (no measured TF32 figure)"
    return peaks, src


def load_traffic(name):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    of this workload (profiles/r02_traffic.json); null when no capture is committed."""
    for f in ("r02_traffic.json",):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", f)))
            if name in d:
                return d[name].get("dram_bytes_per_launch"), d[name].get("source")
        except Exception:
            pass
    if name == "mlp":
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", "r01_gemm_traffic.json")))
            return d["dram_bytes_per_launch"], "ncu --set full capture of round 1 (profiles/r01_gemm_traffic.json)"
        except Exception:
            pass
    return None, None


class Bench:
    def __init__(self, args):
        import torch
        from simple_tensorflow_b200 import _lib
        self.args = args
        self.torch = torch
        self._lib = _lib
        self.L = _lib.load()
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world > 1:
            raise SystemExit("--gpus %d does not match WORLD_SIZE %d" % (args.gpus, self.world))
        if self.L.b200_device_count() < 1:
            raise SystemExit("bench.py needs a CUDA device: libb200tf has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.comm = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            from simple_tensorflow_b200 import replica
            self.comm = replica.init_nccl_comm(self.L, self.rank, self.world, self.local_rank)
        self.peaks, self.peak_src = load_peaks()
        self.outputs = {}   # --dump-outputs: name -> float32 array

    def collective_counts(self):
        p, n = ctypes.c_uint64(), ctypes.c_uint64()
        self.L.b200_collective_counts(ctypes.byref(p), ctypes.byref(n))
        return p.value, n.value

    def run_workload(self, name):
        import workloads as W
        from simple_tensorflow_b200 import client
        args, L, _lib, torch = self.args, self.L, self._lib, self.torch
        world, rank = self.world, self.rank
        w = W.get(name)
        B = w.build(num_replicas=world, seed=1234 + rank)
        tf = B.tf
        sess = client.Session(tf.get_default_graph(), gpu=self.local_rank,
                              collective_comm=self.comm, num_replicas=world)
        init = tf.global_variables_initializer()
        sess.run(init)
        stream = sess.stream()
        ev0, ev1 = ctypes.c_void_p(), ctypes.c_void_p()
        _lib.check(L.b200_event_create(ctypes.byref(ev0)))
        _lib.check(L.b200_event_create(ctypes.byref(ev1)))

        # ---- parity of the full-size graph, before anything is timed (all ranks: collective)
        parity = None
        if not args.no_parity:
            import oracle_bind as o
            o.select("exact")
            o.set_num_threads(host_threads())
            parity = W.check_parity(w, B, sess, o, world=world, rank=rank)
            # restore the initial weights: the timed runs start from the same state every time
            sess.run(init)

        hx, hl = w.host_tensor(B.x), w.host_tensor(B.labels)   # pinned, reused every step

        def barrier():
            _lib.check(L.b200_stream_synchronize(stream))
            torch.cuda.synchronize()
            if world > 1:
                import torch.distributed as dist
                dist.barrier()

        def timed(fetches, feed, steps, prefetch=None):
            """-> (device ms between events on the session stream, launches, last loss).

            prefetch: list of (HostTensor x, HostTensor labels) buffer pairs used round-robin; the
            inputs of step i+1 are staged (Session.stage: H2D on the copy stream) before step i is
            run, so every step's host->device copy is inside the timed region but overlaps the
            previous step's kernels."""
            launches, loss, enq = 0, None, 0
            barrier()
            _lib.check(L.b200_event_record(ev0, stream))
            staged = None
            if prefetch:
                staged = tuple(sess.stage(t) for t in prefetch[0])
            for i in range(steps):
                if prefetch:
                    nxt = (tuple(sess.stage(t) for t in prefetch[(i + 1) % len(prefetch)])
                           if i + 1 < steps else None)
                    loss = sess.run(fetches, {B.xp: staged[0], B.lp: staged[1]})[0]
                    staged = nxt
                else:
                    loss = sess.run(fetches, feed)[0]
                st = sess.last_run_stats()
                launches += st["kernels_launched"]
                enq += st["host_enqueue_us"]
            timed.host_enqueue_us = enq / max(steps, 1)
            _lib.check(L.b200_event_record(ev1, stream))
            barrier()
            ms = ctypes.c_float()
            _lib.check(L.b200_event_elapsed_ms(ev0, ev1, ctypes.byref(ms)))
            timed.last_loss = loss
            loss = float(np.asarray(w.to_f32(loss)).reshape(-1)[0])
            if world > 1:
                import torch.distributed as dist
                t = torch.tensor([ms.value], device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)  # max over ranks
                return float(t.item()), launches, loss
            return ms.value, launches, loss

        res_fetch = list(B.resident)
        fed_fetch = list(B.fed)
        feed = {B.xp: hx, B.lp: hl}
        # second pinned buffer pair: the input pipeline fills one while the other is in flight
        buffers = [(hx, hl), (w.host_tensor(B.x), w.host_tensor(B.labels))]
        sampler = ClockSampler(self.local_rank)
        if rank == 0:
            sampler.start()  # before the warm-up: its one fork stays outside the timed region
        warm = max(args.warmup, 3, MIN_WARMUP)
        for _ in range(warm):
            sess.run(res_fetch)
        for _ in range(max(args.warmup, 3)):
            sess.run(fed_fetch, feed)
        timed(fed_fetch, None, max(args.warmup, 3), prefetch=buffers)
        for _ in range(3):
            sess.run(res_fetch)

        sampler.mark_begin()
        c0 = self.collective_counts()
        ms_res, launches, loss_res = timed(res_fetch, None, args.steps)
        c1 = self.collective_counts()
        host_enqueue_us = timed.host_enqueue_us
        if args.dump_outputs and rank == 0:
            # read back before the passes below train the variables further
            self.outputs["%s_loss" % name] = w.to_f32(timed.last_loss)
            for n, a in zip(B.V, sess.run([v.ref for v in B.V.values()])):
                self.outputs["%s_%s" % (name, n)] = w.to_f32(a)
        # the same K steps again in chunks: the median chunk is the figure robust to a cold start
        chunk = max(1, args.steps // 5)
        chunks = [timed(res_fetch, None, chunk)[0] / chunk for _ in range(5)] if args.steps >= 10 else []
        ms_sync, _, _ = timed(fed_fetch, feed, args.steps)  # feed pinned buffers, copy inside Run()
        h2d = sess.last_run_stats()["h2d_bytes"]
        ms_e2e, _, loss_e2e = timed(fed_fetch, None, args.steps, prefetch=buffers)
        sampler.mark_end()
        clocks = sampler.summary() if rank == 0 else None
        assert sum(client.HostTensor.numpy(t).nbytes for t in buffers[0]) == h2d
        d2h = sess.last_run_stats()["d2h_bytes"]

        # ---- roofline pass: per-launch device time of the tcgen05 kernels, events on the same stream
        _lib.check(L.b200_profile_begin())
        prof_steps = min(args.steps, 20)
        for _ in range(prof_steps):
            sess.run(res_fetch)
        gemm_ms, gemm_n, gemm_fl = ctypes.c_double(), ctypes.c_uint64(), ctypes.c_double()
        _lib.check(L.b200_profile_end(ctypes.byref(gemm_ms), ctypes.byref(gemm_n),
                                      ctypes.byref(gemm_fl)))
        # what an event pair with nothing between costs on this stream
        pair = []
        for _ in range(50):
            _lib.check(L.b200_event_record(ev0, stream))
            _lib.check(L.b200_event_record(ev1, stream))
            _lib.check(L.b200_stream_synchronize(stream))
            ms_pair = ctypes.c_float()
            _lib.check(L.b200_event_elapsed_ms(ev0, ev1, ctypes.byref(ms_pair)))
            pair.append(ms_pair.value * 1e3)
        event_pair_us = statistics.median(pair)
        sess.close()
        if rank != 0:
            return None

        if world > 1:
            peer, nccl = c1[0] - c0[0], c1[1] - c0[1]
            collective = {"kind": "peer" if peer and not nccl else ("nccl" if nccl and not peer
                                                                    else "mixed" if peer else "none"),
                          "peer_backend": (L.b200_peer_arena_backend() or b"").decode(),
                          "peer_kernel_launches": peer, "nccl_calls": nccl,
                          "per_step": (peer + nccl) / max(1, args.steps)}
        else:
            collective = {"kind": "none (1 replica)"}
        kind = "bf16" if w.dtype == "bf16" else "tf32"
        peak, peak_src = self.peaks[kind], self.peak_src[kind]
        achieved = (gemm_fl.value / 1e12) / (gemm_ms.value / 1e3) if gemm_ms.value > 0 else 0.0
        traffic, traffic_src = load_traffic(name)
        base = None
        if not args.no_cpu_baseline:
            base = cpu_baseline(w, max_seconds=10.0 if name == "mlp" else 6.0)
        n_samples = w.batch * world * args.steps
        rec = {
            "metric": METRIC, "value": n_samples / (ms_res / 1e3), "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": ("bf16 graph; GEMMs on kind::f16 (bf16) tensor cores, fp32 accumulate"
                      if w.dtype == "bf16" else
                      "f32 graph; GEMMs / convolutions on TF32 tensor cores, fp32 accumulate"),
            "data": "synthetic",
            "config": {"workload": w.describe, "global_batch": w.batch * world,
                       "parallelism": "dp%d" % world,
                       "l2": "no flush: %d launches per step stream distinct operands; per-step "
                             "working set exceeds the 126 MB L2 for the MLPs (~193 MB fp32), LeNet's "
                             "(~75 MB activations + patches) is re-produced every step"
                             % (launches // max(1, args.steps)),
                       "loss_resident": loss_res, "loss_e2e": loss_e2e,
                       "host_enqueue_us_per_step": host_enqueue_us,
                       "ms_per_step_median_of_5_chunks": statistics.median(chunks) if chunks else None,
                       "collective": collective},
            "clocks": clocks,
            "e2e": {"value": n_samples / (ms_e2e / 1e3), "unit": "samples/s",
                    "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h,
                    "how": ("Session.stage() of step i+1's pinned inputs (copy stream) before "
                            "Session.run of step i; loss fetched to the host every step"),
                    "unpipelined_value": n_samples / (ms_sync / 1e3),
                    "unpipelined_ms_per_step": ms_sync / args.steps},
            "gpu_launches": launches,
            "parity": parity,
            "roofline": {"kernel": "tcgen05 GEMM / implicit-GEMM convolution kernels (kind::%s)"
                                   % ("f16 bf16" if w.dtype == "bf16" else "tf32"),
                         "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak if peak else None, "traffic": traffic,
                         "traffic_source": traffic_src,
                         "peak_source": peak_src, "launches_timed": int(gemm_n.value),
                         "us_per_launch": 1e3 * gemm_ms.value / max(1, gemm_n.value),
                         "empty_event_pair_us": event_pair_us,
                         "achieved_net_of_event_pair": ((gemm_fl.value / 1e12) /
                                                        max(1e-9, gemm_ms.value / 1e3 -
                                                            gemm_n.value * event_pair_us / 1e6)),
                         "flops_per_launch": (gemm_fl.value / max(1, gemm_n.value)),
                         "share_of_step": (gemm_ms.value / prof_steps) / (ms_res / args.steps),
                         "step_tflops": w.flops_per_step * world * args.steps / (ms_res / 1e3) / 1e12},
            "cpu_baseline": base,
        }
        return rec


def dump_outputs(directory, arrays):
    """DIR/<name>.npy for every array, float32; refuses to write more than DUMP_LIMIT_BYTES."""
    arrays = {n: np.ascontiguousarray(a, np.float32) for n, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d byte limit"
                         % (total, DUMP_LIMIT_BYTES))
    os.makedirs(directory, exist_ok=True)
    for n, a in arrays.items():
        np.save(os.path.join(directory, n + ".npy"), a)


def run_b200(args):
    # Libraries we load (NCCL's version banner) write to fd 1; the contract is ONE JSON line on
    # stdout, so everything else goes to stderr and the line is written to the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    b = Bench(args)
    records = {}
    for name in args.workloads:
        records[name] = b.run_workload(name)
    if b.world > 1:
        import torch.distributed as dist
        dist.barrier()
    if b.rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, b.outputs)
        head = args.workloads[0]
        line = dict(records[head])
        line["workloads"] = {n: r for n, r in records.items() if n != head}
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if b.world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--workloads", default=",".join(ALL_WORKLOADS),
                    help="comma list; the first is the line's top-level record (default: mlp = "
                         "BASELINE configs[1], then lenet = configs[2], mlp_bf16 = configs[3])")
    ap.add_argument("--workload", default=None, help="shorthand for --workloads <one>")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and trained variables of each workload's last timed step "
                         "to DIR/<workload>_<name>.npy (float32)")
    args = ap.parse_args()
    args.workloads = [args.workload] if args.workload else [s for s in args.workloads.split(",") if s]
    for n in args.workloads:
        if n not in ALL_WORKLOADS:
            raise SystemExit("unknown workload %r (choose from %s)" % (n, ALL_WORKLOADS))
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs dumps the GPU arm; it has no meaning with --impl reference")
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
