#!/usr/bin/env python
"""bench.py -- batched path-QP solves/s on B200 (BASELINE.json metric), one rank per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--formulation KP|K|KPC]

A "step" is one pass of the hot path (QP assembly -> ADMM solve -> state extraction) over one batch of
synthetic corridor paths.  The default workload is BASELINE config 2 (1024 paths x 100 stations per GPU);
--config selects configs 3, 4, 5 at their named sizes (path_optimizer_b200/workloads.py).  Weak scaling:
every rank solves its own shard; at N > 1 each step ends with ONE NCCL all-gather of the solved Frenet
states.  Rank 0 prints one JSON line.

  value        solves/s with the inputs already resident in HBM (pqp_solve_batch_device, or
               pqp_solve_batch_device_classes for the mixed-length config 5), CUDA events on the launching
               stream, L2 flushed between timed steps, max over ranks.
  e2e          the same metric through the host-buffer C-ABI call (pqp_solve_batch): pinned host inputs,
               H2D + kernels + D2H inside the call, timed by host wall clock around the call
               (time.perf_counter; the library's own event spans are reported beside it as a breakdown).
  roofline     dominant kernel's algorithmic HBM bytes (SURVEY 8d: 52 N + 32 B per solve) / its average
               launch time against the measured HBM copy bandwidth, plus the second figure SURVEY 8d
               mandates: the per-iteration working set W_iter = 944 N B streamed at the measured
               iteration rate, labelled ON-CHIP (the ADMM state never leaves the SM).
  cpu_baseline the CPU oracle (restatement of the reference's assembly + OSQP recurrence, oracle/) on the
               host's physical cores, bounded sample, min / median of repetitions.
  extras       default run only (config 2, one GPU): short measurements of configs 3, 4 and 5 at their
               named per-GPU sizes (QP-only, and config 3 through the chained planner iteration too).

--impl reference times the CPU oracle on the host cores (the reference's own OSQP-based binary cannot be
built here: no Eigen / OSQP / osqp-eigen / glog / gflags in the image), same `config` object, same JSON
contract; each step is a bounded sample of the workload (stated in cpu_baseline.sample).

--dump-outputs DIR writes what the timed call returned in its last timed step (rank 0's shard) as float64
.npy files, so that two builds run with the same arguments can be compared output for output (the inputs
are seeded): status.npy, iters.npy (per path), paths.npy (the path indices the per-station files cover),
states.npy (rows x 7: x, y, z, k, s, v, a) and frenet.npy (rows x 3).  The per-station files cover every
path, or a fixed seeded sample of whole paths where that would exceed 64 MB in all.
"""
import argparse
import ctypes as C
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

from path_optimizer_b200 import synth, workloads  # noqa: E402
from path_optimizer_b200.abi import BOUNDS_DTYPE, STATE_DTYPE, Stats  # noqa: E402

METRIC = "path_qp_solves_per_sec"
UNIT = "solves/s"
CPU_SAMPLE_PATHS = 1024      # paths per CPU step for configs whose shard is larger than that
DUMP_LIMIT_BYTES = 64 * 1000 * 1000
DUMP_SEED = 0


def io_bytes_per_solve(n):
    """SURVEY.md 8(d) contract figure B_io(N) = 52 N + 32 (fp32-packed compulsory I/O)."""
    return 52 * n + 32


def w_iter_bytes(n):
    """SURVEY.md 8(d) per-iteration working set W_iter(N) = 236 N floats = 944 N bytes."""
    return 944 * n


def dump_outputs(out_dir, n_points, states, frenet, status, iters):
    """Writes one step's outputs of a batch as float64 .npy files under `out_dir` (see --dump-outputs)."""
    n_points = np.asarray(n_points, dtype=np.int64)
    B = len(n_points)
    off = np.concatenate([[0], np.cumsum(n_points)])
    row_bytes = (len(STATE_DTYPE.names) + 3) * 8
    max_rows = (DUMP_LIMIT_BYTES - 3 * 8 * B - 5 * 128) // row_bytes    # 5 files, 128-byte .npy headers
    if off[-1] <= max_rows:
        paths = np.arange(B)
    else:
        order = np.random.default_rng(DUMP_SEED).permutation(B)
        paths = np.sort(order[np.cumsum(n_points[order]) <= max_rows])
    rows = np.concatenate([np.arange(off[p], off[p + 1]) for p in paths])
    states = np.asarray(states)[rows]
    out = {"status": status, "iters": iters, "paths": paths,
           "states": np.stack([states[f] for f in STATE_DTYPE.names], axis=1),
           "frenet": np.asarray(frenet).reshape(-1, 3)[rows]}
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(arr, dtype=np.float64))


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML in-process, nvidia-smi fallback)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _nvml_handle(self):
        """NVML handle of CUDA device `index` (matched by UUID: CUDA_VISIBLE_DEVICES may reorder), or None."""
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(self.index).uuid)
                if not uuid.startswith("GPU-"):
                    uuid = "GPU-" + uuid
                return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)
        except Exception:
            return None, None

    def _run(self):
        nv, hdl = self._nvml_handle()
        if hdl is not None:
            bits = {0x8: 2, 0x40: 3, 0x20: 4, 0x4: 5}    # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap -> column
            try:
                mx = nv.nvmlDeviceGetMaxClockInfo(hdl, nv.NVML_CLOCK_SM)
                while not self._stop.is_set():
                    sm = nv.nvmlDeviceGetClockInfo(hdl, nv.NVML_CLOCK_SM)
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(hdl)
                    except Exception:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(hdl)
                    row = [str(sm), str(mx), "Not Active", "Not Active", "Not Active", "Not Active"]
                    for bit, col in bits.items():
                        if r & bit:
                            row[col] = "Active"
                    self.samples.append(row)
                    self._stop.wait(0.005)
                return
            except Exception:
                pass   # fall through to the command-line poller
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[2 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------------
# CPU arm
# ----------------------------------------------------------------------------------------------------

def host_cores():
    """(threads usable by this process, physical cores among them).  The CPU arm runs one thread per physical
    core: the oracle's sparse triangular solves are latency bound and gain nothing from the second hyper-thread,
    while oversubscribing a cgroup-limited container costs a lot (round 1: 3.3 k..15 k solves/s for the same batch)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except Exception:
        cpus = list(range(os.cpu_count() or 1))
    cores = set()
    for c in cpus:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                cores.add(f.read().strip())
        except Exception:
            cores.add(str(c))
    n_log, n_phys = len(cpus), max(1, len(cores))
    quota = None
    try:   # cgroup v2 CPU quota
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, p = f.read().split()
            if q != "max":
                quota = max(1, int(float(q) / float(p)))
    except Exception:
        pass
    if quota:
        n_log, n_phys = min(n_log, quota), min(n_phys, quota)
    return n_log, n_phys


def oracle_bounds_fn(oracle, params):
    field = synth.disc_field_map()

    def fn(cand):
        r = oracle.update_bounds(params, field, cand, mode=1)
        return r["bounds"], r["n_valid"]
    return fn


def cpu_solve(oracle, params, formulation, batch, threads):
    """One CPU-arm solve of `batch` with the formulation's inputs (KPC: limits from the synthetic speed profile)."""
    form = workloads.FORMULATION_IDS[formulation]
    kw = {}
    if formulation == "KPC":
        ref = batch["ref"].copy()
        ref["v"], ref["a"] = workloads.speed_profile(len(ref))
        batch = dict(batch, ref=ref)
        kw["max_k"], kw["max_kp"] = oracle.update_limits(params, ref)
    return oracle.solve_batch(params, form, batch, threads=threads, **kw)


def cpu_sample(config, oracle, params):
    """The bounded per-step sample of a config for the CPU arm + a description of it."""
    c = workloads.CONFIGS[config]
    if c["paths_per_gpu"] <= CPU_SAMPLE_PATHS:
        return workloads.build(config), f"the whole {c['paths_per_gpu']}-path shard of rank 0 per step"
    if config == 3:
        batch = workloads.build(3, paths=CPU_SAMPLE_PATHS, bounds_fn=oracle_bounds_fn(oracle, params))
        return batch, f"the first {CPU_SAMPLE_PATHS} unblocked paths of rank 0's config-3 shard per step (bounds by the oracle's clearance stage, untimed)"
    if config == 5:
        full = workloads.build(5)
        idx = np.arange(0, len(full["n_points"]), len(full["n_points"]) // CPU_SAMPLE_PATHS)[:CPU_SAMPLE_PATHS]
        return synth.take_paths(full, idx), f"every {len(full['n_points']) // CPU_SAMPLE_PATHS}th path of rank 0's {len(full['n_points'])}-path shard ({CPU_SAMPLE_PATHS} paths, same length distribution) per step"
    return workloads.build(config, paths=CPU_SAMPLE_PATHS), f"the first {CPU_SAMPLE_PATHS} paths of rank 0's {c['paths_per_gpu']}-path shard per step"


def run_reference(args, rank, world):
    """CPU arm: the oracle (port of the reference's algorithm) on the host's physical cores."""
    if rank != 0:
        return
    from oracle import oracle
    params = oracle.default_params()
    n_log, n_phys = host_cores()
    threads = args.cpu_threads or n_phys
    batch, sample_text = cpu_sample(args.config, oracle, params)
    B = len(batch["n_points"])
    F = args.formulation
    cpu_solve(oracle, params, F, synth.slice_batch(batch, 0, min(B, 8)), 1)   # builds the symbolic cache
    for _ in range(args.warmup):
        cpu_solve(oracle, params, F, synth.slice_batch(batch, 0, min(B, 4 * threads)), threads)
    step_s = []
    solved = 0
    for _ in range(args.steps):
        r = cpu_solve(oracle, params, F, batch, threads)
        step_s.append(r["seconds"])
        solved += int((r["status"] == 1).sum())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, batch["n_points"], r["states"], r["frenet"], r["status"], r["iters"])
    secs = sum(step_s)
    value = B * args.steps / secs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workloads.describe(args.config, args.gpus, args.formulation),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "hardware_threads_visible": n_log, "physical_cores_visible": n_phys,
                         "sample": sample_text, "paths_per_step": B,
                         "best_step_value": B / min(step_s), "median_step_value": B / statistics.median(step_s),
                         "note": "fp64 C restatement of the reference's assembly + OSQP recurrence (oracle/): the reference's "
                                 "own binary needs Eigen/OSQP/osqp-eigen, absent from this image; one thread per physical core, "
                                 "paths handed out dynamically, per-thread scratch arena"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "solved_fraction": solved / (B * args.steps), "gpu_launches": 0,
        "iters_per_solve_mean": float(r["iters"].mean()),
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------

class GpuWorkload:
    """One config's shard resident on one GPU + the two timed calls (device-resident, host-buffer)."""

    def __init__(self, config, rank, world, local_rank, torch, join_comm=True, formulation="KP"):
        from path_optimizer_b200 import _lib, planner
        self.torch = torch
        self.formulation = formulation
        self.form = workloads.FORMULATION_IDS[formulation]
        self.config, self.rank, self.world = config, rank, world
        self.L = _lib.load()
        self._lib = _lib
        self.dev = torch.device("cuda", local_rank)
        c = workloads.CONFIGS[config]
        self.field = None
        if config == 3:
            self.field = synth.disc_field_map()
            pl = planner.PathPlanner(device=local_rank, max_batch=c["paths_per_gpu"] + 1024,
                                     max_total_points=(c["paths_per_gpu"] + 1024) * 200)
            pl.set_map(self.field)

            def fn(cand):
                r = pl.update_bounds(cand)
                return r["bounds"], r["n_valid"]
            self.batch = workloads.build(3, rank, world, bounds_fn=fn)
            pl.close()
        else:
            self.batch = workloads.build(config, rank, world)
        b = self.batch
        self.B = len(b["n_points"])
        self.total = int(b["offsets"][-1])
        self.nmax = int(b["n_points"].max())
        self.solver = planner.PathPlanner(device=local_rank, max_batch=self.B, max_total_points=self.total)
        self.mk = self.mkp = None
        if formulation == "KPC":
            b["ref"]["v"], b["ref"]["a"] = workloads.speed_profile(self.total)
            self.mk, self.mkp = planner.update_limits(self.solver.params, b["ref"])
        off = b["offsets"]
        self.keep = np.array([self.L.pqp_keep_control_steps(0, np.ascontiguousarray(b["ref"][off[i]:off[i + 1]]).ctypes.data_as(C.c_void_p),
                                                            int(b["n_points"][i])) for i in range(self.B)], dtype=np.int32)
        self.uniform = bool((b["n_points"] == b["n_points"][0]).all() and (self.keep == self.keep[0]).all())

        def dev_bytes(arr):
            t = torch.from_numpy(np.frombuffer(np.ascontiguousarray(arr).tobytes(), dtype=np.uint8).copy())
            return t.to(self.dev)
        self.d = dict(n=dev_bytes(b["n_points"]), off=dev_bytes(b["offsets"]), ref=dev_bytes(b["ref"]),
                      bounds=dev_bytes(b["bounds"]), x0=dev_bytes(b["x0"]), end=dev_bytes(b["end_heading"]))
        self.d_mk = self.d_mkp = None
        if self.mk is not None:
            self._limits_dev = (dev_bytes(self.mk), dev_bytes(self.mkp))     # keep the device copies alive
            self.d_mk, self.d_mkp = self._limits_dev[0].data_ptr(), self._limits_dev[1].data_ptr()
        self.d_out = torch.zeros(self.total * STATE_DTYPE.itemsize, dtype=torch.uint8, device=self.dev)
        self.d_status = torch.zeros(self.B, dtype=torch.int32, device=self.dev)
        self.d_iters = torch.zeros(self.B, dtype=torch.int32, device=self.dev)
        # the all-gather needs equal counts per rank: pad the Frenet buffer to the largest shard
        self.gather_rows = self.total
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([self.total], dtype=torch.int64, device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            self.gather_rows = int(t.item())
        self.d_frenet = torch.zeros(self.gather_rows * 3, dtype=torch.float64, device=self.dev)
        self.gathered = torch.zeros(world * self.gather_rows * 3, dtype=torch.float64, device=self.dev) if world > 1 else None
        self.comm = False
        if world > 1 and join_comm:
            # the data-path collective is the library's own (pqp_allgather: NCCL inside libpqp.so); torch.distributed only
            # carries the 128-byte communicator id and the timing reductions
            import torch.distributed as dist
            uid = (C.c_char * 128)()
            if rank == 0:
                assert self.L.pqp_nccl_unique_id(uid) == 0, self._lib.last_error()
            t = torch.tensor(list(bytes(uid)), dtype=torch.uint8, device=self.dev)
            dist.broadcast(t, 0)
            uid = (C.c_char * 128).from_buffer_copy(bytes(t.cpu().numpy().tobytes()))
            assert self.L.pqp_comm_init_rank(self.solver._h, world, rank, uid) == 0, self._lib.last_error()
            self.comm = True
        self.h_n = np.ascontiguousarray(b["n_points"], dtype=np.int32)
        self._pinned = None
        self.force_classes = False   # route a uniform batch through the per-class entry (it carries a launch order)

    # ---- device-resident call (asynchronous on `stream`)
    def solve_device(self, stream, stats=None):
        d = self.d
        sp = C.c_void_p(stream.cuda_stream)
        st = C.byref(stats) if stats is not None else None
        if self.uniform and not self.force_classes:
            k = int(self.keep[0])
            rc = self.L.pqp_solve_batch_device(self.solver._h, self.form, self.B, self.total, self.nmax, k, k, d["n"].data_ptr(),
                                               d["off"].data_ptr(), d["ref"].data_ptr(), d["bounds"].data_ptr(),
                                               d["x0"].data_ptr(), d["end"].data_ptr(), self.d_mk, self.d_mkp, self.d_out.data_ptr(),
                                               self.d_frenet.data_ptr(), self.d_status.data_ptr(), self.d_iters.data_ptr(), sp, st)
        else:
            rc = self.L.pqp_solve_batch_device_classes(self.solver._h, self.form, self.B, self.total, self.h_n.ctypes.data_as(C.c_void_p),
                                                       self.keep.ctypes.data_as(C.c_void_p), d["n"].data_ptr(), d["off"].data_ptr(),
                                                       d["ref"].data_ptr(), d["bounds"].data_ptr(), d["x0"].data_ptr(),
                                                       d["end"].data_ptr(), self.d_mk, self.d_mkp, self.d_out.data_ptr(),
                                                       self.d_frenet.data_ptr(), self.d_status.data_ptr(),
                                                       self.d_iters.data_ptr(), sp, st)
        assert rc == 0, self._lib.last_error()

    def gather(self, stream=None):
        if self.world > 1:
            if self.comm:
                sp = C.c_void_p(stream.cuda_stream) if stream is not None else None
                rc = self.L.pqp_allgather(self.solver._h, self.d_frenet.data_ptr(), self.gathered.data_ptr(),
                                          self.gather_rows * 3, sp)
                assert rc == 0, self._lib.last_error()
            else:
                import torch.distributed as dist
                dist.all_gather_into_tensor(self.gathered, self.d_frenet)

    # ---- host-buffer call (synchronous)
    def _pin(self):
        torch, b = self.torch, self.batch
        pin = lambda a: torch.from_numpy(np.frombuffer(np.ascontiguousarray(a).tobytes(), dtype=np.uint8).copy()).pin_memory()  # noqa: E731
        self._pinned = dict(ref=pin(b["ref"]), bounds=pin(b["bounds"]), x0=pin(b["x0"]), end=pin(b["end_heading"]),
                            n=pin(b["n_points"]),
                            mk=pin(self.mk) if self.mk is not None else None, mkp=pin(self.mkp) if self.mkp is not None else None,
                            out=torch.zeros(self.total * STATE_DTYPE.itemsize, dtype=torch.uint8).pin_memory(),
                            frenet=torch.zeros(self.total * 3, dtype=torch.float64).pin_memory(),
                            status=torch.zeros(self.B, dtype=torch.int32).pin_memory(),
                            iters=torch.zeros(self.B, dtype=torch.int32).pin_memory())

    def solve_host(self, stats):
        if self._pinned is None:
            self._pin()
        p = self._pinned
        rc = self.L.pqp_solve_batch(self.solver._h, self.form, self.B, p["n"].data_ptr(), p["ref"].data_ptr(), p["bounds"].data_ptr(),
                                    p["x0"].data_ptr(), p["end"].data_ptr(), p["mk"].data_ptr() if p["mk"] is not None else None,
                                    p["mkp"].data_ptr() if p["mkp"] is not None else None, p["out"].data_ptr(),
                                    p["frenet"].data_ptr(), p["status"].data_ptr(), p["iters"].data_ptr(), C.byref(stats))
        assert rc == 0, self._lib.last_error()

    def gather_from(self, other):
        """A gather() for `other` (a workload without a communicator of its own) through this workload's communicator."""
        def g(stream=None):
            sp = C.c_void_p(stream.cuda_stream) if stream is not None else None
            rc = self.L.pqp_allgather(self.solver._h, other.d_frenet.data_ptr(), self.gathered.data_ptr(), self.gather_rows * 3, sp)
            assert rc == 0, self._lib.last_error()
        return g

    def class_mix(self):
        """{kernel name: paths} as the library selects classes for this shard."""
        mix = {}
        v, t, s = C.c_int(), C.c_int(), C.c_int64()
        if self.form != 0:
            for n in self.h_n:
                self.L.pqp_class_info_form(self.form, int(n), 1, 0, C.byref(v), C.byref(t), C.byref(s))
                name = self.L.pqp_class_name(v.value).decode()
                mix[name] = mix.get(name, 0) + 1
            return mix
        if self.uniform:
            self.L.pqp_device_class_info(self.nmax, int(self.keep[0]), int(self.keep[0]), 0, C.byref(v), C.byref(t), C.byref(s))
            return {self.L.pqp_class_name(v.value).decode(): self.B}
        for n, k in zip(self.h_n, self.keep):
            self.L.pqp_class_info(int(n), int(k), 0, C.byref(v), C.byref(t), C.byref(s))
            name = self.L.pqp_class_name(v.value).decode()
            mix[name] = mix.get(name, 0) + 1
        return mix

    def close(self):
        self.solver.close()


def time_workload(w, torch, steps, warmup, flush, stream, barrier, with_e2e=True):
    """Device-resident and host-buffer timings of one workload on this rank (not yet reduced over ranks)."""
    st = Stats()
    w.solve_device(stream, st)           # synchronising call with stats: launches per step
    launches = int(st.kernel_launches)
    for _ in range(max(0, warmup - 1)):
        w.solve_device(stream)
        w.gather(stream)
    barrier()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        flush.fill_(k & 0xFF)            # L2 flush between timed steps (outside the events)
        ev[k][0].record(stream)
        w.solve_device(stream)
        ev[k][1].record(stream)
        w.gather(stream)
        ev[k][2].record(stream)
    barrier()
    wall = time.perf_counter() - t0
    solve_ms = [a.elapsed_time(b) for a, b, _ in ev]
    gather_ms = [b.elapsed_time(c) for _, b, c in ev]
    step_ms = [a.elapsed_time(c) for a, _, c in ev]
    res = dict(launches_per_step=launches, dev_ms=sum(step_ms), solve_ms=sum(solve_ms), gather_ms=sum(gather_ms),
               wall_ms=wall * 1e3, status=w.d_status.cpu().numpy(), iters=w.d_iters.cpu().numpy())
    if with_e2e:
        for _ in range(warmup):
            w.solve_host(st)
        barrier()
        e2e_wall = e2e_span = kern = 0.0
        for _ in range(steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            w.solve_host(st)             # synchronous: returns when the results are in the caller's host buffers
            e2e_wall += time.perf_counter() - t1
            e2e_span += st.h2d_ms + st.kernel_ms + st.d2h_ms
            kern += st.kernel_ms
        barrier()
        res.update(e2e_ms=e2e_wall * 1e3, e2e_span_ms=e2e_span, e2e_kernel_ms=kern, h2d=int(st.h2d_bytes), d2h=int(st.d2h_bytes),
                   e2e_launches=int(st.kernel_launches))
    return res


def profile_units():
    """Measured unit utilisations of the dominant kernel from the committed ncu capture (NOT this run)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.Stream(device=dev)  # non-default: the ABI treats a NULL stream as 'the handle's own'
    torch.cuda.set_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    w = GpuWorkload(args.config, rank, world, local_rank, torch, formulation=args.formulation)
    sampler = ClockSampler(local_rank)
    # warm-up of both arms happens inside time_workload; the clock sampler covers the timed regions
    if rank == 0:
        sampler.start()
    r = time_workload(w, torch, args.steps, args.warmup, flush, stream, barrier)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the device buffers still hold the last timed step: the host-buffer arm writes its own pinned buffers
        dump_outputs(args.dump_outputs, w.h_n, w.d_out.cpu().numpy().view(STATE_DTYPE), w.d_frenet[:w.total * 3].cpu().numpy(),
                     r["status"], r["iters"])

    # ---- reduce over ranks: step time = max over ranks; per-rank breakdown gathered as it is
    t = torch.tensor([r["dev_ms"], r["e2e_ms"], r["wall_ms"]], dtype=torch.float64, device=dev)
    per_rank = torch.tensor([r["solve_ms"] / args.steps, r["gather_ms"] / args.steps, float(r["iters"].mean()),
                             float(r["iters"].max()), float(w.B), float(w.total)], dtype=torch.float64, device=dev)
    all_ranks = per_rank.clone().unsqueeze(0)
    paths_total = torch.tensor([w.B, int((r["status"] == 1).sum())], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        all_ranks = torch.zeros(world, per_rank.numel(), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(all_ranks.view(-1), per_rank)
        dist.all_reduce(paths_total)
    dev_ms, e2e_ms, wall_ms = [float(x) for x in t.cpu()]
    all_ranks = all_ranks.cpu().numpy()
    n_paths, n_solved = [int(x) for x in paths_total.cpu()]

    control = None
    if world > 1 and args.config in (2, 4):
        # control run: every rank solves shard 0 (identical work) -- separates data-dependent tails from the collective
        w0 = GpuWorkload(args.config, 0, 1, local_rank, torch, formulation=args.formulation)
        w0.world, w0.gathered, w0.gather_rows = world, w.gathered, w.gather_rows
        w0.d_frenet = w.d_frenet
        w0.gather = w.gather_from(w0)   # the collective goes through the main workload's communicator
        rc_ = time_workload(w0, torch, max(3, args.steps // 4), 2, flush, stream, barrier, with_e2e=False)
        tc = torch.tensor([rc_["dev_ms"] / max(3, args.steps // 4)], dtype=torch.float64, device=dev)
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        control = {"what": "every rank solves rank 0's shard (identical work), all-gather as usual",
                   "ms_per_step": float(tc.item())}
        w0.close()

    if rank == 0:
        steps = args.steps
        value = n_paths * steps / (dev_ms * 1e-3)
        e2e_value = n_paths * steps / (e2e_ms * 1e-3)
        peak, peak_src = measured_peak_gbs()
        mix = w.class_mix()
        dominant = max(mix, key=lambda k: mix[k])
        mean_n = w.total / w.B
        launch_s = (r["solve_ms"] / steps) * 1e-3            # all of this rank's solve kernels of one step
        alg_bytes = sum(io_bytes_per_solve(int(n)) for n in w.h_n)
        achieved = alg_bytes / launch_s / 1e9
        iters_mean = float(r["iters"].mean())
        it_per_s = float(r["iters"].sum()) / launch_s
        prof = profile_units()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workloads.describe(args.config, world, args.formulation),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "ms_per_step": e2e_ms / steps, "timer": "host wall clock (time.perf_counter) around pqp_solve_batch, max over ranks",
                    "library_event_span_ms_per_step": r["e2e_span_ms"] / steps, "kernel_span_ms_per_step": r["e2e_kernel_ms"] / steps,
                    "kernel_launches_per_step": r["e2e_launches"]},
            "gpu_launches": r["launches_per_step"] * steps,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": prof.get("dram_bytes_per_launch") if args.config == 2 else None,
                         "traffic_source": prof.get("source", "profiles/traffic.json") + " (ncu --set full capture of the same kernel on the same batch; not measured in this run)" if args.config == 2 else None,
                         "peak_source": peak_src, "kernel": dominant, "kernel_classes": mix,
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "on_chip": {"what": "SURVEY 8d second figure: per-iteration working set W_iter = 944 N bytes streamed at the measured "
                                             "ADMM iteration rate; the state is SM-resident, so this is ON-CHIP traffic-equivalent, NOT HBM",
                                     "w_iter_bytes": int(w_iter_bytes(mean_n)), "iterations_per_s": it_per_s,
                                     "equivalent_GBps": it_per_s * w_iter_bytes(mean_n) / 1e9,
                                     "vs_hbm_peak": it_per_s * w_iter_bytes(mean_n) / 1e9 / peak},
                         "units": prof.get("units"),
                         "note": "state is SM-resident by design: compulsory HBM traffic is I/O only (SURVEY 8d); the kernel is bound by "
                                 "dependent-issue latency and the shared-memory pipe, see profiles/"},
            "clocks": clocks, "solved_fraction": n_solved / n_paths, "wall_ms_per_step": wall_ms / steps,
            "iters_per_solve_mean": iters_mean, "iters_per_solve_max": int(r["iters"].max()),
            "per_rank": {"solve_kernel_ms": [float(x) for x in all_ranks[:, 0]], "allgather_ms": [float(x) for x in all_ranks[:, 1]],
                         "iters_mean": [float(x) for x in all_ranks[:, 2]], "iters_max": [float(x) for x in all_ranks[:, 3]],
                         "paths": [int(x) for x in all_ranks[:, 4]], "stations": [int(x) for x in all_ranks[:, 5]],
                         "note": "CUDA events on each rank's stream: solve kernels, then the NCCL all-gather (which also waits for the slowest rank)"},
        }
        if control:
            line["scaling_control"] = control
        if world == 1:
            line["cpu_baseline"] = cpu_baseline(args)
            if args.config == 2 and args.formulation == "KP" and not args.no_extras:
                line["extras"] = {"order_hint": extras_order_hint(w, torch, 5, 3, flush, stream, barrier),
                                  "configs": extras_configs(torch, local_rank, flush, stream, barrier),
                                  "formulations": extras_formulations(local_rank)}
        print(json.dumps(line), flush=True)
    w.close()
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline(args):
    """Bounded CPU sample on rank 0: the oracle on the physical cores (3 repetitions), then on one core."""
    from oracle import oracle
    params = oracle.default_params()
    n_log, n_phys = host_cores()
    threads = args.cpu_threads or n_phys
    batch, sample_text = cpu_sample(args.config, oracle, params)
    B = len(batch["n_points"])
    F = args.formulation
    cpu_solve(oracle, params, F, synth.slice_batch(batch, 0, 8), 1)
    cpu_solve(oracle, params, F, synth.slice_batch(batch, 0, min(B, 4 * threads)), threads)
    secs = [cpu_solve(oracle, params, F, batch, threads)["seconds"] for _ in range(3)]
    one = synth.slice_batch(batch, 0, 32)
    r1 = cpu_solve(oracle, params, F, one, 1)
    return {"value": B / statistics.median(secs), "unit": UNIT, "cores": threads, "hardware_threads_visible": n_log,
            "physical_cores_visible": n_phys, "kind": "port",
            "sample": sample_text.replace("per step", "per repetition") + "; 3 repetitions, median",
            "best_value": B / min(secs), "single_thread_value": 32 / r1["seconds"],
            "reference_logged_ms_per_qp": "7.09-12.79 ms at N=188-244 (BASELINE.md)"}


def extras_configs(torch, local_rank, flush, stream, barrier):
    """Configs 3, 4, 5 at their named per-GPU sizes, a few steps each (context for the default line)."""
    out = {}
    for cfg in (3, 4, 5):
        try:
            w = GpuWorkload(cfg, 0, 1, local_rank, torch)
            r = time_workload(w, torch, 3, 2, flush, stream, barrier)
            stations = float(r["iters"].astype(np.float64) @ w.h_n.astype(np.float64))
            e = {"workload": workloads.CONFIGS[cfg]["text"], "paths": w.B, "stations": w.total,
                 "solves_per_sec": w.B * 3 / (r["dev_ms"] * 1e-3), "ms_per_step": r["dev_ms"] / 3,
                 "e2e_solves_per_sec": w.B * 3 / (r["e2e_ms"] * 1e-3), "e2e_ms_per_step": r["e2e_ms"] / 3,
                 "iters_per_solve_mean": float(r["iters"].mean()), "iters_per_solve_max": int(r["iters"].max()),
                 "solved_fraction": float((r["status"] == 1).mean()),
                 "ns_per_station_iteration": (r["solve_ms"] / 3) * 1e6 / stations,
                 "kernel_classes": w.class_mix(), "kernel_launches_per_step": r["launches_per_step"]}
            if cfg == 3:
                e["plan_chain"] = plan_chain(w, local_rank)
            out[str(cfg)] = e
            w.close()
            del w
            torch.cuda.empty_cache()
        except Exception as ex:  # context only: never fail the bench line on it
            out[str(cfg)] = {"error": repr(ex)[:300]}
    return out


def extras_order_hint(w, torch, steps, warmup, flush, stream, barrier):
    """The launch tail, measured: the same device-resident batch through the per-class entry point in index order and
    with pqp_set_order_hint(iterations of a previous solve) = longest expected work first.  Context only: the headline
    `value` never uses a hint (a bench that repeats one batch would make the hint exact)."""
    try:
        w.force_classes = True
        plain = time_workload(w, torch, steps, warmup, flush, stream, barrier, with_e2e=False)
        it = np.ascontiguousarray(plain["iters"], dtype=np.int32)
        assert w.L.pqp_set_order_hint(w.solver._h, w.B, it.ctypes.data_as(C.c_void_p)) == 0
        hinted = time_workload(w, torch, steps, warmup, flush, stream, barrier, with_e2e=False)
        w.L.pqp_set_order_hint(w.solver._h, 0, None)
        w.force_classes = False
        same = bool(np.array_equal(plain["iters"], hinted["iters"]) and np.array_equal(plain["status"], hinted["status"]))
        return {"what": "config-2 shard through pqp_solve_batch_device_classes: launch order longest path first (= index order "
                        "here) vs pqp_set_order_hint with the iteration counts of a previous solve of the same batch (an exact "
                        "predictor: upper bound of what an ordering can recover)",
                "ms_per_step_index_order": plain["solve_ms"] / steps, "ms_per_step_hinted": hinted["solve_ms"] / steps,
                "solves_per_sec_hinted": w.B * steps / (hinted["solve_ms"] * 1e-3), "same_results": same}
    except Exception as ex:
        w.force_classes = False
        return {"error": repr(ex)[:300]}


def extras_formulations(device, reps=3):
    """The other two type strings of OsqpSolver::create on the config-2 shape (1024 x 100 curved corridors, host buffers,
    host wall clock): "KPC" and "K" run on thread-per-station kernels of their own, assembled in the kernel."""
    out = {}
    try:
        from path_optimizer_b200 import planner
        b = synth.curvy_corridors(1024, 100)
        total = 1024 * 100
        ref = b["ref"].copy()
        ref["v"] = 4.0 + 3.0 * np.sin(np.arange(total) * 0.05)
        ref["a"] = 0.5 * np.cos(np.arange(total) * 0.05)
        s = planner.PathPlanner(device=device, max_batch=1024, max_total_points=total)
        mk, mkp = planner.update_limits(s.params, ref)
        for form, kw in (("KP", {}), ("KPC", dict(max_k=mk, max_kp=mkp)), ("K", {})):
            s.solve(b, form, **kw)
            best = None
            for _ in range(reps):
                t0 = time.perf_counter()
                r = s.solve(b, form, **kw)
                ms = (time.perf_counter() - t0) * 1e3
                best = ms if best is None else min(best, ms)
            out[form] = {"workload": "1024 paths x 100 stations, curved corridors, host buffers", "ms_per_call": best,
                         "solves_per_sec": 1024 / (best * 1e-3), "kernel_span_ms": r["stats"].kernel_ms,
                         "kernel_launches": int(r["stats"].kernel_launches), "iters_per_solve_mean": float(r["iters"].mean()),
                         "solved_fraction": float((r["status"] == 1).mean())}
        s.close()
    except Exception as ex:
        out["error"] = repr(ex)[:300]
    return out


def plan_chain(w, device, reps=3):
    """Config 3 through the chained planner iteration (pqp_plan_batch: clearance bounds on the distance map ->
    KP QP -> collision-checked raw output = solveWithoutSmoothing, path_optimizer.cpp:87-117), host buffers."""
    from path_optimizer_b200 import planner
    pl = planner.PathPlanner(device=device, max_batch=w.B, max_total_points=w.total)
    pl.set_map(w.field)
    torch = w.torch
    # pinned host buffers, as the e2e arm uses: the reference states in, the output path states out
    b = dict(w.batch)
    ref_pin = torch.from_numpy(np.frombuffer(np.ascontiguousarray(b["ref"]).tobytes(), dtype=np.uint8).copy()).pin_memory()
    b["ref"] = np.frombuffer(ref_pin.numpy(), dtype=STATE_DTYPE)
    out_pin = torch.zeros(w.total * STATE_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
    outs = {"states": np.frombuffer(out_pin.numpy(), dtype=STATE_DTYPE)}
    pl.plan(b, out=outs)
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        r = pl.plan(b, out=outs)
        ms = (time.perf_counter() - t0) * 1e3
        best = ms if best is None else min(best, ms)
    out = {"what": "updateBounds -> KP QP -> raw tail with collision check, pinned host buffers, host wall clock, best of 3",
           "ms_per_call": best, "planner_iterations_per_sec": w.B / (best * 1e-3),
           "library_event_span_ms": r["stats"].h2d_ms + r["stats"].kernel_ms + r["stats"].d2h_ms,
           "qp_solved": int(r["solved"].sum()), "ok": int(r["ok"].sum())}
    pl.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", type=int, choices=[2, 3, 4, 5], default=2)
    ap.add_argument("--formulation", choices=["KP", "K", "KPC"], default="KP",
                    help="type string of OsqpSolver::create to solve the config with (default KP: the BASELINE metric)")
    ap.add_argument("--cpu-threads", type=int, default=0, help="CPU arm thread count (default: physical cores)")
    ap.add_argument("--no-extras", action="store_true", help="skip the config 3/4/5 context measurements of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as .npy files under DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
