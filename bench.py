#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on B200: OSC control evaluations / second, batched UR5 6-DOF.

One "step" = one pass of the hot path (the fused OSC kernel: chain walk -> J, M, g, C dq -> solves -> u) over
one batch of B synthetic joint states per GPU (B = 65 536, fp64: the UR5 configuration of BASELINE.json,
configs[1], driven through OSC.generate with use_C so that {J, M, g, c_forces} are all on the path).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # our CUDA path (one JSON line on rank 0)
  python bench.py --impl reference [...]                         # the reference's CPU path on the host cores

Under torchrun (N > 1) every rank owns its own B states (weak scaling, no data-path collective in the timed step);
the optional all-gather of the control outputs is measured separately ("collective": NCCL vs the kernel's fused
peer-store epilogue), and BASELINE configs 4 and 5 are run at their stated multi-GPU scale ("configs").  Timing: CUDA events on the launching stream, barrier +
synchronize on both sides, max over ranks.  L2: the steps rotate over a ring of input/output buffer sets larger
than the 126 MB L2, so every step's inputs come from HBM.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)
sys.path.insert(0, ROOT)

METRIC = "OSC control evals/sec (batched UR5 6-DOF)"
UNIT = "evals/s"
B_PER_GPU = 65536
OSC_KW = dict(kp=10.0, ctrlr_dof=[True] * 6, use_C=True)  # 6 controlled DOF, gravity + Coriolis compensation
WORKLOAD = "ur5_osc_6dof_useC_fp64_B65536_per_gpu"


def synth(B, n, seed, dtype=np.float64):
    """seeded synthetic states as examples/timing_plots.py:18-20: q~U(0,2pi), dq~U(0,5), target~U(-1,1)"""
    rng = np.random.default_rng(seed)
    return (rng.uniform(0, 2 * np.pi, (B, n)).astype(dtype), rng.uniform(0, 5, (B, n)).astype(dtype),
            rng.uniform(-1, 1, (B, 6)).astype(dtype))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.

    Primary source: NVML in this process (the library nvidia-smi itself reads), polled every 2 ms by a thread — it has
    no start-up latency, so even a 50 ms timed region gets samples.  `nvidia-smi --query-gpu=... -lms 10` runs beside
    it as a second source (it needs ~100 ms to print its first line); the two are merged."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index, uuid=None):
        import threading

        self.sm, self.mx, self.reasons, self.src = [], [], set(), []
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self._stop = threading.Event()
        self._thread = None
        period = os.environ.get("ABRB_BENCH_CLOCK_MS", "10")  # tuning knob: "off" disables the sampler (A/B only)
        if period == "off":
            return
        try:
            import pynvml

            pynvml.nvmlInit()
            h = None
            if uuid:
                for cand in (f"GPU-{uuid}", str(uuid)):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                        break
                    except Exception:
                        h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons",
                                 getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons", None))
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)))

            def poll():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        if reasons_fn is not None:
                            mask = int(reasons_fn(h))
                            for bit, name in self.BITS.items():
                                if mask & bit:
                                    self.reasons.add(name)
                    except Exception:
                        pass
                    self._stop.wait(0.002)

            self._thread = threading.Thread(target=poll, daemon=True)
            self._thread.start()
            self.src.append("nvml")
        except Exception:
            self._thread = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                       period, "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": []}
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=1)
        if self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
            self.f.flush()
            self.f.seek(0)
            n_smi = 0
            for line in self.f.read().splitlines():
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    self.sm.append(float(c[1]))
                    self.mx.append(float(c[2]))
                    n_smi += 1
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
            if n_smi:
                self.src.append("nvidia-smi")
        if self.sm:
            out.update(sm_mhz=float(np.median(self.sm)), sm_max_mhz=float(max(self.mx)) if self.mx else None,
                       reasons=sorted(self.reasons), samples=len(self.sm), source=self.src)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ---------------------------------------------------------------------------------------------- reference arm
def ref_lib():
    p = os.path.join(ROOT, "oracle", "_ref", "libabrref_ur5.so")
    return C.CDLL(p) if os.path.exists(p) else None


class OscCfg(C.Structure):
    _fields_ = [("n", C.c_int), ("kp", C.c_double), ("ko", C.c_double), ("kv", C.c_double), ("use_vmax", C.c_int),
                ("vmax", C.c_double * 2), ("dof", C.c_int * 6), ("use_g", C.c_int), ("use_C", C.c_int),
                ("alg", C.c_int), ("damp_kv", C.c_double), ("use_rest", C.c_int), ("rest_kp", C.c_double),
                ("rest_kv", C.c_double), ("rest", C.c_double * 8), ("rest_mask", C.c_int * 8)]


def osc_cfg():
    c = OscCfg()
    c.n = 6
    c.kp = c.ko = OSC_KW["kp"]
    c.kv = float(np.sqrt(c.kp + c.ko))
    for r in range(6):
        c.dof[r] = 1
    c.use_g, c.use_C, c.alg, c.damp_kv = 1, 1, 0, -1.0
    return c


def cpu_reference_run(n_evals, repeats=3):
    """OSC evals/s of the reference's CPU path on all host cores.

    kind "reference": the reference's own SymPy-generated C for J/Tx/M/g/C/R (oracle/_ref, compiled from where the
    reference wrote it) + oracle/c/osc_cpu.c for the NumPy half, pthreads over states.
    kind "port" (fallback when oracle/_ref is absent): the NumPy oracle, one core."""
    q, dq, target = synth(n_evals, 6, 123)
    lib = ref_lib()
    if lib is not None:
        lib.ref_max_threads.restype = C.c_int
        online = int(lib.ref_max_threads())
        try:
            online = min(online, len(os.sched_getaffinity(0)))
        except AttributeError:
            pass
        cfg = osc_cfg()
        u = np.empty((n_evals, 6))

        def run(nthreads, count):
            a = (C.byref(cfg), q.ctypes.data_as(C.c_void_p), dq.ctypes.data_as(C.c_void_p),
                 target.ctypes.data_as(C.c_void_p), C.c_long(count), u.ctypes.data_as(C.c_void_p), C.c_int(nthreads))
            t0 = time.perf_counter()
            lib.ref_ur5_osc_batch(*a)
            return time.perf_counter() - t0

        # the box may expose more hardware threads than it lets us use: pick the best thread count on a short probe
        probe = min(n_evals, 400_000)
        run(online, probe)  # warm (page in)
        cands = sorted({c for c in (1, online // 8, online // 4, online // 2, online) if c >= 1})
        rates = {c: probe / min(run(c, probe) for _ in range(2)) for c in cands}
        cores = max(rates, key=rates.get)
        best = min(run(cores, n_evals) for _ in range(repeats))
        return dict(value=n_evals / best, unit=UNIT, cores=cores, kind="reference",
                    threads_probe={str(k): round(v) for k, v in rates.items()}, hw_threads_online=online,
                    sample=f"{n_evals} UR5 OSC evals (same controller, seeded states), best of {repeats}, "
                           "reference-generated C for J/Tx/M/g/C/R + C restatement of the NumPy half, pthreads"), u, (q, dq, target)
    from oracle import osc_oracle

    n_small = min(n_evals, 300)
    case = dict(arm="ur5", osc=OSC_KW)
    t0 = time.perf_counter()
    u, _ = osc_oracle.run_case(case, q[:n_small], dq[:n_small], target[:n_small])
    dt = time.perf_counter() - t0
    return dict(value=n_small / dt, unit=UNIT, cores=1, kind="port",
                sample=f"{n_small} UR5 OSC evals, NumPy oracle (oracle/_ref absent)"), u, (q[:n_small], dq[:n_small], target[:n_small])


AS_SHIPPED = os.path.join(ROOT, "baseline", "_ref")


def as_shipped_worker(n):
    """Runs INSIDE the reference's environment (PYTHONPATH=baseline/_ref, HOME=baseline/_ref/home): the stock loop of
    /root/reference/examples/timing_plots.py:14-28 — `for i: ctrlr.generate(q[i], dq[i], target[i])` — on the reference's
    own UR5 config and OSC, Cython cache warm.  The only harness addition is the float64 cast NumPy >= 2 needs in
    utils/transformations.py:1225 (SURVEY.md S0.3)."""
    from abr_control.utils import transformations

    _orig = transformations.quaternion_from_matrix
    transformations.quaternion_from_matrix = lambda matrix, isprecise=False: _orig(np.asarray(matrix, dtype=np.float64), isprecise)
    from abr_control.arms import ur5
    from abr_control.controllers import OSC

    rc = ur5.Config()
    ctrlr = OSC(rc, kp=OSC_KW["kp"], ctrlr_dof=[True] * 6, use_C=True)
    q, dq, tg = synth(n, 6, 123)
    for i in range(min(n, 20)):
        ctrlr.generate(q[i], dq[i], tg[i])
    cython = type(rc._M).__name__ == "cython_function_or_method"
    t0 = time.perf_counter()
    for i in range(n):
        ctrlr.generate(q[i], dq[i], tg[i])
    print(json.dumps({"evals_per_s": n / (time.perf_counter() - t0), "cython": cython}))


def as_shipped_run(n_per_worker=2000):
    """evals/s of the reference exactly as shipped: one interpreter on one core, and one interpreter per core"""
    if not os.path.isdir(os.path.join(AS_SHIPPED, "abr_control")) or not os.path.isdir(os.path.join(AS_SHIPPED, "home", ".cache")):
        return {"unavailable": "baseline/_ref (reference + warm UR5 cache, oracle/ref_harness/install_baseline.sh) is absent"}
    env = dict(os.environ, HOME=os.path.join(AS_SHIPPED, "home"), PYTHONPATH=AS_SHIPPED, OMP_NUM_THREADS="1",
               OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1")
    cmd = [sys.executable, "-W", "ignore", os.path.abspath(__file__), "--as-shipped-worker", str(n_per_worker)]

    def launch(count):
        t0 = time.perf_counter()
        procs = [subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, cwd=tempfile.gettempdir())
                 for _ in range(count)]
        outs = [p.communicate(timeout=600)[0] for p in procs]
        wall = time.perf_counter() - t0
        rates = []
        for o in outs:
            try:
                rates.append(json.loads(o.decode().strip().splitlines()[-1]))
            except Exception:
                pass
        return rates, wall

    one, _ = launch(1)
    if not one:
        return {"unavailable": "the reference did not run from baseline/_ref on this box"}
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    workers = max(1, min(cores, 64))
    many, _ = launch(workers)
    return {"evals_per_s_1_core": one[0]["evals_per_s"], "cython_path": bool(one[0]["cython"]),
            "evals_per_s_all_cores": float(sum(r["evals_per_s"] for r in many)), "workers": len(many),
            "sample": f"{n_per_worker} consecutive OSC.generate calls per interpreter (examples/timing_plots.py:14-28), "
                      "one interpreter per worker, sum of the workers' own rates",
            "harness_shim": "float64 cast in transformations.quaternion_from_matrix (NumPy >= 2, SURVEY.md S0.3)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each step a bounded sample of the workload: four batches per call so that starting the worker threads (once per
    # call in oracle/c/ref_ur5_driver.c) stays a small part of it
    n_step = 4 * B_PER_GPU
    base, _, _ = cpu_reference_run(n_step, repeats=1)
    lib = ref_lib()
    q, dq, target = synth(n_step, 6, 123)
    times = []
    if lib is not None:
        cfg = osc_cfg()
        u = np.empty((n_step, 6))
        a = (C.byref(cfg), q.ctypes.data_as(C.c_void_p), dq.ctypes.data_as(C.c_void_p),
             target.ctypes.data_as(C.c_void_p), C.c_long(n_step), u.ctypes.data_as(C.c_void_p), C.c_int(base["cores"]))
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            lib.ref_ur5_osc_batch(*a)
            if i >= args.warmup:
                times.append(time.perf_counter() - t0)
        per_step = float(np.median(times))  # the host cores are shared with other tenants of the box
        value = n_step / per_step
    else:
        value, per_step = base["value"], n_step / base["value"]
    base["value"] = value
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.gpus),
        "sample_per_step": n_step,
        "cpu_baseline": base,
        "generated_c": {"evals_per_s": value, "cores": base.get("cores"), "what": base.get("sample")},
        "as_shipped_python": as_shipped_run(),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------- our arm
def time_kernel(fn, n_launch, torch, sets):
    """average device time of one launch, CUDA events on the current stream, rotating buffer sets"""
    for i in range(3):
        fn(sets[i % len(sets)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n_launch):
        fn(sets[i % len(sets)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / n_launch


def ncu_facts(prefix):
    """dram bytes / FP-pipe fraction of a kernel from the committed ncu capture (profiles/ncu_traffic.json)"""
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        with open(tp) as fh:
            for k, v in json.load(fh).items():
                if k.startswith(prefix):
                    return v
    return {}


def run_ours(args):
    import torch
    import torch.distributed as dist

    from abr_control_b200 import _lib, parallel
    from abr_control_b200.arms import jaco2, ur5
    from abr_control_b200.controllers import OSC, AvoidObstacles, Damping

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    nccl_log = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if rank == 0 and "NCCL_DEBUG" not in os.environ:  # the transport line of the collective record
            nccl_log = os.path.join(tempfile.gettempdir(), f"abrb_nccl_{os.getpid()}.log")
            os.environ.update(NCCL_DEBUG="INFO", NCCL_DEBUG_SUBSYS="INIT,GRAPH", NCCL_DEBUG_FILE=nccl_log)
        dist.init_process_group("nccl", device_id=dev)
    B, n = B_PER_GPU, 6
    rc = ur5.Config()
    ctrlr = OSC(rc, **OSC_KW)
    L = _lib.lib()

    def max_over_ranks(seconds):
        t = torch.tensor([seconds], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ring of buffer sets > L2 (126 MB): each set = q, dq, target in (144 B/state) + u out (48 B/state)
    n_sets = 48
    sets = []
    for s in range(n_sets):
        q, dq, tg = synth(B, n, 1000 * rank + s)
        sets.append(tuple(torch.as_tensor(a, device=dev) for a in (q, dq, tg)))
    ring_mb = n_sets * B * (18 + 6) * 8 / 1e6
    outs = [torch.empty((B, n), dtype=torch.float64, device=dev) for _ in range(n_sets)]

    def step(i):
        q, dq, tg = sets[i % n_sets]
        return ctrlr.generate_into(q, dq, tg, outs[i % n_sets])  # public allocation-free API: one ctypes call

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, n_iter, warm):
        """device-event seconds per iteration of fn(i), barrier + synchronize on both sides, max over ranks"""
        for i in range(warm):
            fn(i)
        fence()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n_iter):
            fn(i)
        e1.record()
        fence()
        return max_over_ranks(e0.elapsed_time(e1) * 1e-3) / n_iter

    for i in range(max(args.warmup, 3)):
        step(i)
    fence()
    sampler = ClockSampler(local, getattr(torch.cuda.get_device_properties(local), "uuid", None)) if rank == 0 else None
    n0 = L.abrb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    fence()
    launches = L.abrb_launch_count() - n0
    t = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    clocks = sampler.stop() if sampler else None
    value = world * B * args.steps / t
    if args.dump_outputs and rank == 0:
        # what the caller of the timed path received in its last step: u of rank 0's batch (B x 6 float64, 3 MB)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "u.npy"), outs[(args.steps - 1) % n_sets].cpu().numpy())

    # ---- the one collective of the path (BASELINE config 5 / SURVEY S8e): all-gather of u so that every rank holds the
    #      (world * B, n) array.  Measured three ways with device events, max over ranks: NCCL all-gather alone, the
    #      kernel followed by NCCL all-gather, and the kernel whose epilogue stores into every rank's gathered array
    #      over NVLink peer memory (parallel.PeerGather) followed by the arrival wait.
    collective = None
    multi = {}
    if world > 1:
        n_it = max(100, min(args.steps, 400))
        gbuf = torch.empty((world * B, n), dtype=torch.float64, device=dev)
        t_ag = timed(lambda i: dist.all_gather_into_tensor(gbuf, outs[i % n_sets]), n_it, 20)

        def step_nccl(i):
            dist.all_gather_into_tensor(gbuf, step(i))

        t_seq = timed(step_nccl, n_it, 20)
        pg = parallel.PeerGather(world * B, n, torch.float64)

        def step_fused(i):
            q, dq, tg = sets[i % n_sets]
            return pg.generate(ctrlr, q, dq, tg)

        t_fused = timed(step_fused, n_it, 20)
        full = step_fused(0)  # parity of the fused gather: every rank's block equals an NCCL gather of the same step
        dist.all_gather_into_tensor(gbuf, step(0))
        torch.cuda.synchronize()
        same = bool(torch.equal(full, gbuf)) and pg.status() == 0
        payload = B * n * 8
        transport = None
        if nccl_log and os.path.exists(nccl_log):
            with open(nccl_log) as fh:
                via = sorted({ln.split(" via ")[1].split()[0] for ln in fh if " via " in ln})
            transport = ",".join(via) or None
        collective = {
            "what": "all-gather of u (float64, %d x %d per rank) so that every rank holds the (%d, %d) array" % (B, n, world * B, n),
            "payload_bytes_per_rank": payload,
            "nccl_allgather_alone_us": t_ag * 1e6,
            "nccl_bus_GBps": payload * (world - 1) / t_ag / 1e9,
            "nccl_transport": transport,
            "kernel_only_us": t / args.steps * 1e6,
            "kernel_then_nccl_allgather_us": t_seq * 1e6,
            "kernel_with_fused_peer_store_us": t_fused * 1e6,
            "fused_nvlink_bytes_out_per_rank": payload * (world - 1),
            "fused_nvlink_GBps_out_per_rank": payload * (world - 1) / t_fused / 1e9,
            "fused_matches_nccl": same,
            "evals_per_s_with_nccl_gather": world * B / t_seq,
            "evals_per_s_with_fused_gather": world * B / t_fused,
            "iterations": n_it,
        }
        pg.close()
        # ---- BASELINE config 5 at its stated scale: Jaco2 OSC x,y,z + vmax + AvoidObstacles + Damping, fp32,
        #      131072 states per GPU (1 048 576 over 8), output gathered on every rank by the fused epilogue
        B5 = 131072
        rc5 = jaco2.Config()
        c5 = OSC(rc5, kp=200, vmax=[0.5, 0], ctrlr_dof=[True, True, True, False, False, False],
                 null_controllers=[AvoidObstacles(rc5, obstacles=[[0.09596, -0.2661, 0.64204, 0.05]], threshold=0.2),
                                   Damping(rc5, kv=10)])
        s5 = []
        for s in range(12):
            q, dq, tg = synth(B5, 6, 7000 + 100 * rank + s, np.float32)
            s5.append(tuple(torch.as_tensor(a, device=dev) for a in (q, dq, tg)))
        u5 = torch.empty((B5, 6), dtype=torch.float32, device=dev)
        t5 = timed(lambda i: c5.generate_into(*s5[i % 12], u5), 40, 5)
        pg5 = parallel.PeerGather(world * B5, 6, torch.float32)
        t5g = timed(lambda i: pg5.generate(c5, *s5[i % 12]), 40, 5)
        g5 = torch.empty((world * B5, 6), dtype=torch.float32, device=dev)

        def step5_nccl(i):
            dist.all_gather_into_tensor(g5, c5.generate_into(*s5[i % 12], u5))

        t5n = timed(step5_nccl, 40, 5)
        ok5 = pg5.status() == 0
        pg5.close()
        multi["config5_jaco2_avoid_f32"] = {
            "states_per_gpu": B5, "global_states": world * B5, "us_per_step_no_gather": t5 * 1e6,
            "us_per_step_fused_gather": t5g * 1e6, "us_per_step_nccl_gather": t5n * 1e6,
            "evals_per_s_fused_gather": world * B5 / t5g, "evals_per_s_no_gather": world * B5 / t5,
            "gather_payload_bytes_total": world * B5 * 6 * 4, "gather_ok": ok5}
    # ---- BASELINE config 4 at its stated scale: UR5 OSC(kp=10) closed-loop rollouts, 512 trajectories per GPU
    #      (4096 over 8) x 128 steps, dt = 1e-3, one launch per rollout; trajectories shard, nothing is exchanged
    traj_per_gpu = 4096 // max(world, 1) if world > 1 else 4096
    c4 = OSC(rc, kp=10.0)
    q4, dq4, tg4 = (torch.as_tensor(a, device=dev) for a in synth(traj_per_gpu, 6, 4242 + rank))
    dq4 = dq4 * 0.1
    t4 = timed(lambda i: c4.rollout(q4, dq4, tg4, steps=128, dt=1e-3, record=()), 5, 2)
    multi["config4_ur5_rollout_f64"] = {
        "trajectories_per_gpu": traj_per_gpu, "global_trajectories": traj_per_gpu * world, "horizon": 128,
        "ms_per_rollout": t4 * 1e3, "us_per_step": t4 / 128 * 1e6, "osc_evals_per_s": world * traj_per_gpu * 128 / t4,
        "note": "latency bound (sequential depth 128); trajectories shard over the GPUs, nothing is exchanged"}

    # ---- end to end through the public API with pinned HOST buffers (H2D + kernel + D2H inside every call).
    #      `sync`: OSC.generate(q, dq, target) call after call, each one waits for its own result.
    #      `pipelined`: OSC.generate_async on the two pipeline slots alternately, each result awaited before its slot is
    #      reused -- batch k+1's upload runs under batch k's kernel and download (every batch still crosses PCIe both ways).
    n_host = 4
    host = []
    for s in range(n_host):
        host.append(tuple(torch.as_tensor(a).pin_memory().numpy() for a in synth(B, n, 77 + 10 * rank + s)))
    ctrlr.record_training_signal = False  # the reference also stores training_signal (osc.py:297); not copied back here
    for s in range(3):
        ctrlr.generate(*host[s % n_host])
    fence()
    calls = max(100, min(args.steps, 400))
    blocks = 5
    per_block = calls // blocks
    sync_t, pipe_t = [], []
    for _ in range(blocks):
        t0 = time.perf_counter()
        for i in range(per_block):
            u_host = ctrlr.generate(*host[i % n_host])
        sync_t.append(time.perf_counter() - t0)
    fence()
    warm = [ctrlr.generate_async(*host[i % n_host], slot=i & 1) for i in range(2)]  # both slots' workspaces, untimed
    for p_ in warm:
        p_.wait()
    warm = [ctrlr.generate_async(*host[i % n_host], slot=i & 1) for i in range(2)]
    for p_ in warm:
        p_.wait()
    fence()
    for _ in range(blocks):
        t0 = time.perf_counter()
        pend = [None, None]
        for i in range(per_block):
            sl = i & 1
            if pend[sl] is not None:
                u_host = pend[sl].wait()
            pend[sl] = ctrlr.generate_async(*host[i % n_host], slot=sl)
        for p_ in pend:
            if p_ is not None:
                u_host = p_.wait()
        pipe_t.append(time.perf_counter() - t0)
    fence()
    t_sync = max_over_ranks(float(np.median(sync_t)))
    t_pipe = max_over_ranks(float(np.median(pipe_t)))
    # what ONE stream of plain pinned cudaMemcpyAsync copies of this size reaches on this box (the library uploads q and dq
    # on two streams at once, so the achieved host->device figure can exceed the one-stream one)
    hbuf = torch.empty(B * 18, dtype=torch.float64).pin_memory()
    dbuf = torch.empty(B * 18, dtype=torch.float64, device=dev)
    def copy_rate(fn, nbytes):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(20):
            fn()
        torch.cuda.synchronize()
        return nbytes * 20 / (time.perf_counter() - t0) / 1e9
    h2d_peak = copy_rate(lambda: dbuf.copy_(hbuf, non_blocking=True), B * 18 * 8)
    d2h_peak = copy_rate(lambda: hbuf.copy_(dbuf, non_blocking=True), B * 18 * 8)
    e2e = {
        "value": world * B * per_block / t_pipe, "unit": UNIT, "h2d_bytes_per_step": int(B * 18 * 8),
        "d2h_bytes_per_step": int(B * 6 * 8), "calls": per_block * blocks, "blocks": blocks,
        "mode": "pipelined: OSC.generate_async on two slots (abrb_osc_generate_host_async_f64 + abrb_osc_host_wait); every "
                "batch is copied host->device and its u device->host inside the timed region, wall clock, median block",
        "sync_value": world * B * per_block / t_sync,
        "sync_mode": "OSC.generate(q, dq, target) on pinned host NumPy buffers, one blocking call per batch",
        "block_range_pipelined": [B * per_block / x for x in (max(pipe_t), min(pipe_t))],
        "block_range_sync": [B * per_block / x for x in (max(sync_t), min(sync_t))],
        "pcie_h2d_GBps_achieved": B * 18 * 8 * per_block / float(np.median(pipe_t)) / 1e9,
        "pcie_h2d_GBps_one_stream_pinned_copy": h2d_peak, "pcie_d2h_GBps_one_stream_pinned_copy": d2h_peak,
        "training_signal_copied": False,
    }

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm_peak, peak_src = peaks()
    bytes_per_state = (6 + 6 + 6) * 8 + 6 * 8  # q, dq, target in; u out (fp64)
    kernel_s = t / args.steps
    facts = ncu_facts("osc:osc_kernel<double, 6")
    traffic = facts.get("dram_mb_per_launch")
    traffic = traffic * 1e6 if traffic is not None else None

    extra = {}
    quick = bool(os.environ.get("ABRB_BENCH_QUICK"))  # tuning knob: headline + e2e only
    if world == 1 and not quick:
        # the other single-GPU kernels, same timing discipline (explain the headline; not bench lines themselves).
        # rbd kernels: inputs AND outputs rotate over a ring larger than L2, so every launch's outputs go to HBM
        shp = lambda Bx: dict(J=(Bx, 6, n), M=(Bx, n, n), g=(Bx, n), C=(Bx, n, n))  # noqa: E731

        def rbd_ring(Bx, want, dtype, ring_bytes=320e6):
            es = 8 if dtype == torch.float64 else 4
            per_set = Bx * (12 + sum(int(np.prod(shp(Bx)[k][1:])) for k in want)) * es
            count = max(3, int(np.ceil(ring_bytes / per_set)))
            out = []
            for s in range(count):
                q, dq, _ = synth(Bx, n, 5000 + s, np.float64 if dtype == torch.float64 else np.float32)
                o = {k: torch.empty(shp(Bx)[k], dtype=dtype, device=dev) for k in want}
                out.append((torch.as_tensor(q, device=dev), torch.as_tensor(dq, device=dev), o))
            return out, count * per_set

        for key, want, nbytes, dtype, Bx in (("rbd_ur5_JMgC_f64", ("J", "M", "g", "C"), 1008, torch.float64, B),
                                             ("rbd_ur5_JMg_f64", ("J", "M", "g"), 672, torch.float64, B),
                                             ("rbd_ur5_JMg_f32", ("J", "M", "g"), 336, torch.float32, B),
                                             ("rbd_ur5_JMgC_f64_B262144", ("J", "M", "g", "C"), 1008, torch.float64, 262144),
                                             ("rbd_ur5_JMg_f64_B262144", ("J", "M", "g"), 672, torch.float64, 262144)):
            ring, ring_b = rbd_ring(Bx, want, dtype)
            dt = time_kernel(lambda s: rc.eval_into(s[0], s[1], s[2]), 200 if Bx == B else 60, torch, ring)
            f = ncu_facts({"rbd_ur5_JMgC_f64": "rbd_JMgC:", "rbd_ur5_JMg_f64": "rbd_JMg:",
                           "rbd_ur5_JMgC_f64_B262144": "rbd_JMgC_B262144:", "rbd_ur5_JMg_f64_B262144": "rbd_JMg_B262144:"}
                          .get(key, "(no capture)"))
            extra[key] = {"states_per_s": Bx / dt, "us_per_launch": dt * 1e6, "bytes_per_state": nbytes,
                          "achieved_gbs": Bx * nbytes / dt / 1e9, "frac_hbm": Bx * nbytes / dt / 1e9 / hbm_peak, "B": Bx,
                          "ring_mb_in_and_out": ring_b / 1e6, "dram_mb_per_launch_ncu": f.get("dram_mb_per_launch"),
                          "fp_pipe_frac_ncu": f.get("fp_pipe_frac")}
            del ring
        # BASELINE config 3: Jaco2 OSC 5-DOF + Damping, fp32, B = 262144
        B3 = 262144
        rc3 = jaco2.Config()
        c3 = OSC(rc3, kp=200, ctrlr_dof=[True] * 5 + [False], null_controllers=[Damping(rc3, kv=10)])
        s3 = []
        for s in range(16):
            q, dq, tg = synth(B3, 6, 9000 + s, np.float32)
            s3.append(tuple(torch.as_tensor(a, device=dev) for a in (q, dq, tg)))
        u3 = torch.empty((B3, 6), dtype=torch.float32, device=dev)
        dt = time_kernel(lambda s: c3.generate_into(s[0], s[1], s[2], u3), 100, torch, s3)
        f = ncu_facts("osc_cfg3:")
        extra["osc_jaco2_cfg3_f32_B262144"] = {"evals_per_s": B3 / dt, "us_per_launch": dt * 1e6, "bytes_per_state": 96,
                                               "achieved_gbs": B3 * 96 / dt / 1e9, "frac_hbm": B3 * 96 / dt / 1e9 / hbm_peak,
                                               "fp_pipe_frac_ncu": f.get("fp_pipe_frac")}
        # BASELINE config 5 (per-GPU share): Jaco2 OSC xyz + vmax + AvoidObstacles(1 obstacle) + Damping, fp32, B = 131072
        B5 = 131072
        c5 = OSC(rc3, kp=200, vmax=[0.5, 0], ctrlr_dof=[True, True, True, False, False, False],
                 null_controllers=[AvoidObstacles(rc3, obstacles=[[0.09596, -0.2661, 0.64204, 0.05]], threshold=0.2),
                                   Damping(rc3, kv=10)])
        s5 = [tuple(t_[:B5].contiguous() for t_ in s) for s in s3[:8]]
        u5 = torch.empty((B5, 6), dtype=torch.float32, device=dev)
        dt = time_kernel(lambda s: c5.generate_into(s[0], s[1], s[2], u5), 50, torch, s5)
        f = ncu_facts("osc_cfg5:")
        extra["osc_jaco2_cfg5_avoid_f32_B131072"] = {"evals_per_s": B5 / dt, "us_per_launch": dt * 1e6, "bytes_per_state": 96,
                                                     "dram_mb_per_launch_ncu": f.get("dram_mb_per_launch"),
                                                     "fp_pipe_frac_ncu": f.get("fp_pipe_frac")}
        extra["rollout_ur5_cfg4_f64_4096x128"] = multi["config4_ur5_rollout_f64"]
        ctrl32 = OSC(ur5.Config(), **OSC_KW)
        s32 = [tuple(t_.float() for t_ in s) for s in sets[:24]]
        u32b = torch.empty((B, 6), dtype=torch.float32, device=dev)
        dt = time_kernel(lambda s: ctrl32.generate_into(s[0], s[1], s[2], u32b), 200, torch, s32)
        f = ncu_facts("osc_ur5_f32:")
        extra["osc_ur5_6dof_f32_B65536"] = {"evals_per_s": B / dt, "us_per_launch": dt * 1e6, "bytes_per_state": 96,
                                            "dram_mb_per_launch_ncu": f.get("dram_mb_per_launch"),
                                            "fp_pipe_frac_ncu": f.get("fp_pipe_frac")}

    cpu = None
    if world == 1 and not quick:
        cpu, u_cpu, (cq, cdq, ctg) = cpu_reference_run(4_000_000 if ref_lib() is not None else 300)
        # parity spot check in the same run: first 4096 states of the CPU sample against the GPU path
        m = min(4096, len(cq))
        ug = ctrlr.generate(cq[:m], cdq[:m], ctg[:m])
        rel = np.abs(ug - u_cpu[:m]).max(axis=1) / np.abs(u_cpu[:m]).max(axis=1)
        cpu["parity_vs_gpu_median_rel"] = float(np.median(rel))
        cpu["parity_vs_gpu_p99_rel"] = float(np.quantile(rel, 0.99))

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": bench_config(world),
        "clocks": clocks,
        "gpu_launches": int(launches),
        "e2e": e2e,
        "roofline": {"bound": "hbm", "achieved": B * bytes_per_state / kernel_s / 1e9,
                     "peak": hbm_peak, "unit": "GB/s",
                     "frac": B * bytes_per_state / kernel_s / 1e9 / hbm_peak, "traffic": traffic,
                     "kernel": "osc_kernel<double,6,ORTHO,KD=6>", "algorithmic_bytes_per_state": bytes_per_state,
                     "peak_source": peak_src,
                     "fp_pipe_frac": facts.get("fp_pipe_frac"),
                     "fp_pipe_frac_source": "sm__inst_executed_pipe_fp64 (pct of peak) of the committed ncu capture, profiles/",
                     "note": "192 B/state against ~10^4 fp64 flops/state: this kernel is FP64-pipe bound, not HBM bound "
                             "(SURVEY.md S8d): fp_pipe_frac is the fraction that binds; the HBM-bound figures are the "
                             "rbd_* kernels under 'kernels'"},
        "collective": collective,
        "configs": multi,
        "kernels": extra,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def bench_config(world):
    """the workload description shared by both arms (the driver compares the dicts)"""
    return {"workload": WORKLOAD, "arm": "ur5", "batch_per_gpu": B_PER_GPU, "global_batch": world * B_PER_GPU,
            "osc": "kp=10, ctrlr_dof=[T]*6, use_C=True, use_g=True, orientation_algorithm=0",
            "parallelism": f"batch sharded over {world} GPU(s), no data-path collective in the timed step "
                           "(the optional all-gather of u is measured separately under 'collective')",
            "l2": "inputs rotate over a ring of 48 buffer sets (604 MB > 126 MB L2)"}


def main():
    # rank 0 must print exactly ONE line on stdout (the JSON); libraries (NCCL's version banner, ...) write there too,
    # so everything else is sent to stderr and the JSON line goes to the saved descriptor
    global print
    real_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    _print = print

    def print(*a, **k):  # noqa: A001
        k.setdefault("file", real_out)
        k.setdefault("flush", True)
        _print(*a, **k)

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of the CUDA path, write the control output u of its last step as "
                         "DIR/u.npy (float64); the inputs are seeded, so two builds can be compared output for output")
    ap.add_argument("--as-shipped-worker", type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.as_shipped_worker:
        as_shipped_worker(args.as_shipped_worker)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
