#!/usr/bin/env python
"""bench.py -- samples/sec of "flow forward + log|det J| + action" on the 64x64 phi^4
workload of BASELINE.json (configs[2]: RQ-spline coupling x4, ConvAct(1->8->8->28)
conditioner, K=10 knots, batch 16384 per GPU), on N GPUs of one node.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU arm: the unmodified reference on the host cores
    python bench.py --steps 10 --warmup 3 --dump-outputs DIR   # also write the last timed step's results

One "step" = one pass of the hot path over one synthetic batch: NormalPrior draw with
log-density -> four checkerboard RQ-spline coupling steps (conditioner + spline +
log|det J|) -> phi^4 action, i.e. `model.posterior.sample__(B)`.  Ranks are independent
(batch sharding, no data-path collective): weak scaling, `value` = all ranks' samples
divided by the slowest rank's device time.

--dump-outputs DIR writes what the last timed step returned on rank 0, as .npy files (float32, or
float64 where the path returns that):
DIR/logq.npy and DIR/logp.npy (B values each) and DIR/y_sample.npy, the transformed fields y of a
fixed, seeded sample of 2048 of the B samples (32 MB; all of them when B <= 2048).  The model
weights and the prior draws are seeded, so two runs with the same arguments see the same inputs
and two builds can be compared output for output.

The JSON line carries, besides the base contract:
  roofline     : the dominant kernel (the fused coupling step), algorithmic bytes (SURVEY 8d:
                 (8 + 4 P) B per site and step = 120 B at P = 28) over its mean launch duration
                 measured with CUDA events inside the timed steps, against the measured copy
                 bandwidth of MEASURED_PEAKS.json
  cpu_baseline : the UNMODIFIED reference (staged into oracle/_ref by oracle/stage_ref.py, float64,
                 all host threads) timed on a bounded sample; the ATen port (oracle/torch_port.py)
                 only if the staged copy is missing
  e2e          : the same metric through the public API with HOST buffers: the prior draw
                 comes from pinned host memory (H2D inside the timed region; the copy of step
                 i+1 runs on a second stream while step i is evaluated) and log q, log p are
                 read back (D2H) with a stream sync every step; `e2e.with_fields` also brings the
                 transformed fields y (268 MB per step) back to pinned host memory
  train_step   : `model.fit.step()` of the same model at the same batch per GPU -- prior draw, flow,
                 action, backward, ONE flat-gradient ncclAllReduce (avg), fused AdamW -- samples/s over
                 all ranks, fraction of the 1 440 V byte model (SURVEY 8d), the collective's measured time
  mcmc         : `model.mcmc.sample(B)` (flow + device Metropolis scan + row gather)
  configs      : the other named workloads of BASELINE.json (configs[0], [1], [3], [4]): sampling and
                 training samples/s, fraction of the SURVEY 8d HBM bound, reference CPU beside them
"""

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench_configs as BC   # noqa: E402

CFG = BC.CONFIGS[3]
LATTICE = CFG['lattice']
KNOTS = BC.KNOTS
HIDDEN = BC.HIDDEN
N_STEPS_FLOW = 4
ACTION = BC.ACTION
METRIC = "samples/sec (flow fwd+logJ+action) 64^2 phi^4"
WORKLOAD = ("configs[2]: 2-D scalar phi^4 64x64, RQ-spline coupling x4 (K=10, xlim=ylim=(-5,5), linear "
            "extrapolation), ConvAct(1->8->8->28, k=3, tanh, circular, no bias) conditioner")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16384, help="samples per GPU and step")
    ap.add_argument("--cpu-batch", type=int, default=256, help="samples per step of the CPU arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip train_step / mcmc / configs")
    ap.add_argument("--train-batch", type=int, default=None, help="samples per GPU of the training step (default: --batch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's logq, logp and a fixed sample of y to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the results of the GPU path (--impl b200)")
    return a


# --------------------------------------------------------------------------- CPU arm
def cpu_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def time_cpu_port(batch, steps, warmup):
    """The reference's CPU path for this workload: oracle/torch_port.py issues the same ATen
    operator sequence as the reference (float64, ATen threads = all host cores).  Test
    infrastructure used here only as the reported CPU baseline."""
    import torch
    from oracle import torch_port as T
    threads = cpu_threads()
    torch.set_num_threads(threads)
    gen = torch.Generator('cpu').manual_seed(0)
    sizes = [1] + HIDDEN + [3 * KNOTS - 2]
    nets = [[(torch.randn(sizes[i + 1], sizes[i], 3, 3, generator=gen, dtype=torch.float64, device='cpu')
              / math.sqrt(9 * sizes[i])) for i in range(3)] for _ in range(N_STEPS_FLOW)]
    mask = T.evenodd_mask(LATTICE)

    def one():
        x = torch.randn(batch, *LATTICE, generator=gen, dtype=torch.float64, device='cpu')
        with torch.no_grad():
            return T.posterior_sample__(x, nets, mask, (-5.0, 5.0), (-5.0, 5.0), ACTION)
    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt, threads


def reference_jobs(jobs, timeout=900):
    """Run oracle/ref_runner.py jobs ([config, what, batch, steps, warmup], ...) in ONE child process with
    the GPUs hidden (the reference makes CUDA its default device when it sees one) and return the parsed
    JSON lines, or None when the staged reference is missing."""
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "normflow_ref")):
        return None
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        r = subprocess.run([sys.executable, "-m", "oracle.ref_runner", "--jobs", json.dumps(jobs)], cwd=ROOT, env=env,
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return None
    out = []
    for ln in r.stdout.splitlines():
        ln = ln.strip()
        if ln.startswith("{"):
            try:
                out.append(json.loads(ln))
            except ValueError:
                pass
    if len(out) != len(jobs):
        sys.stderr.write(r.stderr[-2000:])
        return None
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path -- the UNMODIFIED package staged
    into oracle/_ref (float64, its default; all host threads), `model.posterior.sample__` on a bounded sample
    of `--cpu-batch` samples per step of the same workload.  Falls back to the ATen port of its operator
    sequence (oracle/torch_port.py) only when the staged copy is absent."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    res = reference_jobs([[3, "sample", args.cpu_batch, args.steps, max(args.warmup, 1)]])
    if res and "samples_per_s" in res[0]:
        value, dt, cores, kind = res[0]["samples_per_s"], res[0]["seconds"], res[0]["threads"], "reference"
        what = "the unmodified reference (oracle/_ref/normflow_ref, float64) model.posterior.sample__"
    else:
        value, dt, cores = time_cpu_port(args.cpu_batch, args.steps, max(args.warmup, 1))
        kind, what = "port", "torch ATen float64 port of the reference's operator sequence"
    sample = f"{args.cpu_batch} samples/step x {args.steps} steps of the same workload ({what})"
    line = {
        "metric": METRIC, "value": value, "unit": "samples/s", "impl": "reference",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": args.batch, "lattice": list(LATTICE),
                   "cpu_sample_per_step": args.cpu_batch},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region."""

    def __init__(self, index, period=0.1):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.sm, self.reasons, self.sm_max = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def finish(self):
        self._halt.set()
        self.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons)}


# --------------------------------------------------------------------------- GPU arm
def build_model(torch, config=3):
    import normflow__b200
    model = BC.build_model(normflow__b200, BC.CONFIGS[config])
    model.device_handler.to('cuda')
    return model


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu summary."""
    path = os.path.join(ROOT, "profiles", "dominant_kernel.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh).get("dram_bytes_per_launch")
    return None


def _timed_loop(torch, dist, world, barrier, fn, steps, warmup):
    """ms per call of fn(): `warmup` untimed calls, then `steps` calls between barrier + synchronize,
    CUDA events on the launching stream, max over ranks."""
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    return ms


DUMP_Y_ROWS = 2048


def dump_outputs(path, y, logq, logp):
    """--dump-outputs: the results of one step as DIR/<name>.npy (see the module docstring)."""
    import torch
    os.makedirs(path, exist_ok=True)
    B = y.shape[0]
    rows = np.arange(B) if B <= DUMP_Y_ROWS else np.sort(np.random.default_rng(0).choice(B, DUMP_Y_ROWS, replace=False))
    arrays = {"logq": logq, "logp": logp, "y_sample": y[torch.as_tensor(rows, device=y.device)]}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def _prepare_training(torch, model, world, rank, batch):
    """What Model.fit does before its epoch loop (normflow__b200/_normflowcore.py Fitter.__call__), without the
    printing: data-parallel placement (flat gradient buffer, one all-reduce per step), fused AdamW, device-side
    divergence guard -- so that `model.fit.step()` can be timed call by call."""
    fit, handler = model.fit, model.device_handler
    if world > 1 and handler.nranks != world:
        handler.ddp_wrapper(rank, world, device=torch.device("cuda", torch.cuda.current_device()))
    params = list(model.net_.parameters())
    fit.loss_fn = fit.calc_kl_mean
    fit.optimizer = torch.optim.AdamW(params, lr=1e-3, weight_decay=0.01, fused=True)
    fit.scheduler = None
    fit._guard = dict(found_inf=torch.zeros((), dtype=torch.float32, device=params[0].device),
                      n_skipped=torch.zeros((), dtype=torch.float32, device=params[0].device))
    fit.optimizer.found_inf = fit._guard['found_inf']
    fit.train_batch_size = batch
    return sum(p.numel() for p in params)


def run_extras(args, torch, dist, model, world, rank, barrier, pk):
    """train_step / mcmc at the headline configuration and the table of the other named workloads.
    Every figure: all ranks run, device-timed, max over ranks; samples/s = all ranks' samples / that time."""
    from normflow__b200 import _C
    hbm = pk["hbm_gbs"] * 1e9
    out = {}
    B = args.batch

    def guarded(fn):
        """One failing section (e.g. out of memory on a shared box) must not take the others, or the line, with it.
        Every rank runs the same code on the same shapes, so a failure is collective and the ranks stay in step."""
        try:
            return fn()
        except Exception as err:
            torch.cuda.empty_cache()
            return {"error": f"{type(err).__name__}: {err}"[:300]}

    # ---- mcmc.sample at the headline configuration ------------------------------------------------------
    def mcmc_entry():
        np.random.seed(7 + rank)
        ms = _timed_loop(torch, dist, world, barrier, lambda: model.mcmc.sample(B), steps=min(args.steps, 5), warmup=2)
        return {"what": "model.mcmc.sample(B): flow + device Metropolis scan + row gather (independent chain per rank)",
                "config": BC.CONFIGS[3]['name'], "batch_per_gpu": B, "samples_per_s": world * B / (ms * 1e-3),
                "ms_per_step": ms, "accept_rate_last": float(model.mcmc.history.accept_rate[-1])}
    out["mcmc"] = guarded(mcmc_entry)
    model.mcmc._reset_chain()
    torch.cuda.empty_cache()

    # ---- the training step at the headline configuration (the north-star scaling target) ---------------
    def train_entry(config, m, batch, steps, warmup):
        cfg = BC.CONFIGS[config]
        n_par = _prepare_training(torch, m, world, rank, batch)
        handler = m.device_handler
        timer = _C.KernelTimer()
        orig_sync = handler.sync_gradients

        def timed_sync():
            if world == 1:
                return orig_sync()
            with timer.record("allreduce"):
                orig_sync()
        handler.sync_gradients = timed_sync
        try:
            ms_t = _timed_loop(torch, dist, world, barrier, m.fit.step, steps=steps, warmup=warmup)
        finally:
            handler.sync_gradients = orig_sync
        coll = timer.summary().get("allreduce")
        rate = world * batch / (ms_t * 1e-3)
        bytes_s = BC.train_bytes_per_sample(cfg)
        entry = {"what": "model.fit.step(): prior draw, flow, action, backward, flat-gradient all-reduce, fused AdamW",
                 "config": cfg['name'], "batch_per_gpu": batch, "samples_per_s": rate, "ms_per_step": ms_t,
                 "model_bytes_per_sample": bytes_s, "hbm_model_frac": bytes_s * rate / world / hbm,
                 "collective": None if world == 1 else {
                     "name": "ncclAllReduce (avg) of the flat float32 gradient buffer, on the compute stream",
                     "bytes": 4 * n_par, "avg_us": None if coll is None else 1e3 * coll["avg_ms"],
                     "share_of_step": None if coll is None else coll["avg_ms"] / ms_t}}
        return entry

    tb = args.train_batch or B
    out["train_step"] = guarded(lambda: train_entry(3, model, tb, steps=min(args.steps, 4), warmup=2))
    model.fit.optimizer = None
    torch.cuda.empty_cache()

    # ---- the other named workloads ------------------------------------------------------------------------
    table = {}
    plan = {   # config: (sampling batch per GPU, steps, training batch per GPU, steps)
        1: (BC.CONFIGS[1]['batch'], 50, BC.CONFIGS[1]['batch'], 50),
        2: (BC.CONFIGS[2]['batch'], 50, BC.CONFIGS[2]['batch'], 20),
        4: (max(BC.CONFIGS[4]['batch'] // world, 1), 2, 512, 2),        # 4096 global (SURVEY 8d); training at the 8-GPU share
        5: (BC.CONFIGS[5]['batch'], 2, 128, 2),                          # 2048 per GPU; training batch bounded by memory
    }
    for config, (sb, ss, tbatch, ts) in plan.items():
        cfg = BC.CONFIGS[config]
        m = build_model(torch, config)
        torch.manual_seed(4321 + rank)

        def sample_entry():
            ms_s = _timed_loop(torch, dist, world, barrier, lambda: m.posterior.sample__(sb), steps=ss,
                               warmup=2 if config < 4 else 1)
            rate = world * sb / (ms_s * 1e-3)
            fb = BC.fwd_bytes_per_sample(cfg)
            return {"batch_per_gpu": sb, "samples_per_s": rate, "ms_per_step": ms_s,
                    "model_bytes_per_sample": fb, "hbm_model_frac": fb * rate / world / hbm}
        entry = {"config": cfg['name'], "lattice": list(cfg['lattice']), "sample": guarded(sample_entry)}
        torch.cuda.empty_cache()
        entry["train"] = guarded(lambda: {k: v for k, v in train_entry(config, m, tbatch, steps=ts,
                                                                         warmup=2 if config < 4 else 1).items()
                                          if k not in ("what", "config")})
        if config < 3:
            # launch-bound workloads: the whole optimisation step -- with several ranks including the NCCL all-reduce --
            # replayed as ONE captured CUDA graph (Fitter.cuda_graph).  Two Model.fit runs of different length through
            # the public API, wall clock around each; the difference is `extra` graph replays.
            entry["train_graph"] = guarded(lambda: train_graph_entry(torch, dist, world, rank, barrier, config, tbatch))
        table[str(config)] = entry
        del m
        torch.cuda.empty_cache()
    out["configs"] = table
    return out


def train_graph_entry(torch, dist, world, rank, barrier, config, batch, base=23, extra=2000):
    import contextlib
    import io

    def timed_fit(n_epochs):
        m = build_model(torch, config)
        if world > 1:
            m.device_handler.ddp_wrapper(rank, world, device=torch.device("cuda", torch.cuda.current_device()))
        m.fit.cuda_graph = True
        barrier()
        with contextlib.redirect_stdout(io.StringIO()):
            m.fit(n_epochs=n_epochs, batch_size=batch, hyperparam=dict(lr=1e-3, weight_decay=0.01),
                  checkpoint_dict=dict(print_stride=10 ** 9, print_batch_size=128 * world, snapshot_path=None))
        torch.cuda.synchronize()
        barrier()
        timing = dict(m.fit.graph_timing)          # CUDA events around the replays: the capture (0.5 - 2.6 s) is not in it
        del m
        return timing
    timed_fit(base)                              # first use: allocator warm-up
    timing = timed_fit(base + extra)
    dt = 1e-3 * timing['ms'] / timing['replays']
    if world > 1:
        t = torch.tensor([dt], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = t.item()
    return {"what": "model.fit with fit.cuda_graph = True: one graph replay per epoch (all-reduce captured when n_gpus > 1)",
            "batch_per_gpu": batch, "samples_per_s": world * batch / dt, "ms_per_step": 1e3 * dt,
            "method": f"CUDA events around the {timing['replays']} graph replays of one fit({base + extra} epochs), diagnostics of epochs 1 and 10 inside"}


def attach_cpu(extras, results):
    """Put the reference's CPU figures (oracle/ref_runner.py jobs) beside the GPU ones."""
    for r in results:
        if "samples_per_s" not in r:
            continue
        cpu = {"samples_per_s": r["samples_per_s"], "cores": r["threads"], "kind": "reference", "dtype": "f64",
               "sample": f"{r['batch']} samples/step x {r['steps']} steps, {r['seconds']:.1f} s"}
        c, what = int(r["config"]), r["what"]
        if c == 3:
            key = {"train": "train_step", "mcmc": "mcmc"}.get(what)
            if key and isinstance(extras.get(key), dict):
                extras[key]["cpu_reference"] = cpu
        elif str(c) in extras.get("configs", {}) and isinstance(extras["configs"][str(c)].get(what), dict):
            extras["configs"][str(c)][what]["cpu_reference"] = cpu


def run_b200(args):
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (normflow__b200 has no CPU path); "
                           "use --impl reference for the CPU arm")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    numa = None
    if world > 1 and os.environ.get("NFK_BENCH_AFFINITY", "1") != "0":
        # several ranks share one host: run this rank's threads on the CPUs next to its GPU, so that the pinned host
        # buffers of the end-to-end figure are first touched on the GPU-local NUMA node (8 ranks x 268 MB per step
        # through one memory controller cost 5.6 % at N = 8 in round 1)
        try:
            import pynvml
            pynvml.nvmlInit()
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
            numa = len(os.sched_getaffinity(0))
        except Exception:
            numa = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from normflow__b200 import _C
    model = build_model(torch)
    B, V = args.batch, int(np.prod(LATTICE))
    torch.manual_seed(1234 + rank)          # independent Philox key per rank

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        return model.posterior.sample__(B)

    # warm-up with exactly the timed loop's pattern (results of the previous step still alive
    # while the next one runs, per-kernel event spans on) so that the caching allocator and
    # the event pool are in steady state: a first-use cudaMalloc inside the timed region
    # stalls the host for ~15 ms and shows up as GPU idle time
    _C.kernel_timer = _C.KernelTimer()
    y = logq = logp = None
    for _ in range(max(args.warmup, 3)):
        y, logq, logp = step()
    barrier()

    # ---- timed region: K steps, device time, max over ranks -------------------------
    timer = _C.KernelTimer()
    _C.kernel_timer = timer
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.05)                           # let the sampler thread finish its NVML set-up
    n0 = _C.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        y, logq, logp = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _C.launch_count() - n0
    clock_info = clocks.finish()
    _C.kernel_timer = None
    kernels = timer.summary()
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    value = world * B * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, y, logq, logp)

    # ---- end to end with host buffers ---------------------------------------------------
    e2e = None
    if not args.no_e2e:
        host_x = torch.randn(B, *LATTICE, dtype=torch.float32, device="cpu").pin_memory()
        host_out = torch.empty(2, B, dtype=torch.float32, device="cpu").pin_memory()

        # The step's input arrives in host memory.  It is copied in chunks on a copy stream while
        # the compute stream evaluates the chunks already on the device (public API calls per
        # chunk: prior.log_prob, net_, action), so the PCIe transfer hides behind the kernels.
        # chunk boundaries: whole waves of the fused kernel's persistent grid (2 CTAs per SM), a short
        # first chunk so that compute starts early, then ~1/8 of the batch each
        wave = 2 * torch.cuda.get_device_properties(local).multi_processor_count
        bounds = [0]
        if B >= 16 * wave:
            bounds.append(2 * wave)
            step_c = max(wave, (B // 8) // wave * wave)
            while bounds[-1] + step_c < B:
                bounds.append(bounds[-1] + step_c)
        bounds.append(B)
        n_chunks = len(bounds) - 1
        # two device input buffers: while step i is evaluated, the copy stream already brings in step i + 1
        # (a loader with a prefetch depth of one); every step's copy is issued and completed inside the
        # timed region, only the copy of the first step cannot hide behind an earlier step
        x_dev = [torch.empty(B, *LATTICE, dtype=torch.float32, device="cuda") for _ in range(2)]
        res_dev = torch.empty(2, B, dtype=torch.float32, device="cuda")
        copy_stream = torch.cuda.Stream()
        ready = [[torch.cuda.Event() for _ in range(n_chunks)] for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]

        def chunks_of(i):
            # only the first step's copy is exposed: it goes in chunks so that compute starts early; the later
            # ones complete behind the previous step's kernels and are evaluated whole
            return bounds if i == 0 else [0, B]

        def enqueue_copy(i):
            buf, bnd = i & 1, chunks_of(i)
            copy_stream.wait_event(consumed[buf])          # the step that last read this buffer is done with it
            with torch.cuda.stream(copy_stream):
                for c in range(len(bnd) - 1):
                    lo, hi = bnd[c], bnd[c + 1]
                    x_dev[buf][lo:hi].copy_(host_x[lo:hi], non_blocking=True)
                    ready[buf][c].record(copy_stream)

        host_y = None
        d2h_stream = torch.cuda.Stream()
        y_done = torch.cuda.Event()

        def e2e_run(n_steps, with_fields=False):
            """with_fields: the transformed fields y (B x V floats) also go back to pinned host memory, on a
            third stream, overlapping the next step's kernels; the copy of step i is awaited before step i + 1
            hands over its own fields (and at the end), so every copy lies inside the timed region."""
            main = torch.cuda.current_stream()
            for ev in consumed:
                ev.record(main)
            enqueue_copy(0)
            for i in range(n_steps):
                buf, bnd = i & 1, chunks_of(i)
                with torch.no_grad():
                    for c in range(len(bnd) - 1):
                        lo, hi = bnd[c], bnd[c + 1]
                        main.wait_event(ready[buf][c])
                        x = x_dev[buf][lo:hi]
                        logr = model.prior.log_prob(x)
                        yy, logJ = model.net_(x)
                        torch.sub(logr, logJ, out=res_dev[0, lo:hi])
                        torch.neg(model.action(yy), out=res_dev[1, lo:hi])
                        if with_fields:
                            y_done.synchronize()               # the host buffer is free (previous step's fields landed)
                            d2h_stream.wait_stream(main)
                            with torch.cuda.stream(d2h_stream):
                                host_y[lo:hi].copy_(yy, non_blocking=True)
                            yy.record_stream(d2h_stream)
                            if c == len(bnd) - 2:
                                y_done.record(d2h_stream)
                    consumed[buf].record(main)
                    if i + 1 < n_steps:
                        enqueue_copy(i + 1)
                    host_out.copy_(res_dev, non_blocking=True)
                main.synchronize()                         # this step's result is in host memory
            if with_fields:
                y_done.synchronize()

        e2e_run(2)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        e2e_run(args.steps)
        torch.cuda.synchronize()
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = t.item()
        e2e = {"value": world * B * args.steps / dt, "unit": "samples/s",
               "h2d_bytes_per_step": int(B * V * 4), "d2h_bytes_per_step": int(2 * B * 4),
               "chunks_first_step": n_chunks, "cpus_bound_to_gpu_numa_node": numa,
               "pipeline": "two device input buffers: the pinned-host batch of step i+1 is copied on a second stream "
                           "while step i is evaluated (all copies inside the timed region); per-step D2H + stream sync"}
        # second figure: the fields y come back too (the full result of sample__)
        host_y = torch.empty(B, *LATTICE, dtype=torch.float32, device="cpu").pin_memory()
        y_done.record(torch.cuda.current_stream())
        e2e_run(2, with_fields=True)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        e2e_run(args.steps, with_fields=True)
        torch.cuda.synchronize()
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = t.item()
        e2e["with_fields"] = {"value": world * B * args.steps / dt, "unit": "samples/s",
                              "h2d_bytes_per_step": int(B * V * 4), "d2h_bytes_per_step": int(B * V * 4 + 2 * B * 4),
                              "note": "as `e2e`, plus the transformed fields y copied to pinned host memory on a third "
                                      "stream (overlaps the next step; awaited inside the timed region)"}
        del host_y, host_x, x_dev

    pk, pk_src = peaks()
    extras = None
    if not args.no_extras:
        del y, logq, logp
        torch.cuda.empty_cache()
        try:
            extras = run_extras(args, torch, dist, model, world, rank, barrier, pk)
        except Exception as err:                  # the headline figures above must survive a failure down here
            extras = {"extras_error": f"{type(err).__name__}: {err}"[:500]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant HBM-bound kernel --------------------------------------
    P = 3 * KNOTS - 2
    # dominant kernel: the fused coupling step when the model takes that path, else the
    # unfused RQ-spline apply.  Both are scored under the SAME algorithmic byte model
    # (SURVEY 8d): one atomic step reads x, reads P conditioner channels, writes y.
    fused = kernels.get("fused2d_step", None)
    rq = fused or kernels.get("rqs_fwd", None)
    roofline = None
    if rq:
        bytes_per_launch = (8 + 4 * P) * V * B          # read x, read P params, write y
        achieved = bytes_per_launch / (rq["avg_ms"] * 1e-3) / 1e9
        name = ("nfk_fused2d_step (conditioner + RQ spline + log|det J| in one kernel)" if fused
                else "nfk_rqs_fwd (site_kernel<RqsOp<10,0>>)")
        roofline = {"kernel": name, "bound": "hbm", "achieved": achieved,
                    "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
                    "traffic": ncu_traffic(), "peak_source": pk_src,
                    "algorithmic_bytes_per_launch": bytes_per_launch, "avg_launch_ms": rq["avg_ms"],
                    "share_of_step": rq["total_ms"] / ms}
        if fused:
            # the conditioner output of the byte model never reaches DRAM in the fused kernel
            # (real traffic = 8 B/site): what actually bounds it is the contraction
            flop = 2.0 * 9 * (HIDDEN[0] + HIDDEN[0] * HIDDEN[1] + HIDDEN[1] * P / 2) * V * B
            roofline["note"] = ("compute-bound kernel: 'achieved' is algorithmic bytes (incl. the never-materialised "
                                "conditioner output) per second; real DRAM traffic is 'traffic'")
            roofline["contraction_tflops"] = flop / (rq["avg_ms"] * 1e-3) / 1e12
    step_bytes = (4 + N_STEPS_FLOW * (8 + 4 * P) + 4) * V      # SURVEY 8d: 488 V per sample
    total_ms = sum(k["total_ms"] for k in kernels.values())
    kernel_table = {name: {"launches": k["launches"], "avg_ms": round(k["avg_ms"], 4),
                           "share": round(k["total_ms"] / max(total_ms, 1e-9), 4)} for name, k in kernels.items()}

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cb = args.cpu_batch
        jobs = [[3, "sample", cb, 4, 1]]
        if extras is not None:                  # the other workloads beside their GPU numbers, bounded samples
            jobs += [[3, "train", 64, 2, 1], [3, "mcmc", 128, 2, 1],
                     [1, "sample", 128, 20, 2], [1, "train", 128, 20, 2],
                     [2, "sample", 1024, 3, 1], [2, "train", 512, 3, 1],
                     [4, "sample", 4, 1, 1], [4, "train", 2, 1, 1],
                     [5, "sample", 2, 1, 1], [5, "train", 1, 1, 1]]
        res = reference_jobs(jobs)
        if res and "samples_per_s" in res[0]:
            r0 = res[0]
            cpu = {"value": r0["samples_per_s"], "unit": "samples/s", "cores": r0["threads"], "kind": "reference",
                   "sample": f"{cb} samples/step x 4 steps of the same workload: the unmodified reference "
                             f"(oracle/_ref/normflow_ref, float64) model.posterior.sample__, {r0['seconds']:.1f} s"}
            if extras is not None:
                attach_cpu(extras, res[1:])
        else:
            v, dt, cores = time_cpu_port(cb, steps=4, warmup=1)
            cpu = {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                   "sample": f"{cb} samples/step x 4 steps of the same workload, torch ATen float64 port of the "
                             f"reference's operator sequence, {dt:.1f} s (staged reference oracle/_ref missing)"}

    line = {
        "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": B, "lattice": list(LATTICE),
                   "l2": "inputs larger than L2: every step draws a fresh 268 MB field batch (and writes 4 x 268 MB of intermediate fields), 126 MB L2",
                   "model_bytes_per_sample": step_bytes,
                   "hbm_model_frac_whole_step": step_bytes * value / world / 1e9 / pk["hbm_gbs"]},
        "clocks": clock_info, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu, "kernels": kernel_table,
    }
    if extras is not None:
        line.update(extras)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
