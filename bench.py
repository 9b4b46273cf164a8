#!/usr/bin/env python
"""bench.py — CFR subgame-iters/sec on the BASELINE.json workloads.

    python bench.py --gpus 1 --steps 20 --warmup 5                     # default workload: self-play data generation (configs[2])
    torchrun --nproc-per-node N ... bench.py --gpus N ...              # N GPUs, one process per GPU
    python bench.py --impl reference ...                               # the reference's own CPU path on the host cores
    python bench.py --workload {datagen,solve,config4,config5}

Workloads (`config.workload` names the one that ran):
  datagen  BASELINE configs[2], the metric's own definition (SURVEY 8d): the self-play data-generation loop — RlRunner::step
           for K concurrent 1x6f games per GPU (recursive_solving.cc:160-275), every subgame solved with 1024 CFR iterations and
           the Net2 value net on every iteration, two training examples per subgame into the replay; subgame-iters = solved
           subgames x 1024 = replay.num_add() / 2 x 1024 (selfplay.py:329-332).  One step = one wave = K subgames.
  solve    homogeneous waves of K depth-2 ROOT subgames (the worst-case subgame size; round 1's line).
  config4  BASELINE configs[3]: the data-generation loop on 2x3f, 16384 concurrent games sharded over the GPUs (strong scaling).
  config5  BASELINE configs[4]: recursive_eval --cfr on 2x3f, num_repeats sampled recursive strategies sharded over the GPUs.

Prints ONE JSON line (rank 0).  `value`: everything device resident (device-side walk, examples appended to the device-resident
replay rows), timed with CUDA events on the launching stream.  `e2e`: the same loop through the reference-facing `rela` module
(ModelLocker + ValuePrioritizedReplay + create_cfr_thread + Context) with HOST buffers on both sides — every step the trainer
side pushes fresh weights from host memory (update_model) and reads the step's examples back into host memory (sample to "cpu").
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "cfr_subgame_iters_per_sec"
UNIT = "subgame-iters/s"


WARMUP_WAVES = 20       # data generation: waves before the timed steps (at least; --warmup can ask for more)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="datagen", choices=["datagen", "solve", "config4", "config5"])
    ap.add_argument("--subgames", type=int, default=0, help="concurrent subgames / games per GPU (0 = the workload's BASELINE value)")
    ap.add_argument("--iters", type=int, default=1024)
    ap.add_argument("--dice", type=int, default=0)
    ap.add_argument("--faces", type=int, default=0)
    ap.add_argument("--repeats", type=int, default=0, help="config5: sampled recursive strategies in total (0 = 4097)")
    ap.add_argument("--net", default="auto", choices=["auto", "fp32", "tc", "tcx2"],
                    help="value-net kernel: tcx2 (default) = tcgen05 fp16 operands with the fast fp32 tanh GELU, tc = the same with the logistic fp32 GELU, fp32 = SIMT parity net")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=0, help="subgames in the CPU-baseline sample (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="datagen / config4: write the training examples of the last timed wave (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.workload not in ("datagen", "config4"):
        ap.error("--dump-outputs is implemented for the datagen and config4 workloads")
    return args


def dump_outputs(out_dir, arrays):
    """One float32 .npy per array: the outputs of two builds run with the same arguments can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, np.float32))


def dims(D, F):
    A = 1 + 2 * D * F
    H = F ** D
    return A, H, 2 + A + 2 * H


def workload_beliefs(n, H, first):
    """Synthetic random beliefs b_p[h] = u / sum(u), u ~ U(0,1); subgame g of the whole job uses counter-based stream g."""
    out = np.empty((n, 2, H), np.float64)
    for i in range(n):
        out[i] = np.random.Generator(np.random.Philox(key=first + i)).random((2, H))
    out /= out.sum(-1, keepdims=True)
    return out


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured (MEASURED_PEAKS.json, sustained bf16)"}
    return {"hbm_gbs": 6650.0, "tflops": 1590.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region, in-process through NVML (nvidia_ml_py): polling the
    nvidia-smi CLI at 5 Hz was measured to slow the timed loop by ~9 % (driver-side query cost), NVML calls do not."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index, period=float(os.environ.get("BENCH_SAMPLER_PERIOD", "0.1"))):
        self.index, self.period, self.rows, self.stop_flag, self.t, self.nv, self.h, self.max_mhz = index, period, [], False, None, None, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((mhz, reasons, time.perf_counter()))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def window(self, t0, t1):
        """Keep only the samples taken inside the timed region [t0, t1] (perf_counter)."""
        self.rows = [r for r in self.rows if t0 <= r[2] <= t1]

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.stop_flag = True
        self.t.join(timeout=2)
        sm = [r[0] for r in self.rows]
        active = sorted(name for name, bit in self.REASONS.items() if any(r[1] & bit for r in self.rows))
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(self.max_mhz) if self.max_mhz else None,
                "reasons": active, "samples": len(sm), "source": f"nvml, every {self.period:g} s during the timed steps"}


def effective_cores():
    """Host cores this process may actually use: min(cpu_count, affinity mask, cgroup CPU quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(round(int(quota) / int(period)))))
    except Exception:
        pass
    return n


_SCRIPT = {}


def script_net_file(D, F):
    if (D, F) in _SCRIPT:
        return _SCRIPT[(D, F)]
    _SCRIPT[(D, F)] = _script_net_file(D, F)
    return _SCRIPT[(D, F)]


def _script_net_file(D, F):
    import torch
    from rebel_b200.models import make_selfplay_net
    path = os.path.join(tempfile.mkdtemp(prefix="cfrb_bench_"), "net2.torchscript")
    torch.jit.script(make_selfplay_net(D, F, seed=0)).save(path)
    return path


def cpu_reference_rate(D, F, iters, n, beliefs, threads=None):
    """The reference's CPU implementation of the same workload sample (oracle/_ref when the reference compiled, else the
    C port) on the host cores.  Returns (rate, info)."""
    from oracle.oracle import Oracle, available
    cores = effective_cores()
    if available("ref_fast"):
        # all the host threads it can use: one solver thread per usable core, and 2x (SMT) — the better one is reported
        ref = Oracle("ref_fast")
        best = None
        for t in ([threads] if threads else [cores, 2 * cores]):
            m = max(t, (n // 2 // t) * t) if not threads else n
            m = min(m, n)
            s_ = ref.bench_solve(D, F, m, script_path=script_net_file(D, F), threads=t, num_iters=iters, beliefs=beliefs[:m])
            if best is None or m / s_ > best[0] / best[1]:
                best = (m, s_, t)
        n, secs, threads = best
        kind = "reference"
    else:
        import torch  # noqa: F401
        from rebel_b200.models import flatten_state_dict, make_selfplay_net
        port = Oracle("port")
        w = flatten_state_dict(make_selfplay_net(D, F, seed=0).state_dict())
        secs = port.bench_solve(D, F, n, net_w=w, num_iters=iters, beliefs=beliefs[:n])
        kind, threads = "port", 1
    rate = n * iters / secs
    sample = (f"{n} of the workload's root subgames x {iters} iters, build_solver+multistep with TorchScript Net2 on CPU, {threads} solver "
              f"threads on {cores} usable cores (os.cpu_count()={os.cpu_count()}), {secs:.1f} s wall" if kind == "reference"
              else f"{n} root subgames x {iters} iters, C port, 1 thread, {secs:.1f} s wall")
    return rate, {"value": rate, "unit": UNIT, "cores": cores if kind == "reference" else 1, "threads": threads, "kind": kind, "sample": sample}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    D, F = args.dice, args.faces
    A, H, Q = dims(D, F)
    from oracle.oracle import available
    cores = effective_cores()
    per_core = 12 if available("ref_fast") else 1
    n = args.cpu_sample or max(cores * per_core if available("ref_fast") else 2, 2)
    beliefs = workload_beliefs(n, H, 0)
    for _ in range(args.warmup):
        cpu_reference_rate(D, F, args.iters, min(n, cores if available("ref_fast") else 1), beliefs)
    t0 = time.time()
    rates, info = [], None
    for _ in range(args.steps):
        r, info = cpu_reference_rate(D, F, args.iters, n, beliefs)
        rates.append(r)
    wall = time.time() - t0
    value = n * args.iters * args.steps / sum(n * args.iters / r for r in rates)
    info["value"] = value
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 (CFR) / f32 (value net)", "data": "synthetic",
        # the workload is the B200 arm's (args.subgames concurrent subgames); each step times a bounded sample of it (cpu_baseline.sample)
        "config": workload_config(args, args.subgames), "impl_config": {"parallelism": "cpu threads"}, "cpu_baseline": info,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


WORKLOAD_DEFAULTS = {   # (dice, faces, concurrent subgames / games, scaling)
    "datagen": (1, 6, 8192, "weak"),      # BASELINE configs[2]: per GPU
    "solve": (1, 6, 8192, "weak"),
    "config4": (2, 3, 16384, "strong"),   # BASELINE configs[3]: in total, sharded over the GPUs
    "config5": (2, 3, 8192, "strong"),    # BASELINE configs[4]: wave capacity per GPU; 4097 repeats in total
}


def resolve(args):
    d, f, k, scaling = WORKLOAD_DEFAULTS[args.workload]
    args.dice = args.dice or d
    args.faces = args.faces or f
    args.scaling = scaling
    world = max(1, int(os.environ.get("WORLD_SIZE", "1")) if args.impl == "b200" else args.gpus)
    if args.workload == "config4":
        args.total_games = args.subgames * world if args.subgames else k
        args.subgames = max(1, args.total_games // max(world, 1))
    else:
        args.subgames = args.subgames or k
    args.repeats = args.repeats or 4097
    return args


def workload_config(args, k=None):
    """Identical for both arms (--impl b200 / reference): it names the workload, not how an arm runs it."""
    D, F, it = args.dice, args.faces, args.iters
    net = "Net2 n_hidden=256 n_layers=2 layer_norm, random init seed 0, evaluated on every CFR iteration"
    if args.workload == "solve":
        return {"workload": f"{D}x{F}f Liar's Dice, depth-2 root subgames (last_bid=-1), {args.subgames} concurrent subgames per GPU, "
                            f"{it} linear-CFR iterations each, Net2(256x2,LayerNorm) leaf value net every iteration",
                "subgames_per_gpu": args.subgames, "cfr_iters": it, "max_depth": 2, "value_net": net, "beliefs": "random (Philox counter streams)"}
    if args.workload in ("datagen", "config4"):
        per = (f"{args.subgames} concurrent games per GPU" if args.workload == "datagen"
               else f"{args.total_games} concurrent games in total, sharded over the GPUs")
        return {"workload": f"{D}x{F}f Liar's Dice self-play data generation (RlRunner loop: solve the subgame at the current public state with "
                            f"{it} linear-CFR iterations, depth 2, value net on every iteration; sample the next state at a random iteration; "
                            f"2 training examples per subgame into the replay), {per}; one step = one wave of subgames; "
                            "subgame-iters = solved subgames x cfr_iters = replay.num_add()/2 x cfr_iters",
                "cfr_iters": it, "max_depth": 2, "random_action_prob": 0.25, "sample_leaf": True, "value_net": net,
                "concurrent_games": args.subgames if args.workload == "datagen" else args.total_games}
    return {"workload": f"{D}x{F}f recursive_eval --cfr --subgame_iters {it}: {args.repeats} sampled recursive strategies (depth-2 subgames solved "
                        "level by level down the full tree, iteration count of every subgame sampled), float32 reach-weighted average, "
                        "exploitability; subgame-iters = CFR iterations run summed over all solved subgames",
            "cfr_iters": it, "max_depth": 2, "num_repeats": args.repeats, "value_net": net}


def run_solve(args):
    import torch
    import rebel_b200 as rb
    from rebel_b200 import dist as rbdist
    from rebel_b200.models import flatten_state_dict, make_selfplay_net

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun on this node
        port = 29500 + os.getpid() % 1000
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                   "--master-addr", "127.0.0.1", "--master-port", str(port)] + sys.argv)
    dist = None
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    D, F, K, iters = args.dice, args.faces, args.subgames, args.iters
    A, H, Q = dims(D, F)

    # ---- value-net weights: rank 0 owns them, NCCL broadcast to the other ranks (ModelLocker::updateModel analogue)
    nflat = 256 * Q + 3 * 256 + 256 * 256 + 3 * 256 + H * 256 + H
    w = rbdist.broadcast_weights(flatten_state_dict(make_selfplay_net(D, F, seed=0).state_dict()) if rank == 0 else None, nflat, dev)

    mode, mode_name = {"auto": (rb.NET_TC_F16X2, "tc_f16x2"), "tcx2": (rb.NET_TC_F16X2, "tc_f16x2"), "tc": (rb.NET_TC_F16, "tc_f16"),
                       "fp32": (rb.NET_FP32, "fp32")}[args.net]
    is_tc = mode in (rb.NET_TC_F16, rb.NET_TC_F16X2)
    S = rb.WaveSolver(D, F, K, num_iters=iters, net_mode=mode, device=local)
    S.set_weights(w, version=1)

    # ---- this rank's shard of the job: subgames [rank*K, (rank+1)*K); inputs staged in pinned host memory
    beliefs64 = workload_beliefs(K, H, rbdist.shard_range(rank, world, K)[0])
    pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True)
    t_b = pin((K, 2, H), torch.float64); t_b.numpy()[:] = beliefs64
    t_lb = pin((K,), torch.int32); t_lb.fill_(-1)
    t_pl = pin((K,), torch.int32); t_pl.zero_()
    t_act = pin((K,), torch.int32); t_act.numpy()[:] = np.random.RandomState(rank).randint(0, iters + 1, size=K)
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        return rbdist.max_over_ranks(ms, dev)

    # ================= device-resident throughput (`value`) =================
    S.begin(t_lb.numpy(), t_pl.numpy(), t_b.numpy(), t_act.numpy())
    S.set_profiling(int(os.environ.get("BENCH_PROFILE_EVERY", "16")))   # CUDA-event pairs around every 16th value-net launch of the timed steps
    sampler = ClockSampler(local)           # NVML is initialised and polling before the warm-up: its start-up (driver locks) must not
    if rank == 0 and os.environ.get("BENCH_NO_SAMPLER") != "1":   # land in the timed region; only samples taken inside it are reported
        sampler.start()
    for _ in range(max(args.warmup, 3)):    # (at least 3: eager, graph capture, replay) exactly a timed step: the L2 flush too (the first launch of torch's fill kernel loads its
        flush.fill_(1)                      # module lazily, ~70 ms of host time), and the same run configuration (the run is replayed
        S.reset(stream); S.run(iters, stream)   # from a CUDA graph that is built the second time a configuration is requested)
    barrier()
    launches0 = S.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    net_ms = 0.0
    run_ms, wall = [], []
    t_region0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        tw = time.perf_counter()
        flush.fill_(1)                      # evict L2 between steps (inside the timed region)
        S.reset(stream)
        S.run(iters, stream)
        tr, tn = S.last_run_ms()            # waits for this step; value-net kernel time from per-launch CUDA events
        net_ms += tn
        run_ms.append(round(tr, 2)); wall.append(round(1e3 * (time.perf_counter() - tw), 2))
    e1.record()
    barrier()
    if rank == 0:
        sampler.window(t_region0, time.perf_counter())
    clocks = sampler.stop() if rank == 0 else None
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = S.kernel_launches - launches0
    S.set_profiling(False)
    value = world * K * iters * args.steps / (ms * 1e-3)

    # ================= end to end through the host-buffer C ABI (`e2e`) =================
    ex_all = None
    def e2e_step():
        S.begin(t_lb.numpy(), t_pl.numpy(), t_b.numpy(), t_act.numpy())      # H2D from pinned memory
        S.run(iters, stream)
        q, v = S.examples()                                                   # D2H: training examples of the wave
        return rbdist.gather_examples(q, v, dev)                              # NCCL gather of the example blocks on rank 0
    for _ in range(2):                      # eager, then graph capture of the (unprofiled) run configuration
        e2e_step()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        flush.fill_(1)
        ex_all = e2e_step()
    f1.record()
    barrier()
    ms_e2e = max_over_ranks(f0.elapsed_time(f1))
    e2e_value = world * K * iters * args.steps / (ms_e2e * 1e-3)
    h2d = K * 2 * H * 8 + 3 * K * 4
    d2h = K * 2 * H * 4

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return
    # ================= roofline of the dominant kernel (value net) + CPU baseline =================
    peaks = load_peaks()
    rows = S.leaf_rows
    n_net = args.steps * iters
    flops_launch = 2.0 * rows * (256 * Q + 256 * 256 + 256 * H)
    avg_net_ms = net_ms / max(n_net, 1)
    traffic = None   # DRAM bytes per launch of the value-net kernel from the committed ncu --set full capture (same workload only)
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if is_tc and (D, F, K) == (1, 6, 8192):
            traffic = [v["dram_bytes_per_launch"] for k, v in tj.items() if "leaf_mlp_tc_kernel" in k][0]
    except Exception:
        traffic = None
    achieved = flops_launch / (avg_net_ms * 1e-3) / 1e12 if avg_net_ms > 0 else 0.0
    roofline = {"bound": "tensor", "kernel": "leaf value net (Net2 forward over all pseudo-leaf rows of the wave)",
                "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)", "peak_source": peaks["src"], "avg_launch_ms": avg_net_ms, "launch_timing": "CUDA events around every 16th launch inside the timed steps",
                "step_run_ms": run_ms, "step_wall_ms": wall,
                "rows_per_launch": rows,
                "flops_per_launch": flops_launch, "share_of_step": net_ms / ms if ms > 0 else None,
                "cfr_tables_algorithmic_GBps": (4 * H * (90 + 6 * 45) + 4 * 66 * (Q + H) + 8 * H) * K * iters * args.steps / max(ms - net_ms, 1e-9) / 1e6
                if (D, F) == (1, 6) else None}
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 (CFR tables) / " + ("f16 operands, f32 accumulate + LayerNorm, " + ("f32 tanh" if mode == rb.NET_TC_F16X2 else "f32 logistic") + " GELU (value net, tcgen05)" if is_tc else "f32 (value net)"),
        "data": "synthetic", "config": workload_config(args, K),
        "impl_config": {"value_net_kernel": mode_name, "parallelism": f"dp{world}", "l2": "256 MiB memset between steps, inside the timed region"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "roofline": roofline,
    }
    if world == 1 and not args.no_cpu_baseline:
        from oracle.oracle import available
        cores = effective_cores()
        n = args.cpu_sample or (cores * 24 if available("ref_fast") else 3)
        _, info = cpu_reference_rate(D, F, iters, n, beliefs64)
        out["cpu_baseline"] = info
    print(json.dumps(out), flush=True)
    if dist:
        dist.destroy_process_group()



# ============================================================================================ data generation (default workload)
class DeviceRows:
    """The replay's device-resident row storage (cfrb_rows_*, include/cfrb200.h) driven through ctypes: a ring the `value` loop
    appends every wave's examples to with one device-to-device copy, like rela.ValuePrioritizedReplay does."""

    def __init__(self, device, cap, q_dim, v_dim):
        import ctypes as C
        from rebel_b200 import capi
        self.C, self.L, self.dev, self.cap, self.head = C, capi.lib(), device, cap, 0
        self.h = C.c_void_p()
        capi._check(self.L.cfrb_rows_create(device, cap, q_dim, v_dim, C.byref(self.h)))

    def append_device(self, n, dq, dv):
        from rebel_b200 import capi
        capi._check(self.L.cfrb_rows_write(self.h, self.head, n, dq, dv, 1, self.dev))
        self.head = (self.head + n) % self.cap

    def close(self):
        self.L.cfrb_rows_destroy(self.h)


def rela_cfg(rela, args, K, mode):
    cfg = rela.RecursiveSolvingParams()
    cfg.num_dice, cfg.num_faces, cfg.random_action_prob, cfg.sample_leaf = args.dice, args.faces, 0.25, True
    cfg.concurrent_games, cfg.net_mode = K, mode
    sp = cfg.subgame_params
    sp.num_iters, sp.max_depth, sp.linear_update, sp.use_cfr = args.iters, 2, True, True
    return cfg


def template_dims(D, F, last_bid):
    """(edges E, pseudo-leaves L) of the depth-2 subgame rooted at last_bid."""
    from rebel_b200 import capi
    A = 1 + 2 * D * F
    t = capi.unroll_tree(D, F, int(last_bid), 0, 2)
    nchild = t[:, 3] - t[:, 2]
    return len(t) - 1, int(((nchild == 0) & (t[:, 0] != A - 1)).sum())


def datagen_cpu_baseline(args, seconds=9.0, threads=None):
    """The reference's own data-generation loop (RlRunner x threads with a TorchScript Net2 on CPU, what DataThreadLoop::mainLoop
    runs) on the host cores, timed on a bounded window.  Returns the cpu_baseline object."""
    from oracle.oracle import Oracle, available
    D, F, iters = args.dice, args.faces, args.iters
    cores = effective_cores()
    if not available("ref_fast"):
        import torch  # noqa: F401
        from rebel_b200.models import flatten_state_dict, make_selfplay_net
        port = Oracle("port")
        w = flatten_state_dict(make_selfplay_net(D, F, seed=0).state_dict())
        t0 = time.time()
        q, v = port.rl_runner(D, F, 0, n_games=4, num_iters=iters, net_w=w, cap=4096)
        dt = time.time() - t0
        rate = len(q) / 2 * iters / dt
        return {"value": rate, "unit": UNIT, "cores": 1, "threads": 1, "kind": "port",
                "sample": f"4 self-play games ({len(q) // 2} subgames x {iters} iters) of the C port's RlRunner loop, 1 thread, {dt:.1f} s wall"}
    ref = Oracle("ref_fast")
    out = None
    for t in ([threads] if threads else ([cores] + ([60] if cores >= 60 and cores != 60 else []))):
        counts, secs = ref.bench_datagen_windows(D, F, script_net_file(D, F), t, warmup_s=3.0, n_windows=3, window_s=seconds / 3, num_iters=iters)
        rate = counts.sum() / 2 * iters / secs.sum()
        info = {"value": rate, "unit": UNIT, "cores": cores, "threads": t, "kind": "reference",
                "sample": f"the workload's own loop on the CPU: {t} RlRunner threads (TorchScript Net2 on CPU, one game per thread at a time, seeds 0..{t - 1}) on "
                          f"{cores} usable cores (os.cpu_count()={os.cpu_count()}), {int(counts.sum())} examples in {secs.sum():.1f} s after 3 s of warm-up"}
        if out is None:
            out = info
        else:
            out[f"value_{t}_threads"] = rate      # the README recipe (60 CPU threads), where the box has >= 60 usable cores
            out["sample"] += f"; with {t} threads: {rate:.0f} {UNIT}"
    return out


def run_reference_datagen(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.oracle import Oracle, available
    D, F, iters = args.dice, args.faces, args.iters
    cores = effective_cores()
    if available("ref_fast"):
        ref = Oracle("ref_fast")
        window = 1.0
        counts, secs = ref.bench_datagen_windows(D, F, script_net_file(D, F), cores, warmup_s=3.0 + window * args.warmup, n_windows=args.steps,
                                                 window_s=window, num_iters=iters)
        value = counts.sum() / 2 * iters / secs.sum()
        ms_step = 1e3 * secs.sum() / max(args.steps, 1)
        info = {"value": value, "unit": UNIT, "cores": cores, "threads": cores, "kind": "reference",
                "sample": f"one continuous run of {cores} RlRunner threads (TorchScript Net2 on CPU) on {cores} usable cores (os.cpu_count()={os.cpu_count()}); "
                          f"each step is a {window:g} s window of it ({int(counts.sum())} examples in {secs.sum():.1f} s)"}
    else:
        info = datagen_cpu_baseline(args)
        value, ms_step = info["value"], 0.0
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64 (CFR) / f32 (value net)", "data": "synthetic", "config": workload_config(args),
        "impl_config": {"parallelism": f"{info['threads']} cpu threads, one game per thread"}, "cpu_baseline": info,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
    }), flush=True)


def run_datagen(args):
    import torch
    import rebel_b200 as rb
    import rebel_b200.rela as rela
    from rebel_b200 import dist as rbdist
    from rebel_b200.models import flatten_state_dict, make_selfplay_net

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        port = 29500 + os.getpid() % 1000
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                   "--master-addr", "127.0.0.1", "--master-port", str(port)] + sys.argv)
    dist = None
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    os.environ["CFRB_ACTOR_DEVICE"] = str(local)
    D, F, K, iters, steps = args.dice, args.faces, args.subgames, args.iters, args.steps
    A, H, Q = dims(D, F)
    nflat = 256 * Q + 3 * 256 + 256 * 256 + 3 * 256 + H * 256 + H
    net = make_selfplay_net(D, F, seed=0)
    w = rbdist.broadcast_weights(flatten_state_dict(net.state_dict()) if rank == 0 else None, nflat, dev)   # NCCL: ModelLocker::updateModel analogue
    mode, mode_name = {"auto": (rb.NET_TC_F16X2, "tc_f16x2"), "tcx2": (rb.NET_TC_F16X2, "tc_f16x2"), "tc": (rb.NET_TC_F16, "tc_f16"),
                       "fp32": (rb.NET_FP32, "fp32")}[args.net]
    is_tc = mode in (rb.NET_TC_F16, rb.NET_TC_F16X2)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    # ================= device-resident throughput (`value`): the loop through the C ABI, nothing leaves the GPU =================
    S = rb.WaveSolver(D, F, K, num_iters=iters, net_mode=mode, device=local)
    S.set_weights(w, version=1)
    S.selfplay_create(np.uint32(rank * 1000) + np.arange(K, dtype=np.uint32) * np.uint32(1000000))   # loop seed rank*1000 (selfplay.py:250), game g: + 10^6 g
    ring = DeviceRows(local, 8 * 2 * K, Q, H)

    def finish_and_start(start_next, keep):
        n = S.selfplay_wave(start_next=start_next, keep_examples=keep)
        if n:
            S.wait_examples()
            ring.append_device(n, S._sp_bufs[0], S._sp_bufs[1])
        return n
    sampler = ClockSampler(local)
    if rank == 0 and os.environ.get("BENCH_NO_SAMPLER") != "1":
        sampler.start()
    # warm-up: eager run, CUDA-graph capture, replay — and the start-up transient of a generator: all games begin at the initial state
    # together, so wave times oscillate (211 / 89 / 190 / 93 ... ms) and settle after ~20 waves (profiles/r2_wave_trend.log); the
    # timed steps measure the stationary loop whatever --warmup / --steps are
    for i in range(max(args.warmup, WARMUP_WAVES)):
        S.l2_flush()
        finish_and_start(True, True)
    finish_and_start(False, True)                   # drain: the timed region starts with no wave in flight
    S.sync()
    barrier()
    launches0 = S.kernel_launches
    t_region0 = time.perf_counter()
    S.mark(0)
    no_flush = os.environ.get("BENCH_NO_FLUSH") == "1"      # (diagnostic switch; the reported line always flushes)
    for i in range(steps):                          # step i: L2 flush, finish wave i-1 (examples -> device ring), start wave i
        if not no_flush:
            S.l2_flush()
        finish_and_start(True, True)
    n_last = finish_and_start(False, True)
    S.mark(1)
    ms = S.elapsed_ms(0, 1)
    barrier()
    if rank == 0:
        sampler.window(t_region0, time.perf_counter())
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:             # the last wave's rows, as appended to the replay rows (query, value target)
        q, v = S.selfplay_examples()
        dump_outputs(args.dump_outputs, {"examples_query": q.reshape(-1, Q)[:n_last], "examples_value": v.reshape(-1, H)[:n_last]})
    ms = rbdist.max_over_ranks(ms, dev)
    launches = S.kernel_launches - launches0
    value = world * K * iters * steps / (ms * 1e-3)

    # ---- per-kernel times of the same loop: a few profiled waves right after the timed region (CUDA-event pairs around every
    # 16th value-net launch; the rest of a wave's device time is the CFR kernel)
    prof = []
    S.set_profiling(16)
    for i in range(3):
        S.selfplay_wave(start_next=True, keep_examples=False)
        S.sync()
        tot, tnet = S.last_run_ms()
        lb, _ = S.wave_roots()
        prof.append((tot, tnet, S.leaf_rows, np.bincount(lb + 1, minlength=A)))
    S.set_profiling(0)
    S.selfplay_wave(start_next=False, keep_examples=False)
    S.sync()
    S.close(); ring.close()

    # ================= end to end through the reference-facing `rela` module with host buffers (`e2e`) =================
    ref_model = [torch.jit.script(make_selfplay_net(D, F, seed=0))]
    locker = rela.ModelLocker(ref_model, f"cuda:{local}")
    # capacity: the warm-up waves are appended without being sampled (2 K world rows each) and must fit below the capacity — the
    # producer blocks once 1.25 x capacity rows are stored (blockAppend, prioritized_replay.h:59-96)
    replay = rela.ValuePrioritizedReplay(capacity=max(1 << 18, 2 * K * world * (max(WARMUP_WAVES, args.warmup) + 12)), seed=10001 + rank, alpha=1.0, beta=1.0, prefetch=0, use_priority=False,
                                         compressed_values=False)
    if world > 1:
        # one process per GPU: the library's own NCCL communicator (cfrb_comm_*).  Every wave's examples go to rank 0's device-resident
        # replay by grouped send / recv from the generators' device buffers, and the other ranks' loops follow rank 0's ModelLocker by
        # ncclBroadcast — both enqueued on the generator's stream between two waves
        ids = [rela.comm_unique_id()] if rank == 0 else [None]
        dist.broadcast_object_list(ids, src=0)
        comm_x = rela.Comm(ids[0], rank, world, local)
        rela.set_generator_comm(comm_x, 0)
    loop = rela.create_cfr_thread(locker, replay, rela_cfg(rela, args, K, mode), rank * 1000)
    ctx = rela.Context()
    ctx.push_env_thread(loop)
    ctx.start()
    rows_per_wave = 2 * K * world if rank == 0 else 0          # rows a wave adds to THIS rank's replay (all ranks' rows land on rank 0)

    def wait_waves(target, limit=300.0):
        t0 = time.perf_counter()
        while loop.waves < target:
            if ctx.error() or time.perf_counter() - t0 > limit:
                raise RuntimeError(f"generator loop stalled: {ctx.error()}")
            time.sleep(0.0005)
    wait_waves(max(WARMUP_WAVES, args.warmup))      # warm-up waves: eager run, graph capture, replay, start-up transient (see above)
    barrier()
    w0 = loop.waves
    wait_waves(w0 + 1)
    if rank == 0:                                   # first use of the host-side path (lazy kernel loading waits for the running wave)
        locker.update_model(net)
        replay.sample(rows_per_wave, "cpu")
    # Start at a wave boundary the generator thread has registered IN TIME: the pass above can hold the replay's lock for a whole wave
    # (lazy kernel loading), during which the thread cannot register the waves the GPU completes; counting one of those late
    # registrations inside the timed region would make it one wave short.  Three registrations later the thread is level again.
    w0 = loop.waves
    wait_waves(w0 + 3)
    w0 = loop.waves
    if world > 1:
        loop.reset_between_waves_ms()
    t_sample = t_update = 0.0
    t0 = time.perf_counter()
    for i in range(steps):
        if rank == 0 and os.environ.get("BENCH_E2E_NO_UPDATE") != "1":   # (diagnostic switch; the reported line always updates)
            ta = time.perf_counter()
            locker.update_model(net)                # trainer -> generators: fresh weights from HOST memory (N > 1: + ncclBroadcast between two waves)
            t_update += time.perf_counter() - ta
        wait_waves(w0 + i + 1)
        if rank == 0:
            ta = time.perf_counter()
            batch, _ = replay.sample(rows_per_wave, "cpu")     # the step's examples (of all ranks) back to HOST memory
            t_sample += time.perf_counter() - ta
    t1 = time.perf_counter()
    between = loop.between_waves_ms if world > 1 else (0.0, 0.0)
    if world > 1:
        dist.barrier()
    ctx.terminate()
    if world > 1:
        rela.set_generator_comm(None, 0)
    while not ctx.terminated():
        time.sleep(0.01)
    barrier()
    ms_e2e = rbdist.max_over_ranks(1e3 * (t1 - t0), dev)
    e2e_value = world * K * iters * steps / (ms_e2e * 1e-3)
    Qp = (Q + 1 + 15) // 16 * 16
    h2d = 256 * Qp * 2 + 256 * 256 * 2 + 16 * 256 * 2 + 128 * 16 * 2 + 256 * 16 * 2 + 2 * 256 * 8 + 64 if is_tc else nflat * 4
    d2h = 2 * K * world * (Q + H) * 4               # rank 0 reads every rank's rows
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    # ================= roofline of the two kernels of an iteration =================
    peaks = load_peaks()
    tot = np.array([p[0] for p in prof]); tnet = np.array([p[1] for p in prof]); rows = np.array([p[2] for p in prof], np.float64)
    net_us = tnet.sum() / (len(prof) * iters) * 1e3
    cfr_us = (tot - tnet).sum() / (len(prof) * iters) * 1e3
    flops_launch = 2.0 * rows.mean() * (256 * Q + 256 * 256 + 256 * H)
    hist = sum(p[3] for p in prof)
    bytes_subgame = 0.0
    for t_idx, cnt in enumerate(hist):
        if cnt:
            E, L = template_dims(D, F, t_idx - 1)
            bytes_subgame += cnt * (4 * H * (E + 6 * E / 2) + 4 * L * (Q + H) + 8 * H)      # SURVEY 8(d), fp32-equivalent algorithmic bytes
    bytes_launch = bytes_subgame / len(prof)
    achieved = flops_launch / (net_us * 1e-6) / 1e12 if net_us > 0 else 0.0
    traffic = cfr_traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = tj.get(f"datagen_{D}x{F}_{K}", {}).get("value_net_dram_bytes_per_launch")
        cfr_traffic = tj.get(f"datagen_{D}x{F}_{K}", {}).get("cfr_dram_bytes_per_launch")
    except Exception:
        traffic = cfr_traffic = None
    roofline = {"bound": "tensor", "kernel": "leaf value net (Net2 forward over all pseudo-leaf rows of the wave, tcgen05)",
                "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"], "traffic": traffic,
                "traffic_unit": "bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)", "peak_source": peaks["src"],
                "avg_launch_ms": net_us * 1e-3, "rows_per_launch": float(rows.mean()), "flops_per_launch": flops_launch,
                "share_of_step": float(tnet.sum() / tot.sum()),
                "launch_timing": "CUDA-event pairs around every 16th launch of 3 profiled waves of the same loop, right after the timed region",
                "cfr_kernel": {"bound": "hbm", "kernel": "cfr_iter_d2_kernel (regret matching, reach / EV traversal, query rows; fp64 tables)",
                               "avg_launch_ms": cfr_us * 1e-3, "algorithmic_bytes_per_launch": bytes_launch,
                               "achieved": bytes_launch / (cfr_us * 1e-6) / 1e9 if cfr_us > 0 else 0.0, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                               "frac": bytes_launch / (cfr_us * 1e-6) / 1e9 / peaks["hbm_gbs"] if cfr_us > 0 else 0.0,
                               "share_of_step": float((tot - tnet).sum() / tot.sum()), "traffic": cfr_traffic,
                               "note": "SURVEY 8(d) fp32-equivalent bytes of the subgames actually in the waves; the tables are fp64 (about twice the table bytes move)"},
                "wave_device_ms": [round(float(x), 2) for x in tot]}
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64 (CFR tables, beliefs) / " + ("f16 operands, f32 accumulate + LayerNorm, " + ("f32 tanh" if mode == rb.NET_TC_F16X2 else "f32 logistic") + " GELU (value net, tcgen05)" if is_tc else "f32 (value net)"),
        "data": "synthetic", "config": workload_config(args),
        "impl_config": {"value_net_kernel": mode_name, "parallelism": f"dp{world}", "games_per_gpu": K, "walk": "device (mt19937 streams in HBM)",
                        "replay": "device-resident rows", "l2": "256 MiB memset between steps, inside the timed region; every wave re-initialises its solver tables"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e / steps,
                "host_ms_per_step": {"update_model": round(1e3 * t_update / steps, 3), "sample_to_cpu": round(1e3 * t_sample / steps, 3)},
                "collectives_between_waves_ms": {"mean": round(between[0], 3), "max": round(between[1], 3), "note": "device time on rank 0's generator stream, includes waiting for the slowest rank"} if world > 1 else None,
                "api": "rela.ModelLocker.update_model (weights from host memory) + rela.create_cfr_thread / Context (generator loop) + "
                       "rela.ValuePrioritizedReplay.sample(rows of the step, 'cpu') (the step's examples to host memory)" +
                       ("; N > 1: weights by ncclBroadcast, every rank's examples to rank 0's device-resident replay by ncclSend/Recv (cfrb_comm_*)" if world > 1 else ""),
                "timing": "wall clock between wave boundaries of the generator loop, device idle-synchronised before and after, max over ranks"},
        "gpu_launches": int(launches),
        "roofline": roofline,
    }
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = datagen_cpu_baseline(args)
    print(json.dumps(out), flush=True)
    if dist:
        dist.destroy_process_group()


# ============================================================================================ config 5: recursive evaluation
def run_config5(args):
    import torch
    import rebel_b200 as rb
    import rebel_b200.rela as rela
    from rebel_b200 import dist as rbdist
    from rebel_b200.models import flatten_state_dict, make_selfplay_net
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        port = 29500 + os.getpid() % 1000
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                   "--master-addr", "127.0.0.1", "--master-port", str(port)] + sys.argv)
    dist = None
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    D, F, iters = args.dice, args.faces, args.iters
    A, H, Q = dims(D, F)
    nflat = 256 * Q + 3 * 256 + 256 * 256 + 3 * 256 + H * 256 + H
    w = rbdist.broadcast_weights(flatten_state_dict(make_selfplay_net(D, F, seed=0).state_dict()) if rank == 0 else None, nflat, dev)
    mode, mode_name = {"auto": (rb.NET_TC_F16X2, "tc_f16x2"), "tcx2": (rb.NET_TC_F16X2, "tc_f16x2"), "tc": (rb.NET_TC_F16, "tc_f16"),
                       "fp32": (rb.NET_FP32, "fp32")}[args.net]
    cfg = rela_cfg(rela, args, args.subgames, mode)
    # a step = `per_step` sampled recursive strategies per rank; the run covers min(repeats, what steps allow) of the 4097
    per_rank = (args.repeats + world - 1) // world
    per_step = max(1, min(64, per_rank // max(args.steps, 1) or 1))
    wt = torch.from_numpy(w)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
    comm = None
    if dist:
        ids = [rela.comm_unique_id()] if rank == 0 else [None]
        dist.broadcast_object_list(ids, src=0)
        comm = rela.Comm(ids[0], rank, world, local)
    seed0 = rank * per_rank
    for i in range(max(1, min(args.warmup, 2))):
        rela.recursive_eval_sampled(cfg, local, min(per_step, 8), seed0, per_step, args.subgames, wt)
    barrier()
    t0 = time.perf_counter()
    iters_run, acc_s, acc_r = 0, None, None
    for i in range(args.steps):
        r = rela.recursive_eval_sampled(cfg, local, per_step, seed0 + i * per_step, per_step, args.subgames, wt)
        iters_run += int(r["subgame_iters"])
        s_, r_ = r["summed_strategy"].to(dev), r["summed_reach"].to(dev)
        acc_s = s_ if acc_s is None else acc_s + s_
        acc_r = r_ if acc_r is None else acc_r + r_
    if dist:                                        # the reference sums in strategy_id order on one thread; here ranks are reduced by NCCL (cfrb_comm_reduce_sum)
        comm.reduce_sum(acc_s.contiguous(), 0); comm.reduce_sum(acc_r.contiguous(), 0)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    barrier()
    ms = rbdist.max_over_ranks(1e3 * (t1 - t0), dev)
    tot_iters = rbdist.sum_over_ranks(float(iters_run), dev) if hasattr(rbdist, "sum_over_ranks") else float(iters_run) * world
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return
    final = (acc_s / (acc_r + 1e-6)).double().cpu()
    e0, e1 = rela.exploitability_of_strategy(D, F, final)
    value = tot_iters / (ms * 1e-3)
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64 (CFR tables) / f32 accumulators (as the reference)",
           "data": "synthetic", "config": workload_config(args),
           "impl_config": {"value_net_kernel": mode_name, "parallelism": f"dp{world}", "repeats_run": per_step * args.steps * world, "repeats_per_step_per_gpu": per_step,
                           "timing": "wall clock around the evaluator calls (host-orchestrated level walk + GPU waves), device-synchronised, max over ranks"},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "the evaluator's API is host-facing: value is already end to end"},
           "exploitability": [e0, e1], "gpu_launches": -1}
    print(json.dumps(out), flush=True)
    if dist:
        dist.destroy_process_group()


def run_reference_config5(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle.oracle import Oracle, available
    from rebel_b200.models import flatten_state_dict, make_selfplay_net
    D, F, iters = args.dice, args.faces, args.iters
    kind = "ref_fast" if available("ref_fast") else "port"
    lib = Oracle(kind)
    w = flatten_state_dict(make_selfplay_net(D, F, seed=0).state_dict())
    cores = effective_cores()
    t0 = time.time()
    res = [None] * cores

    def work(i):
        lib.sampled_strategy(D, F, seed=i, num_iters=iters, net_w=w)
        res[i] = 1
    n = cores if kind != "port" else 1
    th = [threading.Thread(target=work, args=(i,)) for i in range(n)]
    [t.start() for t in th]; [t.join() for t in th]
    dt = time.time() - t0
    # iterations per sampled strategy: E[act_iteration] x subgames (weight i/2+1 on even i): measured by the survey as 353 532 on 2x3f at 1024
    per_repeat = 353532 if (D, F, iters) == (2, 3, 1024) else None
    value = n * per_repeat / dt if per_repeat else 0.0
    info = {"value": value, "unit": UNIT, "cores": cores, "threads": n, "kind": "reference" if kind != "port" else "port",
            "sample": f"{n} sampled recursive strategies (compute_sampled_strategy_recursive_to_leaf, Net2 in fp32 on CPU), one per thread, {dt:.1f} s wall; "
                      "353 532 subgame-iters per strategy (SURVEY section 6)"}
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": 1e3 * dt, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64 / f32", "data": "synthetic",
                      "config": workload_config(args), "cpu_baseline": info,
                      "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)


if __name__ == "__main__":
    if os.environ.get("BENCH_STACK_DUMP_S"):      # debugging aid: Python stacks of every thread on stderr after that many seconds
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["BENCH_STACK_DUMP_S"]), exit=False)
    a = resolve(parse_args())
    if a.impl == "reference":
        {"solve": run_reference, "datagen": run_reference_datagen, "config4": run_reference_datagen, "config5": run_reference_config5}[a.workload](a)
    else:
        {"solve": run_solve, "datagen": run_datagen, "config4": run_datagen, "config5": run_config5}[a.workload](a)
