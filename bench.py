#!/usr/bin/env python
"""bench.py -- training_step throughput of the HashGrid + FullyFusedMLP hot path (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one trainer->training_step (fused fwd+loss+bwd kernel + Adam) over one batch of 2^18 synthetic
uniform-[0,1)^3 positions with closed-form targets. Prints ONE JSON line (rank 0). See DESIGN.md "Measurement".
Own arm: N ranks (one per GPU, torchrun), batch sharded over ranks (global batch = N * 2^18 -> weak scaling), gradients
all-reduced over NCCL before the (replicated) Adam step.
Reference arm (--impl reference): the UNMODIFIED reference compiled into oracle/_ref/ref_harness (its sm_100 build, run
on the GPU through its own C++ API; all three modes are timed and the fastest FullyFusedMLP mode is the line's value),
plus the CPU oracle port on the host cores as cpu_baseline. The reference has no CPU implementation of this path.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tiny-cuda-nn_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

BATCH = 1 << 18
N_IN, N_OUT = 3, 3
CONFIG_PATH = os.path.join(ROOT, "tests", "golden", "configs", "headline.json")
METRIC = "training_step samples/sec, HashGrid+FullyFusedMLP(64,2) batch=2^18"
WORKLOAD = "HashGrid(L=16,F=2,T=2^19,base=16,scale=1.5)+FullyFusedMLP(64x2,ReLU)->3, RelativeL2, Adam, batch=2^18/GPU, uniform [0,1)^3"
# SURVEY.md §8(d): algorithmic bytes of the fused kernel per sample (12 in + 12 target + 512 gather + 512 scatter)
FUSED_BYTES_PER_SAMPLE = 1048
ADAM_BYTES_PER_PARAM = 36


L2_NOTE = "per-step working set (tables+optimizer state ~770 MB) exceeds the 126 MB L2; 4 rotating input batches; no explicit flush"
E2E_WARMUP = 10


def config_dict(world, parallelism):
    """The SAME dict for both arms at N=1 (the driver compares them)."""
    return {"workload": WORKLOAD, "global_batch": BATCH * world, "parallelism": parallelism, "l2": L2_NOTE}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md). NVML is initialised when the sampler is
    created -- before the timed region -- so that even a region of a few milliseconds gets samples (one is taken synchronously on
    entry and one on exit, the thread adds one per millisecond in between)."""

    def __init__(self, index=0):
        self.samples = []
        self.reasons = set()
        self.stop = threading.Event()
        self.index = index
        self.nv = None
        try:
            import pynvml as nv

            nv.nvmlInit()
            idx = index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")  # CUDA_VISIBLE_DEVICES-relative index -> NVML index
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                idx = int(vis.split(",")[index])
            self.handle = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM))
            self.bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                         "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            self.nv = nv
        except Exception:  # noqa: BLE001 -- no NVML binding: poll nvidia-smi (slow, a few samples per run)
            self.nv = None
        self.thread = threading.Thread(target=self.run, daemon=True)

    def sample_nvml(self):
        nv = self.nv
        self.samples.append((float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)), self.max_mhz))
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        for n, b in self.bits.items():
            if r & b:
                self.reasons.add(n)

    def run(self):
        if self.nv is None:
            self.run_smi()
            return
        while not self.stop.is_set():
            try:
                self.sample_nvml()
            except Exception:  # noqa: BLE001
                pass
            self.stop.wait(0.001)

    def run_smi(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().splitlines()
                if out:
                    f = [v.strip() for v in out[0].split(",")]
                    self.samples.append((float(f[0]), float(f[1])))
                    for n, v in zip(names, f[3:7]):
                        if v.lower().startswith("active"):
                            self.reasons.add(n)
            except Exception:
                pass
            self.stop.wait(0.1)

    def __enter__(self):
        self.thread.start()
        return self

    def __exit__(self, *a):
        if self.nv is not None:
            try:
                self.sample_nvml()  # the GPU is still under load here: the caller synchronises after leaving the region
            except Exception:  # noqa: BLE001
                pass
        self.stop.set()
        self.thread.join(timeout=5)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": sorted(self.reasons), "samples": 0}
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0][1], "reasons": sorted(self.reasons), "samples": len(sm)}


def cpu_baseline(sample_batch=16384, steps=1):
    """The oracle port timed on the host cores over a bounded sample of the same workload (full-size tables)."""
    import numpy as np

    import oracle_binding as ob

    cfg = json.load(open(CONFIG_PATH))
    m = ob.OracleModel(N_IN, N_OUT, cfg)
    rng = ob.default_rng(1337)
    x = ob.generate_random_uniform(rng, sample_batch * N_IN).reshape(sample_batch, N_IN)
    y = ob.make_targets(x, N_OUT)
    m.training_step(x, y)  # warm-up (page in 13 M parameters)
    t0 = time.perf_counter()
    for _ in range(steps):
        m.training_step(x, y)
    dt = (time.perf_counter() - t0) / steps
    return {"value": sample_batch / dt, "unit": "samples/s", "cores": ob.load().orc_num_threads(), "kind": "port",
            "sample": f"{steps} training step(s) of {sample_batch} samples on the full 13.03M-parameter model (oracle/oracle_cpu.cpp, OpenMP)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    harness = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
    line = {"metric": METRIC, "unit": "samples/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic", "impl": "reference",
            "config": config_dict(1, "dp1")}  # the reference is a single-GPU library: one GPU whatever --gpus says
    modes = {}
    if os.path.exists(harness):
        env = dict(os.environ)
        for name, cfg, jit in (("fully_fused", "headline.json", 0), ("fully_fused_jit", "headline.json", 1), ("cutlass", "headline_cutlass.json", 0)):
            cmd = [harness, "bench", os.path.join(ROOT, "tests", "golden", "configs", cfg), str(N_IN), str(N_OUT), str(BATCH), str(args.steps), str(args.warmup), str(jit)]
            try:
                with ClockSampler() as cs:
                    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
                js = [l for l in out.stdout.splitlines() if l.startswith("{")]
                if js:
                    modes[name] = json.loads(js[-1])
                    modes[name]["clocks"] = cs.summary()
                else:
                    modes[name] = {"error": (out.stderr or out.stdout)[-400:]}
            except Exception as e:  # noqa: BLE001
                modes[name] = {"error": repr(e)}
    ok = {k: v for k, v in modes.items() if "samples_per_s" in v and k != "cutlass"}
    cb = cpu_baseline()
    if ok:
        best = max(ok, key=lambda k: ok[k]["samples_per_s"])
        line.update(value=ok[best]["samples_per_s"], ms_per_step=ok[best]["ms_per_step"], reference_mode=best, clocks=ok[best].get("clocks"),
                    final_loss=ok[best].get("loss_after_steps"))
        line["reference_modes"] = modes
        line["cpu_baseline"] = {"value": ok[best]["samples_per_s"], "unit": "samples/s", "cores": 0, "kind": "reference",
                                "sample": f"the reference's own sm_100 build on the GPU ({best}); it has no CPU path. CPU oracle port: {cb['value']:.3e} samples/s on {cb['cores']} threads"}
        line["cpu_oracle_port"] = cb
    else:
        # reference binary absent: the oracle port on the host cores is the only reference arm available
        line.update(value=cb["value"], ms_per_step=1e3 * BATCH / cb["value"], reference_mode="cpu_oracle_port", reference_modes=modes)
        line["cpu_baseline"] = cb
    line["e2e"] = {"value": line["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    if ok:
        # The reference is a GPU library, so its end-to-end number is measured like the new library's: through its own API with the
        # inputs and targets in pinned HOST buffers (H2D every step) and the loss read back every step (ref_harness `bench ... e2e`).
        cfg_file, jit = ("headline.json", 1) if best == "fully_fused_jit" else ("headline.json", 0)
        e2e_steps = max(args.steps, 100)
        cmd = [harness, "bench", os.path.join(ROOT, "tests", "golden", "configs", cfg_file), str(N_IN), str(N_OUT), str(BATCH), str(e2e_steps), str(E2E_WARMUP), str(jit), "0", "1"]
        try:
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
            js = [l for l in out.stdout.splitlines() if l.startswith("{")]
            r = json.loads(js[-1])
            line["e2e"] = {"value": BATCH / (r["wall_ms_per_step"] * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": int(r["h2d_bytes_per_step"]), "d2h_bytes_per_step": 4,
                           "steps": e2e_steps, "api": f"Trainer::training_step + Trainer::loss ({best}) on pinned host buffers, wall clock"}
        except Exception as e:  # noqa: BLE001
            line["e2e"]["error"] = repr(e)
        # secondary metric (SURVEY.md section 8d): network->inference samples/s, same batch pool
        try:
            cmd = [harness, "bench", os.path.join(ROOT, "tests", "golden", "configs", cfg_file), str(N_IN), str(N_OUT), str(BATCH), str(args.steps), str(args.warmup), str(jit), "1"]
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
            r = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
            line["inference"] = {"value": r["samples_per_s"], "unit": "samples/s", "ms_per_batch": r["ms_per_step"], "mode": best}
        except Exception as e:  # noqa: BLE001
            line["inference"] = {"error": repr(e)}
    line["gpu_launches"] = 0
    print(json.dumps(line))


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/r0N_traffic.json, newest round)."""
    try:
        for name in ("r02_traffic.json", "r01_traffic.json"):
            path = os.path.join(ROOT, "profiles", name)
            if os.path.exists(path):
                t = json.load(open(path))
                return {"kernel": t["kernel"], "bytes": t["dram_bytes_read_per_launch"] + t["dram_bytes_write_per_launch"], "source": "profiles/" + name}
    except Exception:  # noqa: BLE001
        pass
    return {}


def closed_form_targets(torch, x, n_out):
    """y_c = 0.5 + 0.5 sin(2 pi sum_d x_d (c + 1 + d) / 2^d): the smooth synthetic field both arms train on (oracle/ref_harness.cu make_targets)."""
    cols = []
    for c in range(n_out):
        phase = torch.zeros(x.shape[0], dtype=torch.float32, device=x.device)
        for d in range(x.shape[1]):
            phase = phase + x[:, d] * float(c + 1 + d) / float(1 << d)
        cols.append(0.5 + 0.5 * torch.sin(6.2831853 * phase))
    return torch.stack(cols, 1).contiguous()


def run_own(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import tcnn_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cfg = json.load(open(CONFIG_PATH))
    model = tcnn_b200.create_from_config(N_IN, N_OUT, cfg)
    trainer = model.trainer
    global_batch = BATCH * world

    # A pool of distinct batches (each rank draws its own stream) so consecutive steps do not re-read identical inputs.
    pool = 4
    rng = tcnn_b200.Pcg32(1337 + rank)  # the library's own generator (reference sequence); no oracle code on this arm
    xs, ys, xh, yh = [], [], [], []
    for _ in range(pool):
        x = tcnn_b200.generate_random_uniform(rng, BATCH * N_IN).view(BATCH, N_IN)
        y = closed_form_targets(torch, x, N_OUT)
        torch.cuda.synchronize()
        xs.append(x)
        ys.append(y)
        xh.append(x.cpu().pin_memory())
        yh.append(y.cpu().pin_memory())
    from tcnn_b200.dp import DataParallelTrainer

    # world == 1: plain training_step; else shard step + reduce-scatter of the table gradients + Adam on the rank's own table
    # slice + all-gather of the updated fp16 slices (TCNNB_DP_REPLICATED=1: all-reduce + full Adam on every replica)
    dp = DataParallelTrainer(trainer, shard_optimizer=os.environ.get("TCNNB_DP_REPLICATED", "0") != "1", native=os.environ.get("TCNNB_DP_PYTHON", "0") != "1",
                             peer_memory=os.environ.get("TCNNB_DP_NCCL", "0") != "1")  # env switches: A/B of the data-parallel engines (bench only)
    stream = torch.cuda.current_stream()

    def step(i):
        dp.training_step(xs[i % pool], ys[i % pool])

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    sync_all()
    launches0 = tcnn_b200.kernel_launch_count()
    model.set_profiling(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as cs:
        sync_all()
        e0.record(stream)
        for i in range(args.steps):
            step(i)
        e1.record(stream)
        sync_all()
    ms = e0.elapsed_time(e1)
    prof = model.read_profile()
    model.set_profiling(False)
    launches = tcnn_b200.kernel_launch_count() - launches0
    if args.dump_outputs:
        # what a caller of the timed step receives after its last step: the loss of that step and the trained parameters
        loss_last = dp.loss()
        dp.sync_full_precision()
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "loss.npy"), np.array([loss_last], np.float64))
            np.save(os.path.join(args.dump_outputs, "params.npy"), trainer.params_full_precision().cpu().numpy().astype(np.float32))
    # loss of training step number warmup + steps (one more step on the next batch of the pool): the reference arm prints the same
    # quantity after the same number of steps on the same data sequence (rank 0 draws the reference's pcg32{1337} stream)
    step(args.warmup + args.steps)
    final_loss = dp.loss()

    # ---- strong scaling (N > 1): the SAME global batch 2^18 cut into N shards (BASELINE.md section 3) -- bounded by the fixed cost
    # of the gradient exchange + optimizer pass; reported beside the weak-scaling headline
    strong = None
    if world > 1 and BATCH % (world * 256) == 0:
        sh = BATCH // world
        for i in range(max(3, args.warmup // 2)):
            dp.training_step(xs[i % pool][:sh], ys[i % pool][:sh])
        sync_all()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for i in range(args.steps):
            dp.training_step(xs[i % pool][:sh], ys[i % pool][:sh])
        s1.record(stream)
        sync_all()
        t = torch.tensor([s0.elapsed_time(s1)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        strong_ms = float(t.item()) / args.steps
        strong = {"global_batch": BATCH, "shard_batch": sh, "ms_per_step": strong_ms, "value": BATCH / (strong_ms * 1e-3), "unit": "samples/s", "scaling": "strong"}

    # ---- secondary metric: network->inference samples/s over the same batch pool (device-resident, CUDA events)
    inf_steps = max(args.steps, 20)
    for i in range(3):
        model.network.inference(xs[i % pool])
    sync_all()
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record(stream)
    for i in range(inf_steps):
        model.network.inference(xs[i % pool])
    i1.record(stream)
    sync_all()
    inf_ms = i0.elapsed_time(i1) / inf_steps
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())

    # ---- end-to-end through the C ABI with HOST buffers: every step copies its positions + targets host -> device and its loss
    # device -> host. Pipelined public API (tcnnb_training_step_host_submit / _wait): step i+1 is submitted before the loss of
    # step i is collected, so the copies of step i+1 overlap the kernels of step i; every loss is read on the host.
    e2e_steps = max(args.steps, 100)
    xn = [t.numpy() for t in xh]
    yn = [t.numpy() for t in yh]
    gb = None if world == 1 else global_batch

    def e2e_run(n):
        losses = []
        prev = model.training_step_host_submit(xn[0], yn[0], gb)
        for i in range(1, n):
            cur = model.training_step_host_submit(xn[i % pool], yn[i % pool], gb)
            losses.append(model.training_step_host_wait(prev))
            prev = cur
        losses.append(model.training_step_host_wait(prev))
        return losses

    e2e_run(E2E_WARMUP)
    sync_all()
    t0 = time.perf_counter()
    e2e_losses = e2e_run(e2e_steps)
    sync_all()
    e2e_s = time.perf_counter() - t0
    assert len(e2e_losses) == e2e_steps and all(np.isfinite(l) for l in e2e_losses)
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())

    if rank == 0:
        peak, peak_kind = measured_peaks()
        n_prof = max(1, prof["n_steps"])
        fused_ms = prof["fused_ms_total"] / n_prof
        adam_ms = prof["optimizer_ms_total"] / n_prof
        binning_ms = prof["binning_ms_total"] / n_prof
        achieved = FUSED_BYTES_PER_SAMPLE * BATCH / (fused_ms * 1e-3) / 1e9 if fused_ms > 0 else 0.0
        ms_per_step = ms / args.steps
        traffic = ncu_traffic()
        line = {
            "metric": METRIC, "value": global_batch * args.steps / (ms * 1e-3), "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16", "data": "synthetic",
            "config": config_dict(world, f"dp{world}" + ("" if world == 1 else ("-zero1" if dp.shard_optimizer else "-replicated") + ("-" + dp.engine if dp.native else "-torchdist"))),
            "clocks": cs.summary(),
            "e2e": {"value": global_batch * e2e_steps / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": BATCH * (N_IN + N_OUT) * 4, "d2h_bytes_per_step": 4,
                    "steps": e2e_steps, "warmup": E2E_WARMUP, "last_loss": e2e_losses[-1],
                    "api": ("tcnnb_training_step_host_submit/_wait" if world == 1 else "tcnnb_dp_training_step_host_submit/_wait") + " (C ABI, pinned host buffers, two steps in flight, every loss read back)"},
            "inference": {"value": global_batch / (inf_ms * 1e-3), "unit": "samples/s", "ms_per_batch": inf_ms, "steps": inf_steps},
            "strong_scaling": strong,
            "dp_engine": getattr(dp, "engine", "single"),
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": traffic.get("kernel", "fused_ws_kernel"), "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic.get("bytes"), "traffic_unit": "B/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)", "kernel_ms": fused_ms, "optimizer_kernel_ms": adam_ms, "binning_kernels_ms": binning_ms,
                         # algorithmic 36 B/parameter (SURVEY.md section 8d); the zero-gradient skip moves fewer bytes (ncu: profiles/). Only
                         # meaningful at N = 1: the sharded data-parallel optimizer runs inside the collective phase
                         "optimizer_achieved_gbs": ADAM_BYTES_PER_PARAM * model.n_params / (adam_ms * 1e-3) / 1e9 if (adam_ms > 0 and world == 1) else None,
                         "step_share": fused_ms / ms_per_step if ms_per_step > 0 else None},
            "final_loss": final_loss,
        }
        try:
            line["cpu_baseline"] = cpu_baseline() if world == 1 else None
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"error": repr(e)}
        print(json.dumps(line))
    if world > 1:
        dp.close()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss and parameters after the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
