#!/usr/bin/env python
"""bench.py -- SD1.5 PCM-LoRA distillation steps/sec on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's B200 path
    python bench.py --impl reference --gpus N --steps K ...  # the reference loop restated on CPU

Workload (BASELINE configs[1]): SD1.5 UNet (859.5 M params, random init), LoRA r=64 on the 278
target modules, 4-phase PCM, per-GPU batch 8, 512x512 images = 64x64x4 latents, bf16 compute,
CFG solver on (2 teacher passes), Huber loss, clip 1.0, AdamW.  One "step" = the full iteration
of train_pcm_lora_sd15.py:1139-1301 on one per-GPU batch.  `value` = per-GPU-batch steps per
second summed over all ranks (data parallel, weak scaling: global batch = 8 x N).
Prints ONE JSON line on rank 0.
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
sys.dont_write_bytecode = True   # the benchmark leaves the source tree untouched (it may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "distillation steps/sec (SD1.5 PCM-LoRA, bs=8/GPU)"
# algorithmic FLOPs (SURVEY.md section 8d / BASELINE.md section 3): per sample 5F + A + 4L
F_, L_, A_ = 803.6e9, 94.3e9, 126.1e9
FLOP_PER_SAMPLE_64 = 5 * F_ + A_ + 4 * L_


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1370.0), d.get("bf16_tflops", 1602.4), d.get("hbm_gbs", 6589.3), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def synth_batch(cfg, B, hw, seed, pinned=True):
    """Synthetic inputs of SURVEY.md 8(d), NHWC, on (pinned) host memory."""
    def g(s):
        return torch.Generator().manual_seed(seed * 1000 + s)
    t = dict(
        latents=torch.randn(B, hw, hw, 4, generator=g(0)),
        noise=torch.randn(B, hw, hw, 4, generator=g(1)),
        prompt=torch.randn(B, 77, cfg.cross_attention_dim, generator=g(2)).bfloat16(),
        uncond=torch.randn(1, 77, cfg.cross_attention_dim, generator=g(3)).repeat(B, 1, 1).bfloat16(),
        index=torch.randint(0, 50, (B,), generator=g(4)),
        w=4.0 + torch.rand(B, generator=g(5)),
    )
    if cfg.addition_embed:   # SDXL: zero unconditional embeddings, pooled text embedding, time ids
        t["uncond"] = torch.zeros_like(t["uncond"])
        t["index"] = torch.randint(0, 40, (B,), generator=g(4))
        t["text_embeds"] = torch.randn(B, cfg.text_embed_dim, generator=g(6)).bfloat16()
        t["time_ids"] = torch.tensor([[hw * 8, hw * 8, 0, 0, hw * 8, hw * 8]] * B)
    if pinned and torch.cuda.is_available():
        t = {k: v.pin_memory() for k, v in t.items()}
    return t


DUMP_SAMPLE = 1 << 21   # elements kept of each flat LoRA-sized buffer: 8 MB in float32


def output_snapshot(step):
    """What the last step returned to its caller, copied to the host: the loss, the updated LoRA
    factors, the AdamW moments (the optimiser kernel zeroes the LoRA gradient, the first moment
    carries it) and the optimiser state {lr, step count}.  The flat LoRA-sized buffers are sampled at
    the same seeded positions on every run, so two builds can be compared element for element."""
    master = step.unet.lora_master
    n = master.numel()
    idx = None
    if n > DUMP_SAMPLE:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
        idx = idx.to(master.device)
    out = {"loss": step.loss, "optimizer_state": step.opt_state}
    for name, t in (("lora_params", master), ("adam_exp_avg", step.exp_avg), ("adam_exp_avg_sq", step.exp_avg_sq)):
        out[name] = t if idx is None else t.index_select(0, idx)
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def write_outputs(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)


# algorithmic FLOPs of one full step of ONE sample (5F + A + 4L, SURVEY 8d), by latent size
STEP_FLOP = {64: FLOP_PER_SAMPLE_64, 32: 1.006e12}


def usable_cores():
    """Host threads this process may really use: affinity mask and cgroup CPU quota, not os.cpu_count()
    (containers on the GPU boxes report the machine's 128 cores but are throttled far below that;
    oversubscribing torch's thread pool there is ~20x slower than matching the quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    n = min(n, 64)
    # calibrate: containers may be throttled without exposing the quota -> pick the thread count that
    # actually gives the best GEMM throughput
    best, best_t = 1, None
    a = torch.randn(1536, 1536)
    for t in sorted({1, 4, 8, 16, 32, 64, n}):
        if t > n:
            continue
        torch.set_num_threads(t)
        torch.mm(a, a)
        t0 = time.perf_counter()
        for _ in range(3):
            torch.mm(a, a)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t * 0.9:
            best, best_t = t, dt
    return best


_CPU = {}


def cpu_reference_steps(steps, warmup, threads=None):
    """REAL iterations of the reference loop restated on the CPU (oracle/pcm_ref.py::pcm_step_ref with
    need_grad=True = student + 2 teacher + target forwards, Huber loss, autograd backward, then
    clip_grad_norm_ + AdamW: train_pcm_lora_sd15.py:1139-1301), fp32, on the BOUNDED sample BASELINE
    config 1: SD1.5 UNet, bs 1, 256x256 images = 32x32x4 latents, 2-phase.  The LoRA factors are updated
    between iterations like a training run.  Returns (list of seconds per timed step, cores, last loss)."""
    from oracle import pcm_ref, unet_ref
    cores = threads or usable_cores()
    torch.set_num_threads(cores)
    cfg = unet_ref.SD15
    if "P" not in _CPU:   # weights are built once per process, not per timed step
        _CPU["P"] = unet_ref.init_params(cfg, 0)
        _CPU["state"] = {}
    P = _CPU["P"]
    lk = unet_ref.lora_keys(P)
    times, loss = [], None
    for i in range(warmup + steps):
        batch = pcm_ref.make_batch(cfg, 1, 32, seed=i)
        t0 = time.perf_counter()
        r = pcm_ref.pcm_step_ref(cfg, P, batch, multiphase=2, emulate_bf16=False, need_grad=True)
        params = {k: P[k] for k in lk}
        pcm_ref.clip_and_adamw_ref(params, r["grads"], _CPU["state"], lr=5e-6, weight_decay=1e-3, max_grad_norm=1.0)
        dt = time.perf_counter() - t0
        loss = r["loss"].item()
        if i >= warmup:
            times.append(dt)
    return times, cores, loss


CPU_SAMPLE_DESC = ("bounded sample = BASELINE config 1: full reference iteration (student + 2 teacher + target "
                   "UNet forwards, Huber loss, autograd backward, clip_grad_norm_ + AdamW; oracle port of "
                   "train_pcm_lora_sd15.py:1139-1301) on SD1.5 UNet, bs 1, 32x32x4 latents, 2-phase, fp32 torch CPU")


def cpu_line(times, cores, kind="port"):
    t = sum(times) / len(times)
    sps = 1.0 / t
    return {"value": sps, "unit": "steps/s", "cores": cores, "kind": kind,
            "sample": f"{CPU_SAMPLE_DESC}; {len(times)} timed steps, {t:.2f} s/step on {cores} threads "
                      "(1.006 TFLOP per sample step vs 36.17 TFLOP per bs-8 64x64 step)",
            # clearly labelled ESTIMATE of the benchmark workload's rate on the same cores (FLOP-scaled)
            "bs8_64x64_equivalent_steps_per_s_estimate": sps * STEP_FLOP[32] / (8 * STEP_FLOP[64])}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU path.  diffusers / peft / accelerate cannot be installed
    offline (no wheels, no network), so the unmodified reference cannot run; this arm times REAL
    iterations of the oracle port (the reference loop restated in plain PyTorch) on the host cores.
    `value` is the measured rate of that bounded sample (config 1 steps/s) - NOT extrapolated;
    ms_per_step x steps is the wall time actually spent.  Rank 0 only."""
    if rank != 0:
        return
    times, cores, loss = cpu_reference_steps(args.steps, args.warmup)
    base = cpu_line(times, cores)
    value = base["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BOUNDED SAMPLE of the bs-8 workload: BASELINE config 1 = SD1.5 PCM-LoRA 2-phase, "
                               "bs=1, 256x256 (32x32x4 latents), LoRA r=64, CFG solver on, Huber, AdamW, fp32 on CPU",
                   "sample_of": "SD1.5 PCM-LoRA 4-phase, bs=8/GPU, 512x512 (64x64x4 latents)",
                   "note": "real iterations of the reference loop restated on CPU (oracle port); one sample step "
                           "is 1/36 of the algorithmic work of one bs-8 step - value is NOT scaled"},
        "loss": loss,
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--latent", type=int, default=64)
    ap.add_argument("--model", default="sd15", choices=["sd15", "sdxl"],
                    help="sdxl: BASELINE config 4 without the adversarial term (use --batch 4 --latent 128); "
                         "not the headline metric")
    ap.add_argument("--multiphase", type=int, default=4)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-only", action="store_true", help="one eager step, then exit (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (loss, sampled LoRA factors and AdamW "
                         "moments, optimiser state) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.profile_only):
        ap.error("--dump-outputs needs the timed b200 path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch.distributed as dist
    from pcm_b200 import config, ops
    from pcm_b200.step import PCMTrainStep
    from pcm_b200 import weights
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        os.environ.setdefault("NCCL_IB_DISABLE", "1")
        os.environ.setdefault("NCCL_P2P_LEVEL", "NVL")
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    cfg = config.SD15 if args.model == "sd15" else config.SDXL
    B, hw = args.batch, args.latent
    sd = weights.synthetic_state_dict(cfg, seed=0)   # identical on every rank (DDP broadcast semantics)
    step = PCMTrainStep(cfg, sd, dev, batch=B, height=hw, width=hw, multiphase=args.multiphase,
                        num_ddim_timesteps=50 if args.model == "sd15" else 40,
                        lr=5e-6, weight_decay=1e-3, max_grad_norm=1.0, process_group=pg)
    del sd
    host = [synth_batch(cfg, B, hw, seed=100 * (rank + 1) + i) for i in range(4)]  # per-rank seeds (T15:797)

    def load(i):
        h = host[i % len(host)]
        step.load_inputs(h["latents"], h["noise"], h["index"], h["w"], h["prompt"], h["uncond"],
                         text_embeds=h.get("text_embeds"), time_ids=h.get("time_ids"))

    load(0)
    torch.cuda.synchronize()
    if args.profile_only:
        step.run_eager()
        torch.cuda.synchronize()
        print("profile-only step done, loss", step.loss.item())
        return
    use_graph = not args.no_graph
    if use_graph:
        step.capture(warmup=1)
    launches_per_step = ops.LAUNCHES.get("per_step", None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed run: inputs resident in HBM -------------------------------------
    for _ in range(args.warmup):
        step.step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ops.LAUNCHES["count"] = 0
    e0.record()
    for _ in range(args.steps):
        step.step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    ms_per_step = ms / args.steps
    value = world * 1e3 / ms_per_step
    loss_last = step.loss.item()
    # taken before the passes below change the training state
    outputs = output_snapshot(step) if args.dump_outputs and rank == 0 else None

    # ---- end-to-end: pinned-host inputs -> H2D -> step -> loss D2H, every step ------------
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())
    for i in range(2):
        load(i)
        step.step()
        step.loss.cpu()
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        load(i)
        step.step()
        _ = step.loss.cpu()  # device -> host read of the step's result (the reference's loss.item())
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = t.item()
    e2e_value = world * 1e3 / (ms_e2e / args.steps)

    # ---- roofline of the dominant kernel (pcm_gemm_kernel): per-launch CUDA events ----------
    # Every pcm_gemm launch is bracketed by a pair of timing events on its stream.  The pass is
    # captured into a CUDA graph (external events = event-record nodes) and REPLAYED, so the events
    # see device time only - an eager pass adds the host's launch latency to every ~10 us kernel.
    # Fallback (PCM_ROOFLINE_EAGER=1 or capture failure): eager pass.
    sus, burst, hbm, src = peaks()
    roof = None
    if rank == 0:
        ov, step._overlap = step._overlap, False     # no collective here (other ranks do not participate)
        mode = "graph-replay"
        recs = None
        if os.environ.get("PCM_ROOFLINE_EAGER", "0") != "1":
            try:
                ops.PROFILE, ops.PROFILE_EXTERNAL = [], True
                gp = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gp):
                    step.forward_backward()
                    step._optimizer_kernels()
                recs, ops.PROFILE = ops.PROFILE, None
                for _ in range(2):
                    gp.replay()
                torch.cuda.synchronize()
                _ = recs[0][0].elapsed_time(recs[0][1])
            except Exception as e:  # noqa: BLE001
                print(f"roofline: graph-captured events unavailable ({type(e).__name__}: {e}); eager pass",
                      file=sys.stderr)
                recs = None
            finally:
                ops.PROFILE, ops.PROFILE_EXTERNAL = None, False
        if recs is None:
            mode = "eager"
            ops.PROFILE = []
            step.forward_backward()
            step._optimizer_kernels()
            torch.cuda.synchronize()
            recs, ops.PROFILE = ops.PROFILE, None
        step._overlap = ov
        tot_ms = sum(a.elapsed_time(b) for a, b, _ in recs)
        tot_fl = sum(f for _, _, f in recs)
        ach = tot_fl / (tot_ms * 1e-3) / 1e12 if tot_ms > 0 else 0.0
        traffic = None
        tj = os.path.join(ROOT, "profiles", "r2_gemm_traffic.json")
        if os.path.exists(tj):   # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed
            traffic = json.load(open(tj)).get("dram_bytes_per_launch_mean")   # `ncu --set full` capture
        roof = {"bound": "tensor", "kernel": "pcm_gemm_kernel (tcgen05 implicit GEMM, all conv/linear/LoRA/dgrad launches)",
                "achieved": ach, "peak": sus, "unit": "TFLOP/s", "frac": ach / sus, "traffic": traffic,
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({src})", "timing": mode,
                "launches": len(recs), "gemm_ms_per_step": tot_ms, "gemm_flop_per_step": tot_fl,
                "whole_step_achieved": FLOP_PER_SAMPLE_64 * B * (hw / 64.0) ** 2 / (ms_per_step * 1e-3) / 1e12,
                "whole_step_frac": FLOP_PER_SAMPLE_64 * B * (hw / 64.0) ** 2 / (ms_per_step * 1e-3) / 1e12 / sus}
        if args.model != "sd15":   # the 5F + A + 4L count of SURVEY 8(d) and the ncu traffic are the SD1.5 network's
            roof["whole_step_achieved"] = roof["whole_step_frac"] = roof["traffic"] = None
    if world > 1:
        dist.barrier()

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            times, cores, _ = cpu_reference_steps(3, 1)     # ~30 s of CPU work
            cpu = cpu_line(times, cores)
        line = {
            "metric": METRIC if args.model == "sd15" else f"distillation steps/sec (SDXL PCM-LoRA, bs={B}/GPU)",
            "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{'SD1.5' if args.model == 'sd15' else 'SDXL (no adversarial term)'} PCM-LoRA "
                                   f"{args.multiphase}-phase, bs={B}/GPU, {hw * 8}x{hw * 8} "
                                   f"({hw}x{hw}x4 latents), LoRA r=64, CFG solver on, Huber, AdamW",
                       "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
                       "cuda_graph": use_graph,
                       "l2": "working set (1.7 GB weights + >10 GB activations per step) >> 126 MB L2; no flush needed",
                       "value_definition": "per-GPU-batch steps/s summed over ranks"},
            "clocks": clocks, "loss": loss_last,
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
            "gpu_launches": int((launches_per_step or 0) * args.steps),
            "roofline": roof, "cpu_baseline": cpu,
        }
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        step.graph = step.graph_opt = None      # graphs first, then the communicator
        torch.cuda.synchronize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
