#!/usr/bin/env python
"""bench.py -- denoising steps/sec of the U-Net hot path (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|torch-gpu] [--workload cfg3|cfg2a|cfg1|cfg5]
                    [--dump-outputs DIR]
    (N > 1: launched by torch.distributed.run, one rank per GPU)

--dump-outputs DIR writes what the last timed step returned as DIR/image.npy in float32: the sampling image x_{t-1} (with
N > 1, the ranks' shards as the timed path gathers them: finalized to [0, 1], one global batch).  Inputs, weights and the
in-graph noise are seeded, so two builds run with the same arguments can be compared output for output.

Headline workload (default = BASELINE.json configs[2], the configuration the metric's target is quoted on; fits one GPU):
    cfg3: SR U-Net 64->256, `Unet(**Super.defaults, lowres_cond=True, text_embed_dim=768)`, 256x256, batch 32 per GPU
          (weak scaling), T=1000 schedule, cond_scale=1 (one U-Net forward per step), synthetic inputs, random-init weights.
One "step" = one `Imagen._p_sample`: U-Net forward(s) + x0 prediction + exact dynamic-threshold quantile + posterior sample.

Prints ONE JSON line (rank 0).
  value        whole-job steps/s with inputs resident in HBM: the captured step (CUDA graph) replayed K times, noise drawn
               on the device inside the graph, image / timestep updated in place.
  e2e          the same step driven with HOST (pinned) buffers: x, t and the noise copied in, x' copied out, every step.
  roofline     the dominant kernel (tcgen05 3x3 implicit-GEMM convolution): ALGORITHMIC conv FLOPs of its launches divided
               by their CUDA-event durations (launches timed one by one in an eager step), against MEASURED_PEAKS.json.
  secondary    the other BASELINE.json configurations, same metric: cfg 1 (tiny), cfg 2a / 2b (base U-Net, weak, b=64/GPU),
               cfg 4 (cascade base64 + SR256, classifier-free guidance w=7, GLOBAL batch 128 = strong scaling: 128/N per
               GPU) and cfg 5 (SR 256->1024 dim=256, GLOBAL batch 16 = strong scaling), each with its whole-step fraction
               of the measured tensor peak.
  cpu_baseline the CPU oracle port (oracle/restatement.py, the reference's algorithm in torch fp32) on this box's host
               cores at batch 1, 2, 4 (per-image time stated for each), scaled to the workload batch.
  torch_gpu    informational: the same restatement executed by stock PyTorch (cuDNN / cuBLAS) on this GPU, fp32 and fp16
               autocast -- "the only existing kernels to beat on the same box" (SURVEY.md 2.1).
`--impl reference` times the CPU path alone (the reference has no other implementation of this path); `--impl torch-gpu`
prints the stock-PyTorch-on-GPU line alone.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic GFLOP per image per U-Net forward, counted on the reference model (SURVEY.md 8d / BASELINE.md section 2)
GFLOP_PER_IMG = {"cfg1": 1.30, "cfg2a": 131.70, "cfg2b": 76.71, "cfg3": 800.57, "cfg5": 50875.83}
METRIC = "denoising steps/sec (SR256 U-Net, batch 32 per GPU per step)"


def workload(name):
    from minimagen_b200.Unet import Base, BaseTest, Super
    if name == "cfg3":
        return dict(cfg=dict(Super.defaults, lowres_cond=True, text_embed_dim=768), size=256, batch=32, T=1000,
                    E=768, lowres=True, desc="SR U-Net 64->256 dim=128 (Super.defaults, lowres_cond) b=32 256x256 T=1000")
    if name == "cfg2a":
        return dict(cfg=dict(text_embed_dim=768), size=64, batch=64, T=1000, E=768, lowres=False,
                    desc="base U-Net dim=128 (Unet ctor defaults) b=64 64x64 T=1000")
    if name == "cfg2b":
        return dict(cfg=dict(Base.defaults, dim=128, text_embed_dim=768), size=64, batch=64, T=1000, E=768, lowres=False,
                    desc="base U-Net Base.defaults with dim=128 b=64 64x64 T=1000")
    if name == "cfg1":
        return dict(cfg=dict(BaseTest.defaults), size=64, batch=2, T=25, E=512, lowres=False,
                    desc="tiny base U-Net dim=8 b=2 64x64 T=25")
    if name == "cfg5":
        return dict(cfg=dict(Super.defaults, dim=256, lowres_cond=True, text_embed_dim=768), size=1024, batch=2, T=1000,
                    E=768, lowres=True, desc="SR U-Net 256->1024 dim=256 (Super.defaults, lowres_cond) 1024x1024 T=1000")
    raise SystemExit(f"unknown workload {name}")


def synth_inputs(wl, batch, seed):
    """Synthetic conditioning exactly shaped like the reference's inputs (SURVEY.md 8d)."""
    g = torch.Generator().manual_seed(seed)
    s, E = wl["size"], wl["E"]
    lengths = torch.randint(4, 65, (batch,), generator=g)
    L = int(lengths.max())
    text = torch.randn(batch, L, E, generator=g)
    mask = torch.arange(L)[None, :] < lengths[:, None]
    text = text * mask[..., None]                               # t5.py:82 zeroes padded positions
    d = dict(text_embeds=text, text_mask=mask, x=torch.randn(batch, 3, s, s, generator=g))
    if wl["lowres"]:
        d["lowres_img01"] = torch.rand(batch, 3, s, s, generator=g)     # up-sampled low-res image in [0,1]
        d["lowres_noise"] = torch.randn(batch, 3, s, s, generator=g)
    return d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw = [], [], []
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); pw.append(float(parts[3]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            load = [c for c, p in zip(sm, pw) if p > 300] or sm
            out.update(sm_mhz=statistics.median(load), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       power_w_max=max(pw))
        return out


# ------------------------------------------------------------------------------------------------ CPU baseline
def physical_cores():
    """Physical cores this process may run on: distinct SMT sibling sets among os.sched_getaffinity(0).  (One thread per
    physical core: on the 2 x 32-core HT hosts of the B200 boxes 128 threads are ~200x slower than 64.)"""
    cpus = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    sets = set()
    for c in cpus:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                sets.add(f.read().strip())
        except OSError:
            sets.add(str(c))
    return max(1, len(sets)), len(cpus)


def cpu_baseline(wl, sd, batches=(1, 2, 4), steps=2, warmup=1, budget_s=70.0):
    """The reference's algorithm (CPU oracle port) on the host cores: U-Net forward + DDPM step at batch 1, 2 and 4 (each:
    `warmup` + `steps` timed), the per-image time of the LARGEST batch scaled linearly to the workload batch (SURVEY.md 8d;
    the full batch would take ~1 minute per step).  Stops adding batch sizes once `budget_s` of CPU time is spent."""
    from oracle import restatement as R
    cores, logical = physical_cores()
    torch.set_num_threads(cores)
    tabs = R.ddpm_tables(wl["T"])
    sd_cpu = {k: v.detach().float().cpu() for k, v in sd.items()}
    per_image, x_std = {}, None
    spent = 0.0
    with torch.no_grad():
        for b in batches:
            if per_image and spent + (warmup + steps) * b * min(per_image.values()) > budget_s:
                break
            inp = synth_inputs(wl, b, 123)
            t = torch.full((b,), wl["T"] - 1, dtype=torch.long)
            kw = dict(text_embeds=inp["text_embeds"], text_mask=inp["text_mask"])
            if wl["lowres"]:
                t_aug = torch.full((b,), int(wl["T"] * 0.2), dtype=torch.long)
                lr = R.q_sample(tabs, inp["lowres_img01"], t_aug, inp["lowres_noise"]) * 2 - 1
                kw.update(lowres_cond_img=lr, lowres_noise_times=t_aug)
            x = inp["x"]
            times = []
            for i in range(warmup + steps):
                t0 = time.perf_counter()
                eps = R.unet_forward(sd_cpu, wl["cfg"], x, t, **kw)
                x_next = R.p_sample_step(tabs, x, t, eps, torch.randn_like(x))
                dt = time.perf_counter() - t0
                spent += dt
                if i >= warmup:
                    times.append(dt)
            per_image[b] = sum(times) / len(times) / b
            x_std = float(x_next.std())
    b_used = max(per_image)
    per_step = per_image[b_used] * wl["batch"]
    gf = GFLOP_PER_IMG.get(wl.get("name", ""), 0)
    return dict(value=1.0 / per_step, unit="steps/s", cores=cores, logical_cpus=logical, kind="port",
                seconds_per_image={str(b): round(v, 4) for b, v in per_image.items()},
                sample=f"batches {sorted(per_image)} of {wl['batch']}: {warmup} warm-up + {steps} timed (U-Net forward + DDPM "
                       f"step) each on {cores} host threads (physical cores of the affinity mask); per-image seconds "
                       f"{ {b: round(v, 3) for b, v in per_image.items()} }; the batch-{b_used} per-image time x {wl['batch']} "
                       f"= {per_step:.1f} s per workload step (extrapolated, not run)",
                gflops=gf / per_image[b_used] if gf else None), x_std


# ------------------------------------------------------------------------------------------------ stock PyTorch on the GPU
def torch_gpu_baseline(wl, sd, dev, batch, steps=3, warmup=1):
    """Informational arm: oracle/restatement.py (plain torch ops -> cuDNN / cuBLAS) on the same GPU, same step."""
    from oracle import restatement as R
    out = {}
    tabs = {k: v.to(dev) for k, v in R.ddpm_tables(wl["T"]).items()}
    sd_d = {k: v.detach().float().to(dev) for k, v in sd.items()}
    inp = synth_inputs(wl, batch, 123)
    t = torch.full((batch,), wl["T"] - 1, dtype=torch.long, device=dev)
    kw = dict(text_embeds=inp["text_embeds"].to(dev), text_mask=inp["text_mask"].to(dev))
    if wl["lowres"]:
        t_aug = torch.full((batch,), int(wl["T"] * 0.2), dtype=torch.long, device=dev)
        lr = R.q_sample(tabs, inp["lowres_img01"].to(dev), t_aug, inp["lowres_noise"].to(dev)) * 2 - 1
        kw.update(lowres_cond_img=lr, lowres_noise_times=t_aug)
    x = inp["x"].to(dev)
    for name, ctx in (("fp32", None), ("fp16_autocast", torch.float16)):
        try:
            with torch.no_grad():
                def one():
                    if ctx is None:
                        eps = R.unet_forward(sd_d, wl["cfg"], x, t, **kw)
                    else:
                        with torch.autocast("cuda", dtype=ctx):
                            eps = R.unet_forward(sd_d, wl["cfg"], x, t, **kw)
                    return R.p_sample_step(tabs, x, t, eps.float(), torch.randn_like(x))
                for _ in range(warmup):
                    one()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    one()
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / steps
            out[name] = {"ms_per_step": ms, "steps_per_s": 1000.0 / ms}
        except Exception as ex:            # informational arm: never takes the bench down
            out[name] = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}
        torch.cuda.empty_cache()
    out["note"] = (f"oracle/restatement.py run by stock PyTorch {torch.__version__} on this GPU, batch {batch}, eager, "
                   f"cudnn.allow_tf32={torch.backends.cudnn.allow_tf32}, matmul.allow_tf32={torch.backends.cuda.matmul.allow_tf32}; "
                   f"{warmup} warm-up + {steps} timed")
    return out


# ------------------------------------------------------------------------------------------------ our arm: helpers
def make_cond(wl, B, seed, dev, sch, ops):
    """Device-resident conditioning of one (micro-)batch: text, mask and -- for SR U-Nets -- the noise-augmented low-res image."""
    inp = synth_inputs(wl, B, seed)
    kw = dict(text_embeds=inp["text_embeds"].to(dev), text_mask=inp["text_mask"].to(dev), lowres_cond_img=None,
              lowres_noise_times=None)
    if wl["lowres"]:
        n_img = 3 * wl["size"] * wl["size"]
        t_aug = sch._get_times(B, 0.2, device=dev)
        lr = torch.empty((B, 3, wl["size"], wl["size"]), device=dev)
        ops.q_sample(inp["lowres_img01"].to(dev), inp["lowres_noise"].to(dev), t_aug, sch.sqrt_alphas_cumprod,
                     sch.sqrt_one_minus_alphas_cumprod, B, n_img, 2.0, -1.0, lr)     # noise in [0,1] space, then *2-1
        kw.update(lowres_cond_img=lr, lowres_noise_times=t_aug)
    return inp, kw


def timed_replays(g, n, world, dev):
    """n graph replays between CUDA events (barrier + synchronize on both sides); returns ms (this rank)."""
    import torch.distributed as dist
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    return e0.elapsed_time(e1)


def max_over_ranks(v, world, dev):
    if world == 1:
        return float(v)
    import torch.distributed as dist
    t = torch.tensor([float(v)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def measure_config(imagen, unet, wl, name, *, per_gpu, micro, cond_scale, cfg_batched, steps, warmup, world, rank, dev,
                   peak_tf, global_batch, scaling):
    """steps/s of `unet` for `per_gpu` samples per GPU processed as per_gpu/micro micro-batches (captured step replayed)."""
    ops = __import__("minimagen_b200.ops", fromlist=["get_ops"]).get_ops()
    sch = imagen.noise_schedulers[list(imagen.unets).index(unet)]
    n_micro = max(1, per_gpu // micro)
    shape = (micro, 3, wl["size"], wl["size"])
    _, kw = make_cond(wl, micro, 2000 + rank, dev, sch, ops)
    imagen.cfg_batched = cfg_batched
    torch.cuda.reset_peak_memory_stats(dev)
    with torch.no_grad():
        g = imagen._step_graph(unet, shape, noise_scheduler=sch, cond_scale=cond_scale, **kw)
        g.x.normal_()
        g.t.fill_(wl["T"] - 1)
        for _ in range(max(3, warmup)):
            g.replay()
        ms = timed_replays(g, steps * n_micro, world, dev)
        ok = bool(torch.isfinite(g.x).all())
    ms = max_over_ranks(ms, world, dev)
    imagen.cfg_batched = False
    fwd = 2 if cond_scale != 1 else 1
    ms_step = ms / steps                                           # one step of this rank's whole shard (all micro-batches)
    sps = (world if scaling == "weak" else 1) * 1000.0 / ms_step   # weak: N shards advance per step; strong: one global step
    tf = GFLOP_PER_IMG.get(name, 0.0) * per_gpu * fwd / ms_step    # GFLOP / ms = TFLOP/s per GPU
    return {"steps_per_s": sps, "ms_per_step": ms_step, "batch_per_gpu": per_gpu, "micro_batch": micro,
            "global_batch": global_batch, "scaling": scaling, "cond_scale": cond_scale, "forwards_per_step": fwd,
            "cfg_batched": bool(cfg_batched), "timed_steps": steps, "whole_step_tflops_per_gpu": tf,
            "whole_step_frac": tf / peak_tf if tf else None, "finite": ok,
            "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 2 ** 30}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch-gpu"])
    ap.add_argument("--workload", default="cfg3")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-torch-gpu", action="store_true")
    ap.add_argument("--train-batch", type=int, default=8, help="batch of the informational training_step row")
    ap.add_argument("--secondary", default="cfg1,cfg2a,cfg2b,cfg4,cfg5,train", help="comma list of secondary configurations")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--fuse", default=None, choices=["off", "pair", "on", "all"], help="fused GroupNorm+conv kernel usage")
    ap.add_argument("--kernel-table", default=None, help="write a CUPTI per-kernel time table of 3 steps to this path")
    ap.add_argument("--pdl", type=int, default=None, help="programmatic dependent launch on (1) / off (0)")
    ap.add_argument("--profiler-range", action="store_true",
                    help="cudaProfilerStart/Stop around the timed steps (for `ncu --profile-from-start off`: launch lists of exactly K steps)")
    ap.add_argument("--gn-f16", action="store_true", help="GroupNorm inputs in fp16 (faster, 1.05e-3 instead of 9e-4 rel-L2)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the output of the last timed step to DIR/image.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = workload(args.workload)
    wl["name"] = args.workload
    if args.batch:
        wl["batch"] = args.batch
    B = wl["batch"]
    config = {"workload": f"{args.workload}: {wl['desc']}", "batch_per_gpu": B, "global_batch": B * world,
              "image_size": wl["size"], "cond_scale": 1.0, "parallelism": f"dp{world} (batch-sharded sampling)",
              "l2": "per-step working set (activations + 1.4 GB fp16 weights) >> 126 MB L2, no explicit flush needed",
              "algorithmic_gflop_per_image_forward": GFLOP_PER_IMG.get(args.workload)}

    # ------------------------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        from minimagen_b200.Unet import Unet
        torch.manual_seed(0)
        sd = Unet(**wl["cfg"]).state_dict()
        base, _ = cpu_baseline(wl, sd, steps=max(1, min(args.steps, 2)), warmup=max(1, min(args.warmup, 1)))
        v = base["value"]
        print(json.dumps({
            "impl": "reference", "metric": METRIC if args.workload == "cfg3" else f"denoising steps/sec ({args.workload})",
            "value": v, "unit": "steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / v, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": base, "gpu_launches": 0,
            "note": "each step is a BOUNDED SAMPLE of the workload (batch 1/2/4 of 32, per-image time scaled x32): the run "
                    "lasts seconds while value/ms_per_step describe the full-batch step it extrapolates to",
            "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    assert torch.cuda.is_available(), "bench.py --impl ours / torch-gpu needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    # ------------------------------------------------------------------------------------ stock PyTorch on the GPU (info)
    if args.impl == "torch-gpu":
        if rank != 0:
            return
        from minimagen_b200.Unet import Unet
        torch.manual_seed(0)
        sd = Unet(**wl["cfg"]).state_dict()
        r = torch_gpu_baseline(wl, sd, dev, B, steps=max(1, min(args.steps, 5)), warmup=max(1, min(args.warmup, 2)))
        v = r.get("fp32", {}).get("steps_per_s")
        print(json.dumps({"impl": "torch-gpu", "metric": METRIC, "value": v, "unit": "steps/s", "n_gpus": 1,
                          "higher_is_better": True, "dtype": "f32 (and f16 autocast)", "data": "synthetic", "config": config,
                          "torch_gpu": r}))
        return

    # ------------------------------------------------------------------------------------ our arm (B200)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from minimagen_b200 import _native, layers
    from minimagen_b200.Imagen import Imagen
    from minimagen_b200.Unet import BaseTest, Unet
    _native.load()
    if args.pdl is not None:
        _native.load().mi_set_launch_mode(int(args.pdl))
    if args.gn_f16:
        layers.GN_INPUT_F32 = False
    if args.fuse is not None:
        layers.FUSE_GN_CONV = {"off": False, "pair": "pair", "on": True, "all": "all"}[args.fuse]
    ops = __import__("minimagen_b200.ops", fromlist=["get_ops"]).get_ops()

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    burst_tf = peaks.get("bf16_tflops") or 1650.0

    def build(wl_, base_cfg=None):
        """Imagen whose LAST U-Net is the one under test.  SR U-Nets sit behind a base stage (Imagen treats unets[0] as
        the base model, Imagen.py:96-101): the real cfg-2a base U-Net for the cascade, else a tiny stand-in never run."""
        torch.manual_seed(0)
        with torch.device(dev):
            u = Unet(**wl_["cfg"]).eval()
            if wl_["lowres"]:
                first = Unet(**(base_cfg if base_cfg is not None else dict(BaseTest.defaults, text_embed_dim=wl_["E"]))).eval()
                stages, sizes = (first, u), (wl_["size"] // 4, wl_["size"])
            else:
                stages, sizes = (u,), (wl_["size"],)
        im = Imagen(unets=stages, text_encoder_name="t5_base" if wl_["E"] == 768 else "t5_small", image_sizes=sizes,
                    timesteps=wl_["T"], cond_drop_prob=0.1).eval().to(dev)
        assert im.unets[-1] is u, "the U-Net under test was re-instantiated"
        return im, u

    want_secondary = (not args.no_secondary) and args.workload == "cfg3"
    sec_list = [s for s in args.secondary.split(",") if s] if want_secondary else []
    imagen, unet = build(wl, base_cfg=dict(text_embed_dim=768) if ("cfg4" in sec_list or "cfg2a" in sec_list) else None)
    sch = imagen.noise_schedulers[-1]
    shape = (B, 3, wl["size"], wl["size"])
    n_img = 3 * wl["size"] * wl["size"]
    inp, ckw = make_cond(wl, B, 1000 + rank, dev, sch, ops)           # each rank owns its own shard of the global batch
    kw = dict(noise_scheduler=sch, cond_scale=1.0, **ckw)
    x_host = inp["x"].pin_memory()
    x = x_host.to(dev)
    T = wl["T"]

    with torch.no_grad():
        # one eager step: packs weights (timed: the load_state_dict-side cost, SURVEY 8f-3), warms the allocator
        t_dev = torch.full((B,), T - 1, dtype=torch.long, device=dev)
        torch.cuda.synchronize()
        tp0 = time.perf_counter()
        imagen._step(unet, x, t_dev, torch.randn(shape, device=dev), **kw)
        torch.cuda.synchronize()
        first_step_s = time.perf_counter() - tp0
        l0 = _native.launch_count
        tp0 = time.perf_counter()
        imagen._step(unet, x, t_dev, torch.randn(shape, device=dev), **kw)
        torch.cuda.synchronize()
        eager_step_s = time.perf_counter() - tp0
        launches_per_step = _native.launch_count - l0
        print(f"[bench] launches/step={launches_per_step}; first step (weight pack + allocator) {first_step_s:.2f} s, "
              f"eager step {eager_step_s * 1e3:.1f} ms", file=sys.stderr, flush=True)

        # per-kernel timing of the dominant kernel (tcgen05 implicit GEMM): CUDA events around every launch of one eager step
        conv = measure_conv_kernels(imagen, unet, x, t_dev, shape, kw, dev)

        # steady state: the captured step, replayed (device-resident inputs, noise drawn inside the graph)
        use_graph = not args.no_graph
        if use_graph:
            g = imagen._step_graph(unet, shape, **kw)
            g.x.copy_(x)
            g.t.fill_(T - 1)
            replay = g.replay
            state = lambda: g.x
        else:
            cur = [x.clone()]

            def replay():
                cur[0] = imagen._step(unet, cur[0], t_dev, torch.randn(shape, device=dev), **kw)
                ops.step_advance_t(t_dev, B)
            state = lambda: cur[0]

        for _ in range(args.warmup):
            replay()
        gathered = None
        if world > 1:
            # warm the collective too (NCCL builds channels / registers buffers on first use)
            gathered = torch.empty((world * B, *shape[1:]), device=dev)
            slot = gathered[rank * B:(rank + 1) * B]
            ops.step_finalize(state().contiguous(), state().numel(), 1, slot)
            dist.all_gather_into_tensor(gathered, slot)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        sampler = ClockSampler(local_rank) if rank == 0 else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        if args.profiler_range:
            torch.cuda.profiler.start()
        e0.record()
        for _ in range(args.steps):
            replay()
        if args.profiler_range:
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        if world > 1:
            ops.step_finalize(state().contiguous(), state().numel(), 1, slot)     # straight into this rank's gather slot
            dist.all_gather_into_tensor(gathered, slot)                            # the path's single collective, in place
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if sampler else None
        assert torch.isfinite(state()).all(), "non-finite output"
        peak_mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30
        print(f"[bench] device-resident: {ms / args.steps:.2f} ms/step", file=sys.stderr, flush=True)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"image": gathered if world > 1 else state()})

        if args.kernel_table and rank == 0:
            kernel_table(lambda: [replay() for _ in range(3)], 3, args.kernel_table)

        # end-to-end: host buffers (pinned) in, result out, every step
        out_host = torch.empty(shape, dtype=torch.float32).pin_memory()
        noise_host = torch.randn(shape).pin_memory()
        t_host = torch.full((B,), T - 1, dtype=torch.long).pin_memory()
        if use_graph:
            imagen.noise_fn = lambda kind, shp, step: noise_host        # only selects the noise-injecting variant of the graph
            g2 = imagen._step_graph(unet, shape, **kw)
            imagen.noise_fn = None

            def e2e_step():
                g2.x.copy_(x_host, non_blocking=True)
                g2.noise.copy_(noise_host, non_blocking=True)
                g2.t.copy_(t_host, non_blocking=True)
                g2.replay()
                out_host.copy_(g2.x, non_blocking=True)
                torch.cuda.synchronize()
        else:
            def e2e_step():
                r = imagen._p_sample(unet, x_host.to(dev, non_blocking=True), t_host.to(dev, non_blocking=True),
                                     noise=noise_host.to(dev, non_blocking=True), **kw)
                out_host.copy_(r, non_blocking=True)
                torch.cuda.synchronize()
        for _ in range(3):
            e2e_step()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e2e_steps = min(args.steps, 50)
        t0 = time.perf_counter()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(e2e_steps):
            e2e_step()
        f1.record()
        torch.cuda.synchronize()
        e2e_ms = max(f0.elapsed_time(f1), (time.perf_counter() - t0) * 1000.0) / e2e_steps

    ms = max_over_ranks(ms, world, dev)
    e2e_ms = max_over_ranks(e2e_ms, world, dev)

    # ------------------------------------------------------------------------------------ secondary configurations
    secondary = {}
    if sec_list:
        imagen.clear_graphs()
        torch.cuda.empty_cache()
        common = dict(world=world, rank=rank, dev=dev, peak_tf=peak_tf)

        def guarded(key, fn, model=None):
            try:
                secondary[key] = fn()
            except Exception as ex:              # a secondary row must never take the headline down
                secondary[key] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
            if model is not None:
                model.clear_graphs()
            torch.cuda.empty_cache()
            print(f"[bench] secondary {key}: {json.dumps(secondary[key])[:300]}", file=sys.stderr, flush=True)

        if "cfg2a" in sec_list:
            w2 = workload("cfg2a")
            guarded("cfg2a", lambda: dict(measure_config(
                imagen, imagen.unets[0], w2, "cfg2a", per_gpu=64, micro=64, cond_scale=1.0, cfg_batched=False, steps=10,
                warmup=3, global_batch=64 * world, scaling="weak", **common), workload=w2["desc"]), imagen)
        if world > 1 and 32 % world == 0:
            # the headline configuration at a FIXED global batch of 32 (strong scaling: 32/N per GPU); at N = 1 it is the headline
            w3s = workload("cfg3")
            guarded("cfg3_strong", lambda: dict(measure_config(
                imagen, imagen.unets[-1], w3s, "cfg3", per_gpu=32 // world, micro=32 // world, cond_scale=1.0, cfg_batched=False,
                steps=10, warmup=3, global_batch=32, scaling="strong", **common), workload=w3s["desc"] + ", global batch 32"), imagen)
        if "cfg4" in sec_list and 128 % world == 0:
            per = 128 // world
            w2, w3 = workload("cfg2a"), workload("cfg3")

            def cascade():
                r = {"workload": "cascade base64 (cfg 2a U-Net) + SR256 (cfg 3 U-Net), classifier-free guidance w=7, GLOBAL "
                                 "batch 128 sharded over the ranks (strong scaling)", "stages": {}}
                for st_name, u_, wl_, mb in (("base64", imagen.unets[0], w2, min(per, 64)), ("sr256", imagen.unets[1], w3, min(per, 32))):
                    rows = {}
                    for batched in (False, True):
                        try:
                            rows["cfg_batched" if batched else "two_forwards"] = measure_config(
                                imagen, u_, wl_, "cfg2a" if st_name == "base64" else "cfg3", per_gpu=per, micro=mb,
                                cond_scale=7.0, cfg_batched=batched, steps=3, warmup=3, global_batch=128,
                                scaling="strong", **common)
                        except Exception as ex:
                            rows["cfg_batched" if batched else "two_forwards"] = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}
                        imagen.clear_graphs()
                        torch.cuda.empty_cache()
                    good = [v for v in rows.values() if "steps_per_s" in v]
                    best = max(good, key=lambda v: v["steps_per_s"]) if good else {}
                    r["stages"][st_name] = dict(rows, best=("cfg_batched" if best is rows.get("cfg_batched") else "two_forwards"),
                                                steps_per_s=best.get("steps_per_s"), ms_per_step=best.get("ms_per_step"),
                                                whole_step_frac=best.get("whole_step_frac"))
                ms_pair = sum(v["ms_per_step"] for v in r["stages"].values() if v.get("ms_per_step"))
                r["cascade_steps_per_s"] = 1000.0 / ms_pair if ms_pair else None     # one base step + one SR step (T each)
                r["note"] = ("both stages run T=1000 steps: cascade throughput = 1 / (base ms/step + SR ms/step); per-GPU batch "
                             f"{per} as micro-batches of <= 64 (base) / 32 (SR)")
                return r
            guarded("cfg4", cascade, imagen)
        # the remaining rows need their own models: release the headline model first
        del imagen, unet
        if use_graph:
            del g, g2, replay, state, e2e_step
        torch.cuda.empty_cache()
        for key in ("cfg2b", "cfg1", "cfg5"):
            if key not in sec_list:
                continue
            wk = workload(key)
            if key == "cfg5" and 16 % world != 0:
                continue

            def run(key=key, wk=wk):
                im_, u_ = build(wk)
                try:
                    if key == "cfg5":
                        per = 16 // world
                        r = measure_config(im_, u_, wk, key, per_gpu=per, micro=min(per, 2), cond_scale=1.0, cfg_batched=False,
                                           steps=3, warmup=3, global_batch=16, scaling="strong", **common)
                    elif key == "cfg1":
                        r = measure_config(im_, u_, wk, key, per_gpu=2, micro=2, cond_scale=1.0, cfg_batched=False, steps=10,
                                           warmup=3, global_batch=2 * world, scaling="weak", **common)
                    else:
                        r = measure_config(im_, u_, wk, key, per_gpu=64, micro=64, cond_scale=1.0, cfg_batched=False,
                                           steps=10, warmup=3, global_batch=64 * world, scaling="weak", **common)
                    r["workload"] = wk["desc"]
                    r["params_m"] = sum(p.numel() for p in u_.parameters()) / 1e6
                    return r
                finally:
                    im_.clear_graphs()
                    del im_, u_
            guarded(key, run)

    if sec_list and "train" in sec_list and rank == 0:
        # informational: one training step (Imagen.forward -> loss.backward()) through the autograd Functions / backward kernels
        def train_step():
            from minimagen_b200.Unet import Unet as U2
            tcfg = dict(dim=128, dim_mults=(1, 2, 4), num_resnet_blocks=(1, 2, 2), layer_attns=(False, False, True),
                        layer_cross_attns=(False, True, True), memory_efficient=True, text_embed_dim=768)
            torch.manual_seed(0)
            with torch.device(dev):
                tu = U2(**tcfg)
            tim = Imagen(unets=tu, text_encoder_name="t5_base", image_sizes=(64,), timesteps=1000, cond_drop_prob=0.1).to(dev).train()
            gg = torch.Generator().manual_seed(3)
            tb = args.train_batch
            imgs = torch.rand(tb, 3, 64, 64, generator=gg).to(dev)
            te = torch.randn(tb, 16, 768, generator=gg).to(dev)
            tm = torch.ones(tb, 16, dtype=torch.bool, device=dev)
            opt = torch.optim.Adam(tu.parameters(), lr=1e-4)
            def one():
                opt.zero_grad(set_to_none=True)
                loss = tim(imgs, text_embeds=te, text_masks=tm, unet_number=1)
                loss.backward()
                opt.step()
                return loss
            for _ in range(2):
                one()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                loss = one()
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / 3
            row = {"ms_per_training_step": dt * 1e3, "batch": tb, "loss": float(loss.detach()), "params_m": sum(p.numel() for p in tu.parameters()) / 1e6,
                   "workload": f"base U-Net dim 128, mults (1,2,4), 64x64, b={tb}: Imagen.forward + backward + Adam step (eager; convs and the "
                               "attention projections forward, data gradient and weight gradient on tcgen05 with fp16 operands; GroupNorm / "
                               "LayerNorm / attention-core backward fp32)"}
            del loss        # a live loss keeps the parameters' gradient accumulators (bound to the default stream) alive: not capturable
            import gc
            gc.collect()
            try:        # the same step captured in one CUDA graph (Imagen.graphed_train_step): the eager step is host-launch-bound
                gopt = torch.optim.Adam(tu.parameters(), lr=1e-4, capturable=True)   # (tim.unets is a plain list after a training forward, like the reference)
                gstep = tim.graphed_train_step(gopt, imgs, text_embeds=te, text_masks=tm, unet_number=1)
                for _ in range(2):
                    gstep(imgs, te, tm)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(10):
                    gstep(imgs, te, tm)
                torch.cuda.synchronize()
                row["ms_per_training_step_graphed"] = (time.perf_counter() - t0) / 10 * 1e3
                del gstep, gopt
            except Exception as ex:
                import traceback
                traceback.print_exc(file=sys.stderr)
                row["graphed_error"] = f"{type(ex).__name__}: {str(ex)[:200]}"
                torch.cuda.synchronize()
            if not args.no_torch_gpu:
                # the same U-Net (same weights) trained by stock PyTorch on this GPU: restatement forward -> autograd -> Adam
                try:
                    from oracle import restatement as R
                    sd = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point) for k, v in tu.state_dict().items()}
                    leaves = [v for v in sd.values() if v.requires_grad]
                    topt = torch.optim.Adam(leaves, lr=1e-4, capturable=True)
                    tt = torch.randint(0, 1000, (tb,), generator=gg).to(dev)
                    xin, tgt = torch.randn(tb, 3, 64, 64, generator=gg).to(dev), torch.randn(tb, 3, 64, 64, generator=gg).to(dev)
                    for name, dt_ in (("fp32", None), ("fp16_autocast", torch.float16)):
                        scaler = torch.amp.GradScaler("cuda", enabled=dt_ is not None)
                        def tone():
                            topt.zero_grad(set_to_none=True)
                            with torch.autocast("cuda", dtype=dt_ or torch.float16, enabled=dt_ is not None):
                                pred = R.unet_forward(sd, tcfg, xin, tt, text_embeds=te, text_mask=tm)
                            l_ = torch.nn.functional.mse_loss(pred.float(), tgt)
                            scaler.scale(l_).backward()
                            scaler.step(topt)
                            scaler.update()
                        for _ in range(2):
                            tone()
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        for _ in range(3):
                            tone()
                        torch.cuda.synchronize()
                        row[f"torch_gpu_{name}_ms_per_training_step"] = (time.perf_counter() - t0) / 3 * 1e3
                        if dt_ is None:
                            try:        # and stock PyTorch's step captured the same way (no GradScaler in the graph: fp32 arm only)
                                def tcap():
                                    pred = R.unet_forward(sd, tcfg, xin, tt, text_embeds=te, text_mask=tm)
                                    torch.nn.functional.mse_loss(pred, tgt).backward()
                                    topt.step()
                                sdst = torch.cuda.Stream()
                                sdst.wait_stream(torch.cuda.current_stream())
                                with torch.cuda.stream(sdst):
                                    for _ in range(2):
                                        topt.zero_grad(set_to_none=True)
                                        tcap()
                                torch.cuda.current_stream().wait_stream(sdst)
                                torch.cuda.synchronize()
                                tg = torch.cuda.CUDAGraph()
                                topt.zero_grad(set_to_none=True)
                                with torch.cuda.graph(tg):
                                    tcap()
                                tg.replay()
                                torch.cuda.synchronize()
                                t0 = time.perf_counter()
                                for _ in range(10):
                                    tg.replay()
                                torch.cuda.synchronize()
                                row["torch_gpu_fp32_ms_per_training_step_graphed"] = (time.perf_counter() - t0) / 10 * 1e3
                                del tg
                            except Exception as ex:
                                row["torch_gpu_graphed_error"] = f"{type(ex).__name__}: {str(ex)[:200]}"
                except Exception as ex:
                    row["torch_gpu_error"] = f"{type(ex).__name__}: {str(ex)[:200]}"
            return row
        guarded("training_step", train_step)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * args.steps / (ms / 1000.0)
    step_tflops = (value * B * GFLOP_PER_IMG.get(args.workload, 0.0)) / 1000.0 / world    # per GPU
    d = conv["dominant"]
    a = conv["all"]
    d_achieved = d["alg_flops"] / (d["ms"] / 1000.0) / 1e12 if d["ms"] > 0 else 0.0
    a_achieved = a["alg_flops"] / (a["ms"] / 1000.0) / 1e12 if a["ms"] > 0 else 0.0
    traffic, traffic_src = None, None
    for cand in ("r02_dominant_dram.json",):
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", cand)))
            if args.workload == "cfg3" and B == 32 and prof.get("launches") == d["n"]:
                traffic, traffic_src = prof["dram_bytes_per_launch"], cand
        except Exception:
            pass
    ms_step = ms / args.steps
    roofline = {"bound": "tensor",
                "kernel": conv["dominant_name"],
                # launches are timed one by one with CUDA events inside an eager step (idle gaps between launches: not the
                # power-capped regime of the graph-replayed step) -> the BURST cuBLAS figure is the matching denominator
                "achieved": d_achieved, "peak": burst_tf, "unit": "TFLOP/s", "frac": d_achieved / burst_tf,
                "frac_of_sustained_peak": d_achieved / peak_tf,
                "traffic": traffic,
                "traffic_unit": f"DRAM bytes per launch (ncu, profiles/{traffic_src})" if traffic_src else
                                "null: no committed ncu DRAM capture matches this build's launch count",
                "algorithmic_flops_per_launch": d["alg_flops"] / d["n"] if d["n"] else None,
                "executed_flops_per_launch": d["exe_flops"] / d["n"] if d["n"] else None,
                "algorithmic_bytes_per_launch": d["bytes"] / d["n"] if d["n"] else None,
                "flops_note": "algorithmic = the reference's conv FLOPs (stem 3/7/15 kernels on 6 channels, 3x3 conv on the "
                              "up-sampled grid, 3 real output channels of final_conv); executed = what the lowering issues "
                              "(15x1 over the 128-wide unrolled stem operand, 4/9 for the sub-pixel up-sampling convs, N padded "
                              "to 16 in final_conv)",
                "launches_timed": d["n"], "kernel_ms_per_launch": d["ms"] / d["n"] if d["n"] else None,
                "kernel_ms_per_step": d["ms"], "kernel_share_of_step": d["ms"] / ms_step if ms else None,
                "all_conv_launches": {"achieved": a_achieved, "frac": a_achieved / burst_tf, "launches": a["n"],
                                      "ms_per_step": a["ms"], "share_of_step": a["ms"] / ms_step if ms else None,
                                      "algorithmic_tflop_per_step": a["alg_flops"] / 1e12,
                                      "executed_tflop_per_step": a["exe_flops"] / 1e12},
                "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst, kernel timed alone) for `frac`; bf16_tflops_sustained "
                               "(kernel inside a long step) for `whole_step_frac` and `frac_of_sustained_peak`"
                               if peaks else "fallback 1.65 / 1.4 PFLOP/s (B200_PROFILING.md)",
                "whole_step_tflops_per_gpu": step_tflops, "whole_step_frac": step_tflops / peak_tf,
                "whole_step_peak": peak_tf}
    result = {
        "metric": METRIC if args.workload == "cfg3" else f"denoising steps/sec ({args.workload})",
        "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 tensor-core operands, f32 accumulate / residual stream", "data": "synthetic", "config": config,
        "gpu_launches": launches_per_step * args.steps,
        "e2e": {"value": world * 1000.0 / e2e_ms, "unit": "steps/s", "steps": e2e_steps,
                "h2d_bytes_per_step": int(x_host.numel() * 4 + noise_host.numel() * 4 + t_host.numel() * 8),
                "d2h_bytes_per_step": int(out_host.numel() * 4)},
        "roofline": roofline,
        "clocks": clocks, "cuda_graph": use_graph, "launches_per_step": launches_per_step,
        "fused_gn_conv": layers.FUSE_GN_CONV, "gn_input": "f32" if layers.GN_INPUT_F32 else "f16",
        "peak_mem_gb": peak_mem,
        "weight_ingestion": {"first_step_s": first_step_s, "eager_step_s": eager_step_s,
                             "note": "first step = lazy fp16 weight pack of all layers (checkpoint fp32 (C_out,C_in,kh,kw) -> "
                                     "tensor-core layout, mi_pack_conv_weight_f16) + allocator warm-up; paid once per load_state_dict"},
    }
    if secondary:
        result["secondary"] = secondary
    torch.cuda.empty_cache()
    sd = None
    if not args.no_torch_gpu or not args.no_cpu_baseline:
        torch.manual_seed(0)
        sd = Unet(**wl["cfg"]).state_dict()
    if not args.no_torch_gpu and world == 1:
        result["torch_gpu"] = torch_gpu_baseline(wl, sd, dev, B)
    if not args.no_cpu_baseline:
        base, _ = cpu_baseline(wl, sd)
        result["cpu_baseline"] = base
    print(json.dumps(result))
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Each array as <path>/<name>.npy in float32.  An array beyond DUMP_BYTES is written as a fixed seeded sample of
    its elements (flat, in index order), the same sample on every run."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() * 4 > DUMP_BYTES:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_BYTES // 4].sort().values
            t = t.flatten()[idx.to(t.device)]
        np.save(os.path.join(path, f"{name}.npy"), t.cpu().numpy())


def kernel_table(fn, steps, path):
    """Diagnostics only (never a bench value): CUPTI kernel records of `steps` un-serialised steps, summed per kernel, plus
    the idle gaps between consecutive kernels (start of the next minus end of the previous) attributed to the PRECEDING kernel."""
    import collections
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        fn()
        torch.cuda.synchronize()
    agg = collections.defaultdict(lambda: [0, 0.0])
    recs = []
    for ev in prof.events():
        if ev.device_type is not None and str(ev.device_type).endswith("CUDA"):
            a = agg[ev.name[:110]]
            a[0] += 1
            dur = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
            a[1] += dur
            try:
                recs.append((ev.time_range.start, ev.time_range.start + dur, ev.name[:70]))
            except Exception:
                pass
    tot = sum(t for _, t in agg.values())
    with open(path, "w") as f:
        f.write(f"# per-step kernel time (CUPTI, {steps} steps averaged), total {tot / steps / 1e3:.3f} ms/step\n")
        for name, (c, t) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write(f"{t / steps / 1e3:9.3f} ms {c / steps:7.1f} launches  {name}\n")
        if len(recs) > 2:
            recs.sort()
            gaps = collections.defaultdict(lambda: [0, 0.0])
            span = recs[-1][1] - recs[0][0]
            for (s0, e0, n0), (s1, e1, n1) in zip(recs, recs[1:]):
                g = max(0.0, s1 - e0)
                gaps[n0][0] += 1
                gaps[n0][1] += g
            gtot = sum(v[1] for v in gaps.values())
            f.write(f"# idle gaps between consecutive kernels: {gtot / steps / 1e3:.3f} ms/step of a {span / steps / 1e3:.3f} ms/step "
                    f"span; by preceding kernel (total ms/step, mean us per boundary):\n")
            for name, (c, t) in sorted(gaps.items(), key=lambda kv: -kv[1][1])[:12]:
                f.write(f"#   {t / steps / 1e3:7.3f} ms  {t / max(c, 1):6.2f} us x {c / steps:6.1f}  after {name}\n")


def measure_conv_kernels(imagen, unet, x, t_dev, shape, kw, dev):
    """Run one eager step with CUDA events around every tcgen05 conv launch.  Returns totals over all conv launches and,
    separately, over the launches of the dominant kernel family (conv3x3_halo_t_kernel / its fused-GroupNorm form: 3x3 / 15x1
    stride-1 convs with C_out % 128 == 0 on a 32x8- or 16x16-tileable grid -- the selection rule of csrc/conv_tc.cu).
    FLOPs are counted twice: ALGORITHMIC (what the reference's conv computes) and EXECUTED (what the lowering issues)."""
    from minimagen_b200 import ops as ops_mod
    real = ops_mod.get_ops()
    events = []
    stem = unet.init_conv
    stem_alg_per_pixel = sum(2.0 * c.kernel_size[0] ** 2 * c.in_channels * c.out_channels for c in stem.convs)

    def is_halo_t(H, W, c_out, kh, kw_, mode):
        if 2 <= mode <= 5:          # sub-pixel phase on the swapped-operand kernel's Sub geometry
            return c_out % 128 == 0 and H % 32 == 0 and W % 8 == 0 and W != 16 and not os.environ.get("MI_SUBPIX_PAIR")
        return (mode == 0 and (kh, kw_) in ((3, 3), (15, 1)) and c_out % 128 == 0 and
                ((W == 16 and H % 16 == 0 and kh == 3) or (H % 32 == 0 and W % 8 == 0 and W != 16)))

    class Timed(type(real)):
        def conv_igemm(self, act, B, H, W, lda, c_off, c_in, wp, c_out, kh, kw_, mode, bias, residual, out_f32, out_f16,
                       *a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            super().conv_igemm(act, B, H, W, lda, c_off, c_in, wp, c_out, kh, kw_, mode, bias, residual, out_f32, out_f16,
                               *a, **k)
            e.record()
            n_valid = k.get("n_valid", 0) or c_out
            px = B * H * W
            exe = 2.0 * px * c_out * kh * kw_ * c_in
            if (kh, kw_) == (15, 1) and c_in == 128:
                alg = px * stem_alg_per_pixel                              # CrossEmbedLayer: k=3/7/15 on the real channels
            elif 2 <= mode <= 5:
                alg = 2.0 * px * 9 * c_in * c_out                          # this phase's share of the 3x3 conv on the 2H x 2W grid
            else:
                alg = 2.0 * px * n_valid * kh * kw_ * c_in
            mn = px * c_out
            nbytes = (px * c_in * 2 * (4 if mode == 6 else 1) + c_out * kh * kw_ * c_in * 2 +
                      (4 * mn if residual is not None else 0) + (4 * mn if out_f32 is not None else 0) +
                      (2 * mn if out_f16 is not None else 0))
            events.append((s, e, alg, exe, nbytes, is_halo_t(H, W, c_out, kh, kw_, mode)))

        def conv_res1x1(self, act, B, H, W, lda, c_in, act2, lda2, c_in1, x, ldx, x_cin, x2, ldx2, x_cin1, wp, c_out, bias,
                        residual, out_f32, out_f16, out_stats):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            super().conv_res1x1(act, B, H, W, lda, c_in, act2, lda2, c_in1, x, ldx, x_cin, x2, ldx2, x_cin1, wp, c_out, bias,
                                residual, out_f32, out_f16, out_stats)
            e.record()
            px = B * H * W
            fl = 2.0 * px * c_out * (9 * c_in + x_cin)               # the 3x3 conv plus the folded 1x1 res_conv
            mn = px * c_out
            nbytes = (px * (c_in + x_cin) * 2 + c_out * (9 * c_in + x_cin) * 2 + (4 * mn if residual is not None else 0) +
                      (4 * mn if out_f32 is not None else 0) + (2 * mn if out_f16 is not None else 0))
            events.append((s, e, fl, fl, nbytes, True))

        def conv_gn(self, src0, c0, src1, c1, scale1, B, H, W, groups, stats0, stats1, gamma, beta, scale_shift, ss_ld,
                    eps, wp, c_out, bias, residual, out_f32, out_f16, out_stats, *a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            super().conv_gn(src0, c0, src1, c1, scale1, B, H, W, groups, stats0, stats1, gamma, beta, scale_shift, ss_ld,
                            eps, wp, c_out, bias, residual, out_f32, out_f16, out_stats, *a, **k)
            e.record()
            px, c_in = B * H * W, c0 + c1
            fl = 2.0 * px * c_out * 9 * c_in
            mn = px * c_out
            nbytes = (px * c_in * 4 + c_out * 9 * c_in * 2 + (4 * mn if residual is not None else 0) +
                      (4 * mn if out_f32 is not None else 0) + (2 * mn if out_f16 is not None else 0))
            events.append((s, e, fl, fl, nbytes, True))

    ops_mod.set_ops(Timed())
    streams = unet.batch_streams
    unet.batch_streams = 1            # one stream: every launch is timed alone, not while sharing SMs with the other half
    try:
        imagen._step(unet, x, t_dev, torch.randn(shape, device=dev), **kw)
        torch.cuda.synchronize()
    finally:
        ops_mod.set_ops(real)
        unet.batch_streams = streams
    zero = lambda: {"ms": 0.0, "alg_flops": 0.0, "exe_flops": 0.0, "n": 0, "bytes": 0.0}
    res = {"all": zero(), "dominant": zero()}
    for s, e, alg, exe, nb, dom in events:
        ms = s.elapsed_time(e)
        for key in (("all", "dominant") if dom else ("all",)):
            r = res[key]
            r["ms"] += ms; r["alg_flops"] += alg; r["exe_flops"] += exe; r["n"] += 1; r["bytes"] += nb
    res["dominant_name"] = ("conv3x3_halo_t_kernel family (tcgen05 swapped-operand halo conv: 3x3, 3x3 + folded 1x1 res_conv, 15x1 "
                            "stem, 2x2 sub-pixel phases; incl. the fused GroupNorm-prologue form when enabled)")
    if res["dominant"]["n"] == 0:
        res["dominant"] = res["all"]
        res["dominant_name"] = "tcgen05 implicit-GEMM convolutions (all launches)"
    return res


if __name__ == "__main__":
    main()
