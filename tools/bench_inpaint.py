#!/usr/bin/env python
"""Overhead of inpainting on the captured sampling step (DESIGN.md 4.6), on one GPU.

    python tools/bench_inpaint.py [--workloads cfg3,cfg1] [--rounds 3] [--replays 100] [--U 5] [--out FILE]

For each workload (bench.py's definitions; cfg 3 = SR U-Net 64->256, b=32, cond_scale 1; cfg 1 = tiny base U-Net, b=2):
  * captures the plain step graph and the inpainting step graph (step + 2 extra in-graph normal draws + mi_inpaint_blend +
    mi_inpaint_advance) over the same weights and conditioning, warms both, then times them alternately (A, B, A, B, ...)
    for `rounds` rounds of `replays` replays between CUDA events; reports ms per step of each and the difference;
  * times blend + advance alone with CUDA events: 100 back-to-back launch pairs (working set L2-resident), and 100 pairs
    each preceded by a 512 MB write that evicts L2 (each pair timed on its own, the flush outside the events); achieved
    GB/s uses the blend's traffic bound: x, known, z_known and z_renoise read, x written (5 image-sized fp32 tensors) plus
    the uint8 mask -- the kernel reads only one of the known/noise pairs per pixel, so this over-counts what it moves;
  * records the device name and power limit (read-only nvidia-smi query) in the same run.
Prints one JSON line (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload / synth_inputs / make_cond: the configurations bench.py times)

HBM_TBPS = 7.7          # HGX B200 data sheet, one GPU


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(index)],
                       capture_output=True, text=True)
    name, limit = (q.stdout.strip().split(", ") + ["?", "?"])[:2] if q.returncode == 0 else (torch.cuda.get_device_name(), "?")
    return {"device": name, "power_limit": limit}


def blob_mask(b, s, seed):
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(s), torch.arange(s), indexing="ij")
    m = []
    for _ in range(b):
        cy, cx = (torch.rand(2, generator=g) * 0.5 + 0.25) * s
        r = (0.15 + 0.15 * torch.rand((), generator=g)) * s
        m.append(((yy - cy) ** 2 + (xx - cx) ** 2) > r * r)
    return torch.stack(m).to(torch.uint8)


def build(wl, dev):
    """bench.py's model under test: SR U-Nets sit behind a tiny stand-in base stage that is never run."""
    from minimagen_b200.Imagen import Imagen
    from minimagen_b200.Unet import BaseTest, Unet
    torch.manual_seed(0)
    with torch.device(dev):
        u = Unet(**wl["cfg"]).eval()
        if wl["lowres"]:
            stages, sizes = (Unet(**dict(BaseTest.defaults, text_embed_dim=wl["E"])).eval(), u), (wl["size"] // 4, wl["size"])
        else:
            stages, sizes = (u,), (wl["size"],)
    im = Imagen(unets=stages, text_encoder_name="t5_base" if wl["E"] == 768 else "t5_small", image_sizes=sizes,
                timesteps=wl["T"], cond_drop_prob=0.1).eval().to(dev)
    assert im.unets[-1] is u
    return im, u


def time_replays(g, n, T):
    g.t.fill_(T - 1)
    if g.u is not None:
        g.u.zero_()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def measure(name, U, rounds, replays, dev):
    from minimagen_b200.ops import get_ops
    ops = get_ops()
    wl = bench.workload(name)
    B, s, T = wl["batch"], wl["size"], wl["T"]
    im, u = build(wl, dev)
    sch = im.noise_schedulers[-1]
    shape = (B, 3, s, s)
    _, kw = bench.make_cond(wl, B, 2000, dev, sch, ops)
    known = (bench.synth_inputs(wl, B, 7)["x"].clamp(-1, 1)).to(dev).contiguous()       # normalised image in [-1, 1]
    mask = blob_mask(B, s, 8).to(dev)
    res = {"workload": f"{name}: {wl['desc']}", "batch": B, "image": [3, s, s], "cond_scale": 1.0, "U": U}
    with torch.no_grad():
        plain = im._step_graph(u, shape, noise_scheduler=sch, cond_scale=1.0, **kw)
        inp = im._step_graph(u, shape, noise_scheduler=sch, cond_scale=1.0, inpaint=(known, mask, U), **kw)
        for g in (plain, inp):
            g.x.normal_()
            time_replays(g, 5, T)
        ms = {"plain": [], "inpaint": []}
        for _ in range(rounds):
            for key, g in (("plain", plain), ("inpaint", inp)):
                g.x.normal_()
                ms[key].append(time_replays(g, replays, T))
        finite = bool(torch.isfinite(plain.x).all()) and bool(torch.isfinite(inp.x).all())

        # blend + advance alone, on the inpainting graph's static buffers
        sa, sb = sch.inpaint_tables(dev)
        tabs = (sch.sqrt_alphas_cumprod, sch.sqrt_one_minus_alphas_cumprod, sa, sb)
        x, t, uu = inp.x, inp.t, inp.u

        def pair():
            ops.inpaint_blend(x, inp.known, inp.mask, inp.z_known, inp.z_renoise, t, uu, U, 0, *tabs)
            ops.inpaint_advance(t, uu, U, B)
        t.fill_(T - 1)
        uu.zero_()
        for _ in range(10):
            pair()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(100):
            pair()
        e1.record()
        torch.cuda.synchronize()
        hot_us = e0.elapsed_time(e1) * 1000 / 100
        flush = torch.empty(512 * 2 ** 20 // 4, dtype=torch.float32, device=dev)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(100)]
        for a, b in ev:
            flush.fill_(1.0)
            a.record()
            pair()
            b.record()
        torch.cuda.synchronize()
        cold = sorted(a.elapsed_time(b) * 1000 for a, b in ev)
        cold_us = cold[len(cold) // 2]
    n_img = B * 3 * s * s
    nbytes = 5 * 4 * n_img + B * s * s
    mp, mi = min(ms["plain"]), min(ms["inpaint"])
    res.update({
        "ms_per_step_plain": ms["plain"], "ms_per_step_inpaint": ms["inpaint"], "rounds": rounds, "replays_per_round": replays,
        "ms_per_step_plain_best": mp, "ms_per_step_inpaint_best": mi, "delta_ms": mi - mp,
        "delta_pct": 100.0 * (mi - mp) / mp, "finite": finite,
        "blend_advance_bytes_bound": nbytes,
        "blend_advance_us_l2_hot": hot_us, "blend_advance_us_l2_flushed_median": cold_us,
        "blend_gbps_l2_flushed": nbytes / (cold_us * 1e3), "blend_frac_of_hbm_l2_flushed": nbytes / (cold_us * 1e3) / (HBM_TBPS * 1e3),
        "blend_gbps_l2_hot": nbytes / (hot_us * 1e3),
    })
    im.clear_graphs()
    del im, u, plain, inp
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg3,cfg1")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replays", type=int, default=100)
    ap.add_argument("--U", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tools/bench_inpaint.py measures on a CUDA device"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    from minimagen_b200 import _native
    _native.load()
    out = {"tool": "tools/bench_inpaint.py", **gpu_info(0), "hbm_tbps_datasheet": HBM_TBPS,
           "results": [measure(w, args.U, args.rounds, args.replays, dev) for w in args.workloads.split(",") if w]}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
