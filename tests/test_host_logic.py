"""Host-side logic on CPU: the class surfaces / checkpoint ABI mirror the reference, and the orchestration in
minimagen_b200/{layers,Unet,Imagen}.py -- executed through the torch EMULATION of the ops interface (tests/emu_ops.py)
-- reproduces the reference's outputs.  (The emulation rounds tensor-core operands to fp16 like the kernels do, hence
the 2e-3 bound; the tiny config runs its convolutions in fp32 and lands near 2e-4.)"""
import ast
import json
import os

import pytest
import torch

from conftest import GOLDEN, load_golden, rel_l2
from oracle import make_golden as MG, restatement as R


def _mine(cfg, sd):
    from minimagen_b200.Unet import Unet
    u = Unet(**cfg).eval()
    u.load_state_dict(sd)
    return u


@pytest.mark.parametrize("name", ["unet_tiny_base.pt", "unet_tiny_sr.pt"])
def test_state_dict_abi_matches_reference_checkpoint(name):
    from minimagen_b200.Unet import Unet
    g = load_golden(name)
    u = Unet(**g["cfg"])
    mine = u.state_dict()
    assert list(mine.keys()) == list(g["state_dict"].keys())          # same keys, same order
    for k, v in g["state_dict"].items():
        assert mine[k].shape == v.shape and mine[k].dtype == v.dtype, k
    assert not u.load_state_dict(g["state_dict"]).missing_keys


@pytest.mark.parametrize("name", ["unet_tiny_base.pt", "unet_tiny_sr.pt"])
def test_unet_forward_orchestration_vs_golden(emu, name):
    g = load_golden(name)
    u = _mine(g["cfg"], g["state_dict"])
    inp = g["inputs"]
    kw = {k: v for k, v in inp.items() if k not in ("x", "time")}
    with torch.no_grad():
        assert rel_l2(u(inp["x"], inp["time"], **kw), g["out_cond"]) < 1e-3
        assert rel_l2(u(inp["x"], inp["time"], cond_drop_prob=1., **kw), g["out_null"]) < 1e-3
        assert rel_l2(u(inp["x"], inp["time"], **dict(kw, text_mask=None)), g["out_nomask"]) < 1e-3
        assert rel_l2(u.forward_with_cond_scale(inp["x"], inp["time"], cond_scale=3., **kw), g["out_cfg3"]) < 1e-3
    assert "conv_direct" in emu.calls and "attention" in emu.calls


def test_static_text_projection_cache(emu):
    """Unet.register_static_text: the step-invariant text_to_cond projection is computed once per registered (static) text
    buffer and reused by forward -- same output; an in-place change of the buffer without re-registering misses the cache
    (the projection is recomputed inside forward), re-registering hits it again."""
    g = load_golden("unet_tiny_base.pt")
    u = _mine(g["cfg"], g["state_dict"])
    inp = g["inputs"]
    kw = {k: v for k, v in inp.items() if k not in ("x", "time")}
    te = kw["text_embeds"].clone().float().contiguous()
    kw["text_embeds"] = te
    with torch.no_grad():
        ref = u(inp["x"], inp["time"], **kw)
        n_lin = emu.calls.count("linear_f32")
        u.register_static_text(te)
        emu.calls.clear()
        hit = u(inp["x"], inp["time"], **kw)
        assert torch.equal(hit, ref) and emu.calls.count("linear_f32") == n_lin - 1          # one projection fewer in the step
        te.mul_(0.5)                                                                             # modified, not re-registered
        emu.calls.clear()
        miss = u(inp["x"], inp["time"], **kw)
        assert emu.calls.count("linear_f32") == n_lin and not torch.equal(miss, ref)
        u.register_static_text(te)
        emu.calls.clear()
        assert torch.equal(u(inp["x"], inp["time"], **kw), miss) and emu.calls.count("linear_f32") == n_lin - 1
        u.unregister_static_text(te)
        assert u._static_text_proj(te) is None


@pytest.mark.parametrize("cfg,s,lowres", [
    (dict(dim=64, dim_mults=(1, 2), attend_at_middle=True, text_embed_dim=768), 32, False),
    (dict(dim=64, dim_mults=(1, 2, 4), num_resnet_blocks=(1, 2, 2), layer_attns=(False, False, True),
          layer_cross_attns=(False, True, True), lowres_cond=True, memory_efficient=True), 32, True),
])
def test_unet_forward_tensor_core_shaped_configs(emu, cfg, s, lowres):
    """Channel counts that route through conv_igemm / fp16 operands (vs the bit-exact-pinned restatement)."""
    from minimagen_b200.Unet import Unet
    torch.manual_seed(0)
    u = Unet(**cfg).eval()
    sd = u.state_dict()
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 3, s, s, generator=g)
    te = torch.randn(2, 20, cfg.get("text_embed_dim", 512), generator=g)
    tm = torch.ones(2, 20, dtype=torch.bool)
    tm[1, 5:] = False
    kw = dict(text_embeds=te, text_mask=tm)
    if lowres:
        kw.update(lowres_cond_img=torch.randn(2, 3, s, s, generator=g), lowres_noise_times=torch.tensor([200, 3]))
    t = torch.tensor([999, 0])
    with torch.no_grad():
        ref_out = R.unet_forward(sd, cfg, x, t, **kw)
        out = u(x, t, **kw)
    assert emu.calls.count("conv_igemm") > 20
    assert rel_l2(out, ref_out) < 3e-3


def test_step_kernels_contract_vs_golden(emu):
    from minimagen_b200.Imagen import Imagen
    from minimagen_b200.Unet import Unet, BaseTest
    for T in (25, 1000):
        g = load_golden("ddpm_step.pt")[T]
        im = Imagen(unets=Unet(**BaseTest.defaults), text_encoder_name="t5_small", image_sizes=(64,), timesteps=T,
                    cond_drop_prob=0.15)
        sch = im.noise_schedulers[0]
        for k, v in g["tables"].items():
            assert torch.equal(getattr(sch, k), v), k
        with torch.no_grad():
            out = im._step(im.unets[0], g["x"], g["t"], g["noise"], noise_scheduler=sch, text_embeds=None,
                           text_mask=None, lowres_cond_img=None, lowres_noise_times=None, cond_scale=1.,
                           model_output=g["eps"])
            mean, _, logvar = im._p_mean_variance(im.unets[0], g["x"], g["t"], noise_scheduler=sch,
                                                  model_output=g["eps"])
        assert torch.equal(out, g["out"])
        assert torch.equal(mean, g["mean"]) and torch.equal(logvar, g["logvar"])


@pytest.mark.parametrize("graph", [False])
def test_sample_loop_vs_golden(emu, graph):
    from minimagen_b200.Imagen import Imagen
    from minimagen_b200.Unet import Unet
    g = load_golden("sample_loop.pt")
    u = _mine(g["cfg"], g["state_dict"])
    im = Imagen(unets=u, text_encoder_name="t5_small", image_sizes=(64,), timesteps=g["timesteps"],
                cond_drop_prob=0.15).eval()
    im.unets[0].load_state_dict(g["state_dict"])
    im.use_cuda_graph = graph
    draws = {"init": g["x_T"]}
    im.noise_fn = lambda kind, shape, step: g["x_T"] if kind == "init" else g["noises"][g["timesteps"] - 1 - step]
    out = im._p_sample_loop(im.unets[0], (2, 3, 64, 64), noise_scheduler=im.noise_schedulers[0],
                            text_embeds=g["text_embeds"], text_mask=g["text_mask"], cond_scale=g["cond_scale"],
                            max_steps=3)
    expect = (g["traj"][2].clamp(-1, 1) + 1) * 0.5
    assert rel_l2(out, expect) < 2e-3


def test_imagen_surface_and_asserts(emu):
    from minimagen_b200.Imagen import Imagen
    from minimagen_b200.Unet import Unet, Base, Super, BaseTest, SuperTest
    assert BaseTest.defaults["dim"] == 8 and SuperTest.defaults["memory_efficient"] is True
    assert Base.defaults["dim_mults"] == (1, 2, 3, 4) and Super.defaults["num_resnet_blocks"] == (2, 4, 8, 8)
    u0, u1 = Unet(**BaseTest.defaults), Unet(**SuperTest.defaults)
    im = Imagen(unets=(u0, u1), text_encoder_name="t5_small", image_sizes=(32, 64), timesteps=25, cond_drop_prob=0.)
    assert im.unets[0] is u0 and im.unets[1] is not u1 and im.unets[1].lowres_cond      # re-instantiated like the reference
    assert len(im.noise_schedulers) == 2 and im.lowres_noise_schedule.num_timesteps == 25
    sd = im.state_dict()
    assert all(k.startswith("unets.") for k in sd)            # schedule buffers are non-persistent (diffusion_model.py:39)
    with pytest.raises(AssertionError, match="text or text encodings"):
        im.sample()
    with pytest.raises(AssertionError, match="invalid text embedding dimension"):
        im.sample(text_embeds=torch.zeros(1, 4, 7))
    with pytest.raises(AssertionError, match="classifier free guidance"):
        im._step(u0, torch.zeros(1, 3, 32, 32), torch.zeros(1, dtype=torch.long), torch.zeros(1, 3, 32, 32),
                 noise_scheduler=im.noise_schedulers[0], text_embeds=torch.zeros(1, 4, 512), text_mask=None,
                 lowres_cond_img=None, lowres_noise_times=None, cond_scale=3.)
    with pytest.raises(AssertionError, match="at least 20"):
        Imagen(unets=u0, text_encoder_name="t5_small", image_sizes=(32,), timesteps=10)
    with pytest.raises(AssertionError, match="you must specify which unet"):
        im(torch.zeros(1, 3, 64, 64), text_embeds=torch.zeros(1, 4, 512))
    with pytest.raises(AssertionError, match="invalid text embedding dimension"):
        im(torch.zeros(1, 3, 64, 64), text_embeds=torch.zeros(1, 4, 7), unet_number=1)
    loss = im(torch.rand(1, 3, 64, 64), text_embeds=torch.zeros(1, 4, 512), unet_number=1)      # training.py:368
    assert loss.dim() == 0 and loss.requires_grad


def test_signatures_match_reference():
    """Same parameters (name, kind, default) and presets as the reference's, recorded in tests/golden/signatures.json."""
    import minimagen_b200.Unet as MU
    import minimagen_b200.Imagen as MI
    import minimagen_b200.diffusion_model as MD
    with open(os.path.join(GOLDEN, "signatures.json")) as f:
        ref = json.load(f)
    mine = MG.signature_table(MU, MI, MD)
    for key in ("Unet.__init__", "Imagen.__init__", "GaussianDiffusion.__init__", "Unet.forward"):
        assert mine[key] == ref[key], key
    ref_sample = [p[0] for p in ref["Imagen.sample"]]
    assert [p[0] for p in mine["Imagen.sample"]][:len(ref_sample)] == ref_sample
    for cls, text in ref["presets"].items():
        assert getattr(MU, cls).defaults == ast.literal_eval(text), cls
    # training.get_default_args introspection (training.py:660-671) must see the same defaults
    ref_defaults = {name: default for name, _, default in ref["Unet.__init__"]}
    assert {name: default for name, _, default in mine["Unet.__init__"]} == ref_defaults


def test_subpixel_upsample_conv_equals_upsample_then_conv(emu):
    """Upsample (layers.py:502-515: nearest x2 + 3x3 conv) lowered to four 2x2 sub-pixel convs on the low-res tensor:
    same function as the literal composition (fp16 operands either way; the folded weights are rounded once)"""
    from minimagen_b200 import layers
    torch.manual_seed(3)
    conv = layers.Conv2d(64, 128, 3, padding=1)
    x = torch.randn(2, 8, 8, 64)
    ref = torch.nn.functional.conv2d(
        torch.nn.functional.interpolate(x.half().float().permute(0, 3, 1, 2), scale_factor=2, mode="nearest"),
        conv.weight, conv.bias, padding=1).permute(0, 2, 3, 1)
    outs = {}
    for flag in (True, False):
        layers.SUBPIXEL_UPSAMPLE = flag
        try:
            with torch.no_grad():
                act = conv.run(x, upsample=True, f32=True, f16=True, stats=True)
        finally:
            layers.SUBPIXEL_UPSAMPLE = True
        outs[flag] = act
        assert rel_l2(act.f32, ref) < 1e-3
        blk = act.f32.double().reshape(2, 256, 8, 16)
        assert rel_l2(act.stats[:, :, 0], blk.sum(dim=(1, 3))) < 1e-6
        assert rel_l2(act.stats[:, :, 1], (blk * blk).sum(dim=(1, 3))) < 1e-6
    assert "conv_igemm" in emu.calls
    assert rel_l2(outs[True].f32, outs[False].f32) < 1e-3


@pytest.mark.parametrize("n_in,n_out,pad,clamp", MG.RESIZE_CASES)
def test_resize_image_to_vs_reference_helper(emu, n_in, n_out, pad, clamp):
    """helpers.resize_image_to (inter-stage resize, SURVEY.md 8f-1) vs the reference's helper running on the
    resize_right stand-in (published algorithm; the third-party source is not in the container: parity-unpinned).
    The reference's output is stored as a fixed seeded sample of up to 4096 elements plus its full sum
    (tests/golden/resize.pt)."""
    from minimagen_b200 import helpers
    want = load_golden("resize.pt")[(n_in, n_out, pad, clamp)]
    x = MG.resize_input(n_in)
    got = helpers.resize_image_to(x, n_out, clamp_range=clamp, pad_mode=pad)
    assert got.shape == want["shape"] == (2, 3, n_out, n_out)
    assert (got.flatten()[want["idx"].long()] - want["values"]).abs().max().item() < 2e-6
    assert abs(got.double().sum().item() - want["sum"]) < 2e-6 * got.numel()
    assert "resize_separable" in emu.calls
    assert helpers.resize_image_to(x, n_in) is x


def _cascade_from_golden(g, device):
    from minimagen_b200.Imagen import Imagen
    from minimagen_b200.Unet import Unet
    unets = [Unet(**c) for c in g["cfgs"]]
    im = Imagen(unets=unets, text_encoder_name="t5_small", image_sizes=g["image_sizes"], timesteps=g["timesteps"],
                cond_drop_prob=0.1).eval().to(device)
    for u, sd in zip(im.unets, g["state_dicts"]):
        u.load_state_dict(sd)
    it = iter(g["draws"])

    def noise_fn(kind, shape, step):
        d = next(it)
        assert tuple(d.shape) == tuple(shape), (kind, step, d.shape, shape)
        return d
    im.noise_fn = noise_fn
    return im, it


def test_full_cascade_sample_vs_reference_golden(emu):
    """Imagen.sample over a 2-stage cascade (base 16x16 -> SR 32x32, T=25, CFG w=2, lowres noise augmentation and the
    inter-stage resize included) against the unmodified reference's output, replaying the reference's normal draws in
    call order (tests/golden/cascade_tiny.pt, made by oracle/make_golden.py::cascade_case)."""
    g = load_golden("cascade_tiny.pt")
    im, it = _cascade_from_golden(g, "cpu")
    out = im.sample(text_embeds=g["text_embeds"], text_masks=g["text_mask"], cond_scale=g["cond_scale"],
                    lowres_sample_noise_level=g["lowres_noise_level"])
    assert next(it, None) is None                      # every recorded draw was consumed, in the reference's order
    assert out.shape == g["out"].shape
    assert rel_l2(out, g["out"]) < 1e-3
    assert "resize_separable" in emu.calls


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver times next to the GPU arm) prints ONE JSON line with the
    contract's keys; run here on the tiny config so that it finishes in seconds."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "cfg1",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_cfg_as_one_batch_matches_two_forwards(emu):
    """Imagen.cfg_batched: the conditional and unconditional passes of classifier-free guidance as one 2B-sample forward
    (explicit per-sample keep mask, Unet._forward_impl(cond_keep=...)) give the same step as the reference's two forwards
    (Unet.py:474-506, Imagen.py:295-301)."""
    g = load_golden("cascade_tiny.pt")
    outs = []
    for batched in (False, True):
        im, it = _cascade_from_golden(g, "cpu")
        im.cfg_batched = batched
        outs.append(im.sample(text_embeds=g["text_embeds"], text_masks=g["text_mask"], cond_scale=g["cond_scale"],
                              lowres_sample_noise_level=g["lowres_noise_level"]))
    assert rel_l2(outs[1], outs[0]) < 1e-5
    assert rel_l2(outs[1], g["out"]) < 1e-3


def test_fused_groupnorm_conv_orchestration(emu):
    """layers.FUSE_GN_CONV routes Block.forward through conv_gn (one call instead of gn_apply_silu + conv_igemm) wherever
    the geometry allows, with the same result as the un-fused lowering."""
    from minimagen_b200 import layers
    from minimagen_b200.Unet import Unet
    cfg = dict(dim=128, dim_mults=(1, 2), num_resnet_blocks=(1, 1), layer_attns=False, layer_cross_attns=(False, True),
               lowres_cond=True, memory_efficient=True, text_embed_dim=512)
    torch.manual_seed(0)
    u = Unet(**cfg).eval()
    g = torch.Generator().manual_seed(4)
    x = torch.randn(1, 3, 64, 64, generator=g)
    kw = dict(text_embeds=torch.randn(1, 9, 512, generator=g), text_mask=torch.ones(1, 9, dtype=torch.bool),
              lowres_cond_img=torch.randn(1, 3, 64, 64, generator=g), lowres_noise_times=torch.tensor([200]))
    t = torch.tensor([321])
    prev = layers.FUSE_GN_CONV
    try:
        with torch.no_grad():
            layers.FUSE_GN_CONV = False
            a = u(x, t, **kw)
            n_apply = emu.calls.count("gn_apply_silu")
            emu.calls.clear()
            layers.FUSE_GN_CONV = 'all'
            b = u(x, t, **kw)
    finally:
        layers.FUSE_GN_CONV = prev
    assert emu.calls.count("conv_gn") > 0 and emu.calls.count("gn_apply_silu") < n_apply
    assert "conv_res1x1" in emu.calls          # with the fused kernel off, res_conv rides block2's conv (FOLD_RES_CONV)
    # two lowerings = two draws of the fp16 operand-rounding noise: a 1e-7 input perturbation already moves the output of this
    # random-init net by ~1e-3 (measured), so equivalence holds at the operand-rounding tolerance, not bit-wise
    assert rel_l2(b, a) < 2e-3
