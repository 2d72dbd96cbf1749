"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/* by running the UNMODIFIED reference (oracle/reference.py)
on the CPU.  Re-run with:  python oracle/make_golden.py [train | reference]
The fixtures pin (a) oracle/restatement.py and (b) the CUDA path, on machines where the reference is absent.
`signature_table` and `state_dict_digest` are shared with the tests that read the `reference` fixtures.
"""
import hashlib
import inspect
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import reference  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
# torch's fp32 CPU kernels split their sums by the intra-op thread count, so the last bits of every fixture depend on it
# (and on the ISA: AVX-512).  The fixtures were made with this many threads; the bit-exact tests run with it too.
CPU_THREADS = 8


def _inputs(b, s, L, E, seed, lowres):
    g = torch.Generator().manual_seed(seed)
    d = dict(x=torch.randn(b, 3, s, s, generator=g), time=torch.tensor([17, 3][:b]),
             text_embeds=torch.randn(b, L, E, generator=g))
    mask = torch.ones(b, L, dtype=torch.bool)
    mask[0, L // 2:] = False
    d['text_embeds'][0, L // 2:] = 0.          # t5.py:82 zeroes padded positions
    d['text_mask'] = mask
    if lowres:
        d['lowres_cond_img'] = torch.randn(b, 3, s, s, generator=g)
        d['lowres_noise_times'] = torch.full((b,), 5)
    return d


def unet_case(name, cfg, s, lowres):
    from minimagen.Unet import Unet
    torch.manual_seed(0)
    u = Unet(**cfg).eval()
    inp = _inputs(2, s, 11, cfg.get('text_embed_dim', 512), 1, lowres)
    kw = {k: v for k, v in inp.items() if k not in ('x', 'time')}
    with torch.no_grad():
        out_cond = u(inp['x'], inp['time'], **kw)
        out_null = u(inp['x'], inp['time'], cond_drop_prob=1., **kw)
        out_nomask = u(inp['x'], inp['time'], **{**kw, 'text_mask': None})
        out_cfg = u.forward_with_cond_scale(inp['x'], inp['time'], cond_scale=3., **kw)
    torch.save(dict(cfg=cfg, state_dict=u.state_dict(), inputs=inp, out_cond=out_cond, out_null=out_null,
                    out_nomask=out_nomask, out_cfg3=out_cfg), os.path.join(OUT, name + ".pt"))
    print(name, "params", sum(p.numel() for p in u.parameters()), "out std", out_cond.std().item())


def step_case():
    """_p_mean_variance/_p_sample on injected model output + noise, T = 25 (the shipped tiny config) and T = 1000."""
    from minimagen.Imagen import Imagen
    from minimagen.Unet import Unet, BaseTest
    cases = {}
    for T in (25, 1000):
        torch.manual_seed(0)
        u = Unet(**BaseTest.defaults)
        im = Imagen(unets=u, text_encoder_name='t5_small', image_sizes=(64,), timesteps=T, cond_drop_prob=0.15)
        sch = im.noise_schedulers[0]
        g = torch.Generator().manual_seed(5 + T)
        x = torch.randn(3, 3, 64, 64, generator=g)
        eps = torch.randn(3, 3, 64, 64, generator=g) * 1.5
        noise = torch.randn(3, 3, 64, 64, generator=g)
        t = torch.tensor([T - 1, T // 3, 0])
        with torch.no_grad():
            mean, var, logvar = im._p_mean_variance(u, x=x, t=t, noise_scheduler=sch, model_output=eps)
            x0 = sch.predict_start_from_noise(x, t=t, noise=eps)
            s = torch.quantile(x0.flatten(1).abs(), 0.9, dim=-1)
            nz = (1 - (t == 0).float()).reshape(3, 1, 1, 1)
            out = mean + nz * (0.5 * logvar).exp() * noise
        tables = {k: v.clone() for k, v in sch.named_buffers()}
        cases[T] = dict(x=x, eps=eps, noise=noise, t=t, mean=mean, logvar=logvar, x0=x0, s_quantile=s, out=out,
                        tables=tables)
    # quantile rank arithmetic at the BASELINE image sizes (fp32 rank, SURVEY.md 8a row 12)
    ranks = {}
    for n in (3 * 64 * 64, 3 * 256 * 256, 3 * 1024 * 1024):
        r = torch.tensor(0.9, dtype=torch.float32) * (n - 1)
        ranks[n] = (int(r.floor()), int(r.ceil()), float(r - r.floor()))
    cases['ranks'] = ranks
    torch.save(cases, os.path.join(OUT, "ddpm_step.pt"))
    print("ddpm_step ranks", ranks)


def sample_case():
    """3 iterations of Imagen._p_sample_loop (tiny base U-Net, T=25, cond_scale=3) with injected noise."""
    import minimagen.Imagen as MI
    from minimagen.Imagen import Imagen
    from minimagen.Unet import Unet, BaseTest
    torch.manual_seed(0)
    u = Unet(**BaseTest.defaults)
    im = Imagen(unets=u, text_encoder_name='t5_small', image_sizes=(64,), timesteps=25, cond_drop_prob=0.15).eval()
    sd = u.state_dict()
    g = torch.Generator().manual_seed(11)
    inp = _inputs(2, 64, 9, 512, 2, False)
    x_T = torch.randn(2, 3, 64, 64, generator=g)
    noises = [torch.randn(2, 3, 64, 64, generator=g) for _ in range(3)]
    sch = im.noise_schedulers[0]
    img = x_T
    traj = []
    it = iter(noises)
    real = MI.torch.randn_like
    MI.torch.randn_like = lambda z: next(it)
    try:
        with torch.no_grad():
            for i, t in enumerate(sch._get_sampling_timesteps(2, device='cpu')[:3]):
                img = im._p_sample(u, img, t, text_embeds=inp['text_embeds'], text_mask=inp['text_mask'], cond_scale=3.,
                                   noise_scheduler=sch)
                traj.append(img)
    finally:
        MI.torch.randn_like = real
    torch.save(dict(cfg=dict(BaseTest.defaults), state_dict=sd, text_embeds=inp['text_embeds'],
                    text_mask=inp['text_mask'], x_T=x_T, noises=noises, traj=traj, timesteps=25, cond_scale=3.),
               os.path.join(OUT, "sample_loop.pt"))
    print("sample_loop x std", [t.std().item() for t in traj])


def cascade_case():
    """The unmodified reference's Imagen.sample over a tiny 2-stage cascade (base 16x16 -> SR 32x32, T=25, CFG w=2): every
    normal draw is recorded in call order so that the implementation under test can replay it (inter-stage resize runs on
    the resize_right stand-in, see oracle/shims)."""
    import minimagen.Imagen as MI
    from minimagen.Imagen import Imagen
    from minimagen.Unet import Unet, BaseTest, SuperTest
    torch.manual_seed(5)
    u0, u1 = Unet(**BaseTest.defaults), Unet(**SuperTest.defaults)
    im = Imagen(unets=(u0, u1), text_encoder_name='t5_small', image_sizes=(16, 32), timesteps=25, cond_drop_prob=0.1).eval()
    g = torch.Generator().manual_seed(21)
    te = torch.randn(2, 7, 512, generator=g)
    tm = torch.ones(2, 7, dtype=torch.bool)
    tm[1, 5:] = False
    te = te * tm[..., None]
    draws = []
    real_randn, real_like = MI.torch.randn, MI.torch.randn_like

    def rec_randn(*a, **k):
        out = real_randn(*a, **{kk: v for kk, v in k.items() if kk != 'device'})
        draws.append(out.clone())
        return out

    def rec_like(z):
        out = real_like(z)
        draws.append(out.clone())
        return out
    MI.torch.randn, MI.torch.randn_like = rec_randn, rec_like
    try:
        torch.manual_seed(77)
        with torch.no_grad():
            out = im.sample(text_embeds=te, text_masks=tm, cond_scale=2., lowres_sample_noise_level=0.2)
    finally:
        MI.torch.randn, MI.torch.randn_like = real_randn, real_like
    torch.save(dict(cfgs=(dict(BaseTest.defaults), dict(SuperTest.defaults)),
                    state_dicts=(im.unets[0].state_dict(), im.unets[1].state_dict()), text_embeds=te, text_mask=tm,
                    draws=draws, out=out, image_sizes=(16, 32), timesteps=25, cond_scale=2., lowres_noise_level=0.2),
               os.path.join(OUT, "cascade_tiny.pt"))
    print("cascade_tiny: draws", [tuple(d.shape) for d in draws], "out", tuple(out.shape), float(out.mean()))


def train_case():
    """Training side (SURVEY 8f-2): the reference's own `Imagen._p_losses` (Imagen.py:512-573) + `loss.backward()` on the tiny
    base and super-resolution U-Nets, with every random draw pinned: `times` / `noise` are passed in, the conditional-dropout
    keep mask (Unet.py:587 `prob_mask_like`) and the low-res augmentation noise (`torch.randn_like`, Imagen.py:556) are recorded."""
    import minimagen.Imagen as MI
    import minimagen.Unet as MU
    from minimagen.Imagen import Imagen
    from minimagen.Unet import Unet, BaseTest, SuperTest
    torch.manual_seed(0)
    im = Imagen(unets=(Unet(**BaseTest.defaults), Unet(**SuperTest.defaults)), text_encoder_name='t5_small',
                image_sizes=(16, 32), timesteps=25, cond_drop_prob=0.15)
    g = torch.Generator().manual_seed(11)
    b = 3
    te = torch.randn(b, 9, 512, generator=g)
    tm = torch.ones(b, 9, dtype=torch.bool)
    tm[1, 5:] = False
    te[1, 5:] = 0.
    keep = torch.tensor([True, False, True])
    cases = []
    real_mask, real_like = MU.prob_mask_like, MI.torch.randn_like
    MU.prob_mask_like = lambda shape, prob, device: keep.to(device)
    try:
        for idx, size in ((0, 16), (1, 32)):
            unet = im.unets[idx]
            for p in im.parameters():
                p.grad = None
            x0 = torch.rand(b, 3, size, size, generator=g)                  # training images in [0, 1]
            noise = torch.randn(b, 3, size, size, generator=g)
            times = torch.tensor([3, 24, 11])
            kw = dict(noise_scheduler=im.noise_schedulers[idx], text_embeds=te, text_mask=tm, noise=noise)
            rec = {}
            if idx == 1:
                kw.update(lowres_cond_img=torch.rand(b, 3, size, size, generator=g), lowres_aug_times=torch.tensor([7, 7, 7]))

                def rec_like(t, **k2):
                    rec['lowres_noise'] = real_like(t, **k2)
                    return rec['lowres_noise']
                MI.torch.randn_like = rec_like
            torch.manual_seed(5)
            loss = im._p_losses(unet, x0, times, **kw)
            MI.torch.randn_like = real_like
            loss.backward()
            grads = {k: p.grad.clone() for k, p in unet.named_parameters() if p.grad is not None}
            cases.append(dict(cfg=dict(BaseTest.defaults if idx == 0 else SuperTest.defaults), unet_index=idx, size=size,
                              state_dict={k: v.clone() for k, v in unet.state_dict().items()}, x0=x0, noise=noise,
                              times=times, lowres_cond_img=kw.get('lowres_cond_img'),
                              lowres_aug_times=kw.get('lowres_aug_times'), lowres_noise=rec.get('lowres_noise'),
                              loss=loss.detach().clone(), grads=grads))
            print("train case", idx, "loss", float(loss), "grad tensors", len(grads),
                  "missing grads", [k for k, p in unet.named_parameters() if p.grad is None])
    finally:
        MU.prob_mask_like, MI.torch.randn_like = real_mask, real_like
    torch.save(dict(cases=cases, text_embeds=te, text_mask=tm, keep=keep, image_sizes=(16, 32), timesteps=25,
                    cond_drop_prob=0.15), os.path.join(OUT, "train_tiny.pt"))


def signature_table(unet_mod, imagen_mod, diffusion_mod):
    """Parameter lists (name, kind, repr of the default) of the public constructors / entry points and the U-Net
    presets' defaults (repr), as JSON-ready lists and strings."""
    def params(f):
        return [[p.name, p.kind.name, "<empty>" if p.default is inspect.Parameter.empty else repr(p.default)]
                for p in inspect.signature(f).parameters.values()]
    return {"Unet.__init__": params(unet_mod.Unet.__init__), "Imagen.__init__": params(imagen_mod.Imagen.__init__),
            "GaussianDiffusion.__init__": params(diffusion_mod.GaussianDiffusion.__init__),
            "Unet.forward": params(unet_mod.Unet.forward), "Imagen.sample": params(imagen_mod.Imagen.sample),
            "presets": {c: repr(getattr(unet_mod, c).defaults) for c in ("Base", "Super", "BaseTest", "SuperTest")}}


def state_dict_digest(sd):
    """SHA-256 over a state dict's names, dtypes, shapes and bytes (in order): pins weights too large to store."""
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(f"{k}:{v.dtype}:{tuple(v.shape)};".encode())
        h.update(v.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


# inputs of the fixtures below; the tests rebuild them from the same seeds
LIVE_UNET_CFGS = [
    (dict(dim=32, dim_mults=(1, 2), attend_at_middle=True, text_embed_dim=768), 32, False),
    (dict(dim=32, dim_mults=(1, 2), lowres_cond=True, memory_efficient=True, num_resnet_blocks=(1, 2),
          layer_attns=(False, True), layer_cross_attns=(False, True)), 32, True),
]
RESIZE_CASES = [(64, 256, "reflect", None), (16, 64, "reflect", (0., 1.)), (128, 64, "reflect", (-1., 1.)),
                (24, 36, "constant", None), (32, 128, "edge", None)]
RESIZE_SAMPLE = 4096


def live_unet_inputs(cfg, s, lowres):
    g = torch.Generator().manual_seed(7)
    x = torch.randn(2, 3, s, s, generator=g)
    te = torch.randn(2, 20, cfg.get("text_embed_dim", 512), generator=g)
    tm = torch.ones(2, 20, dtype=torch.bool)
    tm[1, 5:] = False
    kw = dict(text_embeds=te, text_mask=tm)
    if lowres:
        kw.update(lowres_cond_img=torch.randn(2, 3, s, s, generator=g), lowres_noise_times=torch.tensor([200, 3]))
    return x, torch.tensor([999, 0]), kw


def resize_input(n_in):
    return torch.rand(2, 3, n_in, n_in, generator=torch.Generator().manual_seed(n_in)) * 2 - 0.5


def reference_cases():
    """What the tests used to compare against the live reference: its signatures (signatures.json), its U-Net forward
    at two dim-32 configs (unet_dim32.pt: outputs + digest of the seed-0 weights, 6-9 MB each, which the test rebuilds)
    and its inter-stage resize helper (resize.pt: a fixed seeded sample of each output plus the full-output sum)."""
    import minimagen.Unet as RU
    import minimagen.Imagen as RI
    import minimagen.diffusion_model as RD
    ref = sys.modules["minimagen"]
    with open(os.path.join(OUT, "signatures.json"), "w") as f:
        json.dump(signature_table(RU, RI, RD), f, indent=1)
        f.write("\n")
    cases = []
    for cfg, s, lowres in LIVE_UNET_CFGS:
        torch.manual_seed(0)
        r = RU.Unet(**cfg).eval()
        x, t, kw = live_unet_inputs(cfg, s, lowres)
        with torch.no_grad():
            outs = {cdp: r(x, t, cond_drop_prob=cdp, **kw) for cdp in (0., 1.)}
        cases.append(dict(cfg=cfg, weights_sha256=state_dict_digest(r.state_dict()), outs=outs))
    torch.save(cases, os.path.join(OUT, "unet_dim32.pt"))
    res = {}
    for n_in, n_out, pad, clamp in RESIZE_CASES:
        want = ref.helpers.resize_image_to(resize_input(n_in), n_out, clamp_range=clamp, pad_mode=pad)
        n = want.numel()
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:min(n, RESIZE_SAMPLE)].sort().values
        res[(n_in, n_out, pad, clamp)] = dict(shape=tuple(want.shape), idx=idx.int(), values=want.flatten()[idx].clone(),
                                              sum=want.double().sum().item())
    torch.save(res, os.path.join(OUT, "resize.pt"))
    print("reference cases: unet_dim32", [c["weights_sha256"][:12] for c in cases], "resize", len(res))


if __name__ == "__main__":
    reference.load()
    torch.set_num_threads(CPU_THREADS)
    os.makedirs(OUT, exist_ok=True)
    from minimagen.Unet import BaseTest, SuperTest
    if len(sys.argv) > 1 and sys.argv[1] == "train":
        train_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "reference":
        reference_cases()
        sys.exit(0)
    unet_case("unet_tiny_base", dict(BaseTest.defaults), 64, False)
    unet_case("unet_tiny_sr", dict(SuperTest.defaults, lowres_cond=True), 64, True)
    step_case()
    sample_case()
    cascade_case()
    train_case()
    reference_cases()
