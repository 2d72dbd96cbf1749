"""Text-guided inpainting (Imagen.sample(inpaint_images=, inpaint_masks=, inpaint_resample_times=)) against the algorithm
restated below from oracle.restatement.  The reference has no inpainting, so the oracle is the algorithm itself:

    per stage of size s:  K = normalize(resize_image_to(images, s)),  m[b,i,j] = masks[b, i*Hm//s, j*Wm//s]
    x = N(0, I);  x = where(m, sqrt_acp[T-1] K + sqrt_1macp[T-1] z_k, x)                        # prime
    for t = T-1 .. 0, u = 0 .. U_t-1  (U_t = U for t > 0, 1 at t = 0):
        x' = p_sample(x, t)                                                                     # U-Net(s), CFG, threshold
        u < U_t-1:  x = where(m, sqrt_acp[t] K + sqrt_1macp[t] z_k, sqrt(1-beta_t) x' + sqrt(beta_t) z_r)   # RePaint
        t > 0:      x = where(m, sqrt_acp[t-1] K + sqrt_1macp[t-1] z_k, x')
        t = 0:      x = where(m, K, x')                                                          # final paste
    finalize: (clamp(x, -1, 1) + 1) / 2

Noise comes from a seeded bank keyed by (kind, key, image shape): ('step', t*U+u), ('renoise', t*U+u) when the step
renoises, ('inpaint', t*U+u) unless it is the final paste, ('inpaint', -1) for the prime, ('init', -1), ('lowres', stage).
The bank draws for a batch of 4 and hands out rows, so shards see the rows the full batch sees."""
import contextlib
import zlib

import pytest
import torch

from conftest import load_golden, rel_l2
from emu_ops import EmuOps
from oracle import restatement as R


# ------------------------------------------------------------------------------------------------ emulation
class InpaintEmuOps(EmuOps):
    """The torch emulation of the ops interface (tests/emu_ops.py) plus the contracts of the two inpainting entry points."""

    def inpaint_blend(self, x, known, mask, z_known, z_renoise, t, u, U, prime, sqrt_acp, sqrt_1macp, sqrt_alphas,
                      sqrt_betas):
        """contract of mi_inpaint_blend"""
        self._log("inpaint_blend")
        B, C, H, W = x.shape
        mh, mw = mask.shape[-2:]
        iy = torch.arange(H, device=x.device) * mh // H
        ix = torch.arange(W, device=x.device) * mw // W
        m = (mask[:, iy][:, :, ix] != 0)[:, None]                                   # B,1,H,W
        col = lambda tab, tt: tab[tt].reshape(B, 1, 1, 1)
        if prime:
            x.copy_(torch.where(m, col(sqrt_acp, t) * known + col(sqrt_1macp, t) * z_known, x))
            return
        ut = torch.where(t > 0, U, 1)
        renoise = (u.long() < ut - 1).reshape(B, 1, 1, 1)
        tk = torch.where(renoise.reshape(B), t, (t - 1).clamp(min=0))
        target = torch.where((t == 0).reshape(B, 1, 1, 1) & ~renoise, known,
                             col(sqrt_acp, tk) * known + col(sqrt_1macp, tk) * z_known)
        y = torch.where(renoise, col(sqrt_alphas, t) * x + col(sqrt_betas, t) * z_renoise, x)
        x.copy_(torch.where(m, target, y))

    def inpaint_advance(self, t, u, U, B):
        """contract of mi_inpaint_advance"""
        self._log("inpaint_advance")
        renoised = int(u.item()) < (U if int(t[0].item()) > 0 else 1) - 1
        if renoised:
            u.add_(1)
        else:
            u.zero_()
            t.copy_((t - 1).clamp(min=0))


@pytest.fixture
def emu():
    """This module's emulation (InpaintEmuOps) installed as the ops backend, restored afterwards."""
    import minimagen_b200.ops as ops_mod
    prev = ops_mod._OPS
    e = InpaintEmuOps()
    ops_mod.set_ops(e)
    yield e
    ops_mod.set_ops(prev)


# ------------------------------------------------------------------------------------------------ oracle
def repaint_tables(T):
    """ddpm_tables plus sqrt(1 - beta) / sqrt(beta), from the same fp64 schedule, cast to fp32."""
    tabs = R.ddpm_tables(T)
    scale = 1000 / T
    betas = torch.linspace(scale * 0.0001, scale * 0.02, T, dtype=torch.float64)
    tabs['sqrt_alphas'] = torch.sqrt(1. - betas).float()
    tabs['sqrt_betas'] = torch.sqrt(betas).float()
    return tabs


def stage_mask(masks, s):
    """Nearest-neighbour by integer arithmetic: m[b, i, j] = masks[b, i*Hm//s, j*Wm//s], as [B, 1, s, s] bool."""
    hm, wm = masks.shape[-2:]
    iy, ix = torch.arange(s) * hm // s, torch.arange(s) * wm // s
    return masks.bool()[:, iy][:, :, ix][:, None]


def restated_stage(sd, cfg, tabs, U, K, m, draw, *, text_embeds, text_mask, cond_scale, lowres=None, max_steps=None):
    """One stage of the inpainting loop on CPU, returning the un-finalised x.  draw(kind, key) -> noise of K's shape."""
    T = tabs['betas'].shape[0]
    B = K.shape[0]
    acp, macp = tabs['sqrt_alphas_cumprod'], tabs['sqrt_one_minus_alphas_cumprod']
    known_at = lambda t, z: acp[t] * K + macp[t] * z
    lowres = lowres or {}
    x = draw('init', -1)
    x = torch.where(m, known_at(T - 1, draw('inpaint', -1)), x)
    n = 0
    for t in reversed(range(T)):
        ut = U if t > 0 else 1
        for u in range(ut):
            if max_steps is not None and n == max_steps:
                return x
            key = t * U + u
            tt = torch.full((B,), t, dtype=torch.long)
            eps = R.unet_forward(sd, cfg, x, tt, text_embeds=text_embeds, text_mask=text_mask, **lowres)
            if cond_scale != 1:
                eps = R.cfg_combine(eps, R.unet_forward(sd, cfg, x, tt, text_embeds=text_embeds, text_mask=text_mask,
                                                        cond_drop_prob=1., **lowres), cond_scale)
            xp = R.p_sample_step(tabs, x, tt, eps, draw('step', key))
            if u < ut - 1:
                y = tabs['sqrt_alphas'][t] * xp + tabs['sqrt_betas'][t] * draw('renoise', key)
                x = torch.where(m, known_at(t, draw('inpaint', key)), y)
            elif t > 0:
                x = torch.where(m, known_at(t - 1, draw('inpaint', key)), xp)
            else:
                x = torch.where(m, K, xp)
            n += 1
    return x


def finalize(x):
    return (x.clamp(-1, 1) + 1) * 0.5


class NoiseBank:
    """Draws for a batch of `full` images, each seeded from (seed, kind, step, image shape) alone -- so a draw does not
    depend on which other draws were made before it; `lo` selects the rows handed out."""

    def __init__(self, seed, full=4):
        self.seed, self.full, self.lo, self.bank = seed, full, 0, {}
        self.kinds = []

    def __call__(self, kind, shape, step):
        key = (kind, step, tuple(shape[1:]))
        if key not in self.bank:
            gen = torch.Generator().manual_seed(zlib.crc32(repr((self.seed, *key)).encode()))
            self.bank[key] = torch.randn(self.full, *shape[1:], generator=gen)
        self.kinds.append((kind, step))
        return self.bank[key][self.lo:self.lo + shape[0]]

    def drawer(self, shape):
        return lambda kind, step: self(kind, shape, step)


@contextlib.contextmanager
def emulated_ops():
    """The torch emulation of the ops interface for the oracle's CPU-side resizes (helpers.resize_image_to)."""
    import minimagen_b200.ops as ops_mod
    prev = ops_mod._OPS
    ops_mod.set_ops(InpaintEmuOps())
    try:
        yield
    finally:
        ops_mod.set_ops(prev)


def known_image(b, s, seed):
    """A smooth image in [0, 1]: bilinear upsampling of a coarse random grid."""
    g = torch.Generator().manual_seed(seed)
    coarse = torch.rand(b, 3, 4, 4, generator=g)
    return torch.nn.functional.interpolate(coarse, size=(s, s), mode='bilinear', align_corners=True).contiguous()


def blob_mask(b, s, seed):
    """True = known pixel: everything except a disc per image (centre and radius vary), plus a few random holes."""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(s), torch.arange(s), indexing='ij')
    masks = []
    for _ in range(b):
        cy, cx = (torch.rand(2, generator=g) * 0.5 + 0.25) * s
        r = (0.15 + 0.15 * torch.rand((), generator=g)) * s
        masks.append(((yy - cy) ** 2 + (xx - cx) ** 2) > r * r)
    m = torch.stack(masks)
    return m & (torch.rand(b, s, s, generator=g) > 0.05)


# ------------------------------------------------------------------------------------------------ fixtures of the loops
def _tiny_base(device, graph):
    from minimagen_b200.Imagen import Imagen
    from minimagen_b200.Unet import Unet
    g = load_golden("sample_loop.pt")
    u = Unet(**g["cfg"]).eval()
    u.load_state_dict(g["state_dict"])
    im = Imagen(unets=u, text_encoder_name="t5_small", image_sizes=(64,), timesteps=g["timesteps"],
                cond_drop_prob=0.15).eval().to(device)
    im.unets[0].load_state_dict(g["state_dict"])
    im.use_cuda_graph = graph
    return im, g


def _count_forwards(unet):
    calls = [0]
    fwd = unet.forward

    def counted(*a, **k):
        calls[0] += 1
        return fwd(*a, **k)
    unet.forward = counted
    return calls


def run_tiny_loop(device, graph, U, mask_fn=blob_mask):
    """Tiny base U-Net (sample_loop.pt), T=25, CFG w=3, b=2 at 64x64: (output, restated output, U-Net calls)."""
    im, g = _tiny_base(device, graph)
    bank = NoiseBank(5)
    im.noise_fn = bank
    calls = _count_forwards(im.unets[0])
    B, s = 2, 64
    imgs, masks = known_image(B, s, 1), mask_fn(B, s, 2)
    te, tm = g["text_embeds"], g["text_mask"]
    out = im.sample(text_embeds=te.to(device), text_masks=tm.to(device), cond_scale=g["cond_scale"],
                    inpaint_images=imgs.to(device), inpaint_masks=masks.to(device), inpaint_resample_times=U)
    tabs = repaint_tables(g["timesteps"])
    x = restated_stage(g["state_dict"], g["cfg"], tabs, U, imgs * 2 - 1, stage_mask(masks, s), bank.drawer((B, 3, s, s)),
                       text_embeds=te, text_mask=tm, cond_scale=g["cond_scale"])
    return out, finalize(x), calls[0], (imgs, masks)


def run_cascade(device, graph, U=2):
    """cascade_tiny.pt (base 16 -> SR 32, T=25, CFG w=2) with inputs at the last stage's size: (output, restated output)."""
    from minimagen_b200 import helpers
    from minimagen_b200.Imagen import Imagen
    from minimagen_b200.Unet import Unet
    g = load_golden("cascade_tiny.pt")
    unets = [Unet(**c) for c in g["cfgs"]]
    im = Imagen(unets=unets, text_encoder_name="t5_small", image_sizes=g["image_sizes"], timesteps=g["timesteps"],
                cond_drop_prob=0.1).eval().to(device)
    for u, sd in zip(im.unets, g["state_dicts"]):
        u.load_state_dict(sd)
    im.use_cuda_graph = graph
    bank = NoiseBank(9)
    im.noise_fn = bank
    B, S = 2, g["image_sizes"][-1]
    imgs, masks = known_image(B, S, 3), blob_mask(B, S, 4)
    kw = dict(text_embeds=g["text_embeds"], text_mask=g["text_mask"], cond_scale=g["cond_scale"])
    out = im.sample(text_embeds=kw["text_embeds"].to(device), text_masks=kw["text_mask"].to(device),
                    cond_scale=g["cond_scale"], lowres_sample_noise_level=g["lowres_noise_level"],
                    inpaint_images=imgs.to(device), inpaint_masks=masks.to(device), inpaint_resample_times=U)
    T = g["timesteps"]
    tabs = repaint_tables(T)
    img = None
    with emulated_ops():
        for i, (cfg, sd, s) in enumerate(zip(g["cfgs"], g["state_dicts"], g["image_sizes"])):
            lowres = None
            if i > 0:
                t_aug = torch.full((B,), int(T * g["lowres_noise_level"]), dtype=torch.long)
                up = helpers.resize_image_to(img, s, pad_mode='reflect')
                lr = R.q_sample(tabs, up, t_aug, bank('lowres', up.shape, i + 1))
                lowres = dict(lowres_cond_img=lr * 2 - 1, lowres_noise_times=t_aug)
            K = helpers.resize_image_to(imgs, s, pad_mode='reflect') * 2 - 1
            x = restated_stage(sd, dict(cfg, lowres_cond=i > 0), tabs, U, K, stage_mask(masks, s),
                               bank.drawer((B, 3, s, s)), lowres=lowres, **kw)
            img = finalize(x)
    return out, img


def run_sharded(device, graph):
    """A batch of 4 sampled whole and as two shards of 2 (what two ranks compute): (whole, shards concatenated)."""
    im, g = _tiny_base(device, graph)
    bank = NoiseBank(11)
    im.noise_fn = bank
    gen = torch.Generator().manual_seed(12)
    te = torch.randn(4, 9, 512, generator=gen).to(device)
    tm = torch.ones(4, 9, dtype=torch.bool).to(device)
    imgs, masks = known_image(4, 64, 13).to(device), blob_mask(4, 64, 14).to(device)
    kw = dict(cond_scale=3., inpaint_resample_times=2)
    full = im.sample(text_embeds=te, text_masks=tm, inpaint_images=imgs, inpaint_masks=masks, **kw)
    parts = []
    for lo in (0, 2):
        bank.lo = lo
        sl = slice(lo, lo + 2)
        parts.append(im.sample(text_embeds=te[sl], text_masks=tm[sl], inpaint_images=imgs[sl], inpaint_masks=masks[sl],
                               **kw))
    return full, torch.cat(parts)


# ------------------------------------------------------------------------------------------------ blend / advance contract
def explicit_blend(x, K, mask, zk, zr, t, u, U, prime, tabs):
    """The blend written per image with explicit mask indexing."""
    B, C, H, W = x.shape
    mh, mw = mask.shape[-2:]
    out = x.clone()
    acp, macp = tabs['sqrt_alphas_cumprod'], tabs['sqrt_one_minus_alphas_cumprod']
    for b in range(B):
        mb = torch.tensor([[bool(mask[b, i * mh // H, j * mw // W]) for j in range(W)] for i in range(H)])
        tb = int(t[b])
        if prime:
            out[b] = torch.where(mb, acp[tb] * K[b] + macp[tb] * zk[b], x[b])
            continue
        ut = U if tb > 0 else 1
        if int(u[0]) < ut - 1:
            y = tabs['sqrt_alphas'][tb] * x[b] + tabs['sqrt_betas'][tb] * zr[b]
            out[b] = torch.where(mb, acp[tb] * K[b] + macp[tb] * zk[b], y)
        elif tb > 0:
            out[b] = torch.where(mb, acp[tb - 1] * K[b] + macp[tb - 1] * zk[b], x[b])
        else:
            out[b] = torch.where(mb, K[b], x[b])
    return out


def blend_case(B, s, mask_hw, seed):
    g = torch.Generator().manual_seed(seed)
    x, K, zk, zr = (torch.randn(B, 3, s, s, generator=g) for _ in range(4))
    mask = (torch.rand(B, *mask_hw, generator=g) > 0.5).to(torch.uint8)
    return x, K, mask, zk, zr


# (t, u, prime) per U: prime, renoise (U > 1), the last round of t > 0, the final paste at t = 0
BRANCHES = {1: [(24, 0, 1), (24, 0, 0), (7, 0, 0), (0, 0, 0)],
            3: [(24, 0, 1), (24, 0, 0), (24, 1, 0), (24, 2, 0), (1, 2, 0), (0, 0, 0)]}


@pytest.mark.parametrize("U", [1, 3])
@pytest.mark.parametrize("mask_hw", [(32, 32), (64, 64), (16, 16), (17, 23)])
def test_blend_and_advance_contract(emu, U, mask_hw):
    """InpaintEmuOps.inpaint_blend / inpaint_advance equal the explicit per-image algorithm bit for bit on every branch, with the
    mask at the stage size, at 2x, at 1/2 and at an odd size."""
    tabs = repaint_tables(25)
    B, s = 2, 32
    for k, (t0, u0, prime) in enumerate(BRANCHES[U]):
        x, K, mask, zk, zr = blend_case(B, s, mask_hw, 100 + k)
        t = torch.full((B,), t0, dtype=torch.long)
        u = torch.tensor([u0], dtype=torch.int32)
        want = explicit_blend(x, K, mask, zk, zr, t, u, U, prime, tabs)
        got = x.clone()
        emu.inpaint_blend(got, K, mask, zk, zr, t, u, U, prime, tabs['sqrt_alphas_cumprod'],
                          tabs['sqrt_one_minus_alphas_cumprod'], tabs['sqrt_alphas'], tabs['sqrt_betas'])
        assert torch.equal(got, want), (t0, u0, prime)
        if prime:
            continue
        emu.inpaint_advance(t, u, U, B)
        renoised = u0 < (U if t0 > 0 else 1) - 1
        assert int(u[0]) == (u0 + 1 if renoised else 0)
        assert torch.equal(t, torch.full((B,), t0 if renoised else max(t0 - 1, 0), dtype=torch.long))


def test_schedule_and_noise_keys(emu):
    """(T-1)*U + 1 steps; the draws are keyed t*U + u in the documented order."""
    from minimagen_b200.Imagen import Imagen
    sched = Imagen._inpaint_schedule(25, 3)
    assert len(sched) == 24 * 3 + 1 and sched[:4] == [(24, 0), (24, 1), (24, 2), (23, 0)] and sched[-1] == (0, 0)
    im, g = _tiny_base("cpu", False)
    bank = NoiseBank(0)
    im.noise_fn = bank
    im.sample(text_embeds=g["text_embeds"], text_masks=g["text_mask"], cond_scale=1., inpaint_images=known_image(2, 64, 0),
              inpaint_masks=blob_mask(2, 64, 0), inpaint_resample_times=2)
    want = [('init', -1), ('inpaint', -1)]
    for t, u in Imagen._inpaint_schedule(25, 2):
        key = t * 2 + u
        want.append(('step', key))
        if t > 0 and u == 0:
            want.append(('renoise', key))
        if t > 0:
            want.append(('inpaint', key))
    assert bank.kinds == want
    # the loop works on its own copies: the injected draws themselves are left as they were drawn
    for (kind, step, shp), v in bank.bank.items():
        assert torch.equal(v, NoiseBank(0)(kind, (4, *shp), step)), (kind, step)


# ------------------------------------------------------------------------------------------------ loops on CPU (emulation)
@pytest.mark.parametrize("U", [1, 2])
def test_tiny_loop_vs_restatement(emu, U):
    out, ref, calls, _ = run_tiny_loop("cpu", False, U)
    err = rel_l2(out, ref)
    print(f"tiny inpainting loop U={U}: rel-L2 vs restatement = {err:.3e}")
    assert err < 1e-3
    assert calls == 2 * (24 * U + 1)                       # (T-1)*U + 1 steps, two guidance passes each
    assert emu.calls.count("inpaint_blend") == 24 * U + 2 and emu.calls.count("inpaint_advance") == 24 * U + 1


def test_u1_all_false_mask_is_plain_sampling(emu):
    """U = 1 with nothing known reproduces Imagen.sample without inpainting exactly (same draws, same kernels)."""
    outs = []
    for inpaint in (False, True):
        im, g = _tiny_base("cpu", False)
        im.noise_fn = NoiseBank(21)
        kw = dict(inpaint_images=known_image(2, 64, 0), inpaint_masks=torch.zeros(2, 64, 64, dtype=torch.bool),
                  inpaint_resample_times=1) if inpaint else {}
        outs.append(im.sample(text_embeds=g["text_embeds"], text_masks=g["text_mask"], cond_scale=g["cond_scale"], **kw))
    assert torch.equal(outs[0], outs[1])


def test_known_pixels_are_pasted_exactly(emu):
    """Masked pixels of the result are exactly the finalised known image ((2K-1).clamp(-1, 1) + 1) * 0.5."""
    for masks in (torch.ones(2, 64, 64, dtype=torch.bool), blob_mask(2, 64, 2)):
        out, _, _, (imgs, m) = run_tiny_loop("cpu", False, 1, mask_fn=lambda b, s, seed: masks)
        want = ((2 * imgs - 1).clamp(-1, 1) + 1) * 0.5
        m4 = m[:, None].expand_as(out)
        assert torch.equal(out[m4], want[m4])
        if bool(m.all()):
            assert torch.equal(out, want)


def test_cascade_vs_restatement(emu):
    out, ref = run_cascade("cpu", False)
    err = rel_l2(out, ref)
    print(f"cascade inpainting (16 -> 32, U=2): rel-L2 vs restatement = {err:.3e}")
    assert out.shape == (2, 3, 32, 32) and err < 1e-3


def test_validation(emu):
    im, g = _tiny_base("cpu", False)
    te, tm = g["text_embeds"], g["text_mask"]
    img, msk = known_image(2, 64, 0), blob_mask(2, 64, 0)
    cases = [
        (dict(inpaint_images=img), "given together"),
        (dict(inpaint_masks=msk), "given together"),
        (dict(inpaint_images=img.double().numpy(), inpaint_masks=msk), "float tensor"),
        (dict(inpaint_images=(img * 255).to(torch.uint8), inpaint_masks=msk), "float tensor"),
        (dict(inpaint_images=img[:1], inpaint_masks=msk), r"must be \(2, 3, h, h\)"),
        (dict(inpaint_images=img[:, :1], inpaint_masks=msk), r"must be \(2, 3, h, h\)"),
        (dict(inpaint_images=img[..., :32], inpaint_masks=msk), r"must be \(2, 3, h, h\)"),
        (dict(inpaint_images=img, inpaint_masks=msk.float()), "bool tensor"),
        (dict(inpaint_images=img, inpaint_masks=msk[:, None]), "bool tensor"),
        (dict(inpaint_images=img, inpaint_masks=msk[:1]), "bool tensor"),
        (dict(inpaint_images=img, inpaint_masks=msk[:, :32, :32]), "differs from the inpaint_images size"),
        (dict(inpaint_images=img, inpaint_masks=msk, inpaint_resample_times=0), "int >= 1"),
        (dict(inpaint_images=img, inpaint_masks=msk, inpaint_resample_times=2.0), "int >= 1"),
        (dict(inpaint_images=img, inpaint_masks=msk, inpaint_resample_times=True), "int >= 1"),
    ]
    for kw, msg in cases:
        emu.calls.clear()
        with pytest.raises(AssertionError, match=msg):
            im.sample(text_embeds=te, text_masks=tm, **kw)
        assert not emu.calls                                # rejected before any work


def test_sharding_invariance(emu):
    full, parts = run_sharded("cpu", False)
    err = rel_l2(parts, full)
    print(f"inpainting batch 4 vs two shards of 2: rel-L2 = {err:.3e}")
    assert err < 1e-6


def test_schedule_tables_are_not_buffers():
    """The RePaint tables are cached beside the schedule, not registered: the module's buffers stay the reference's."""
    from minimagen_b200.diffusion_model import GaussianDiffusion
    d = GaussianDiffusion(timesteps=25)
    names = [n for n, _ in d.named_buffers()]
    sa, sb = d.inpaint_tables("cpu")
    assert [n for n, _ in d.named_buffers()] == names and d.inpaint_tables("cpu")[0] is sa
    tabs = repaint_tables(25)
    assert torch.equal(sa, tabs['sqrt_alphas']) and torch.equal(sb, tabs['sqrt_betas'])


# ------------------------------------------------------------------------------------------------ on the B200
@pytest.mark.gpu
def test_kernels_vs_emulation_bit_exact(native):
    """mi_inpaint_blend / mi_inpaint_advance against the emulation, bit for bit, on every branch (B=3, 40x40, mask 17x23)."""
    emu = InpaintEmuOps()
    tabs = repaint_tables(25)
    dtabs = [tabs[k].cuda() for k in ('sqrt_alphas_cumprod', 'sqrt_one_minus_alphas_cumprod', 'sqrt_alphas', 'sqrt_betas')]
    ctabs = [tabs[k] for k in ('sqrt_alphas_cumprod', 'sqrt_one_minus_alphas_cumprod', 'sqrt_alphas', 'sqrt_betas')]
    B, s = 3, 40
    n = 0
    for U, branches in BRANCHES.items():
        for k, (t0, u0, prime) in enumerate(branches):
            x, K, mask, zk, zr = blend_case(B, s, (17, 23), 200 + k)
            t = torch.full((B,), t0, dtype=torch.long)
            u = torch.tensor([u0], dtype=torch.int32)
            want = x.clone()
            emu.inpaint_blend(want, K, mask, zk, zr, t, u, U, prime, *ctabs)
            xd, td, ud = x.cuda(), t.cuda(), u.cuda()
            native.inpaint_blend(xd, K.cuda(), mask.cuda(), zk.cuda(), zr.cuda(), td, ud, U, prime, *dtabs)
            assert torch.equal(xd.cpu(), want), (U, t0, u0, prime)
            if not prime:
                emu.inpaint_advance(t, u, U, B)
                native.inpaint_advance(td, ud, U, B)
                assert torch.equal(td.cpu(), t) and torch.equal(ud.cpu(), u), (U, t0, u0)
            n += 1
    torch.cuda.synchronize()
    print(f"inpaint kernels: {n} branch cases bit-exact vs emulation")


@pytest.mark.gpu
def test_device_errors(native):
    from minimagen_b200 import _native as N
    lib = N.load()
    assert lib.mi_inpaint_advance(None, None, 2, 1, None) == -1 and b"mi_inpaint_advance" in lib.mi_last_error()
    t = torch.zeros(2, dtype=torch.long, device="cuda")
    u = torch.zeros(1, dtype=torch.int32, device="cuda")
    assert lib.mi_inpaint_advance(t.data_ptr(), u.data_ptr(), 0, 2, None) == -1
    x = torch.zeros(2, 3, 8, 8, device="cuda")
    m = torch.zeros(2, 8, 8, dtype=torch.uint8, device="cuda")
    p = x.data_ptr()
    assert lib.mi_inpaint_blend(p, p, m.data_ptr(), 8, 8, p, p, t.data_ptr(), u.data_ptr(), 1, 0, p, p, p, None,
                                2, 3, 8, 8, None) == -1
    assert lib.mi_inpaint_blend(p, p, m.data_ptr(), 0, 8, p, p, t.data_ptr(), u.data_ptr(), 1, 0, p, p, p, p,
                                2, 3, 8, 8, None) == -1


@pytest.mark.gpu
@pytest.mark.parametrize("U", [1, 2])
def test_tiny_loop_on_device(native, U):
    res = {graph: run_tiny_loop("cuda", graph, U) for graph in (False, True)}
    ref = res[False][1]
    for graph, (out, _, calls, (imgs, m)) in res.items():
        err = rel_l2(out, ref)
        print(f"tiny inpainting loop U={U} graph={graph}: rel-L2 vs restatement = {err:.3e}")
        assert err < 1e-3
        m4 = m[:, None].expand(out.shape)
        assert torch.equal(out.cpu()[m4], (((2 * imgs - 1).clamp(-1, 1) + 1) * 0.5)[m4])
    assert res[False][2] == 2 * (24 * U + 1)
    e = rel_l2(res[True][0], res[False][0])
    print(f"tiny inpainting loop U={U}: graph vs eager rel-L2 = {e:.3e}")
    assert e < 1e-5


@pytest.mark.gpu
def test_u1_all_false_mask_is_plain_sampling_on_device(native):
    for graph in (False, True):
        outs = []
        for inpaint in (False, True):
            im, g = _tiny_base("cuda", graph)
            im.noise_fn = NoiseBank(21)
            kw = dict(inpaint_images=known_image(2, 64, 0).cuda(),
                      inpaint_masks=torch.zeros(2, 64, 64, dtype=torch.bool, device="cuda"),
                      inpaint_resample_times=1) if inpaint else {}
            outs.append(im.sample(text_embeds=g["text_embeds"].cuda(), text_masks=g["text_mask"].cuda(),
                                  cond_scale=g["cond_scale"], **kw))
        e = rel_l2(outs[1], outs[0])
        print(f"U=1, all-False mask vs plain sampling (graph={graph}): rel-L2 = {e:.3e}")
        assert e < 1e-5                                     # GroupNorm statistics use atomics: summation order may differ


@pytest.mark.gpu
def test_cascade_on_device(native):
    res = {graph: run_cascade("cuda", graph) for graph in (False, True)}
    for graph, (out, ref) in res.items():
        err = rel_l2(out, ref)
        print(f"cascade inpainting graph={graph}: rel-L2 vs restatement = {err:.3e}")
        assert err < 1e-3
    e = rel_l2(res[True][0], res[False][0])
    print(f"cascade inpainting: graph vs eager rel-L2 = {e:.3e}")
    assert e < 1e-5


@pytest.mark.gpu
def test_tensor_core_sr_stage_vs_restatement(native):
    """The sr_d64 configuration of test_gpu_unet.CFGS (tensor-core convolutions, fp16 operands) as the SR stage at 64x64,
    b=2, U=2, 6 steps of the inpainting loop, graph and eager."""
    from minimagen_b200.Imagen import Imagen
    from minimagen_b200.Unet import BaseTest, Unet
    from test_gpu_unet import CFGS
    name, cfg, s, lowres, b = next(c for c in CFGS if c[0] == "sr_d64")
    torch.manual_seed(0)
    u = Unet(**cfg).eval()
    sd = {k: v.clone() for k, v in u.state_dict().items()}
    T, U, steps = 25, 2, 6                  # T = 25: large betas, so six steps from T-1 move x far from x_T
    gen = torch.Generator().manual_seed(31)
    te = torch.randn(b, 20, 512, generator=gen)
    tm = torch.ones(b, 20, dtype=torch.bool)
    tm[-1, 5:] = False
    lr01 = torch.rand(b, 3, s, s, generator=gen)
    t_aug = torch.full((b,), 200, dtype=torch.long)
    imgs, masks = known_image(b, s, 32), blob_mask(b, s, 33)
    tabs = repaint_tables(T)
    bank = NoiseBank(34)
    ref = restated_stage(sd, cfg, tabs, U, imgs * 2 - 1, stage_mask(masks, s), bank.drawer((b, 3, s, s)), text_embeds=te,
                         text_mask=tm, cond_scale=1., lowres=dict(lowres_cond_img=lr01 * 2 - 1, lowres_noise_times=t_aug),
                         max_steps=steps)
    ref = finalize(ref)
    outs = {}
    for graph in (False, True):
        im = Imagen(unets=(Unet(**BaseTest.defaults), u), text_encoder_name="t5_small", image_sizes=(s // 4, s),
                    timesteps=T, cond_drop_prob=0.1).eval().cuda()
        assert im.unets[1] is u
        im.use_cuda_graph = graph
        im.noise_fn = bank
        outs[graph] = im._p_sample_loop(u, (b, 3, s, s), noise_scheduler=im.noise_schedulers[1], text_embeds=te.cuda(),
                                        text_mask=tm.cuda(), lowres_cond_img=lr01.cuda(), lowres_noise_times=t_aug.cuda(),
                                        max_steps=steps,
                                        inpaint=((imgs * 2 - 1).cuda(), masks.to(torch.uint8).cuda(), U))
        err = rel_l2(outs[graph], ref)
        print(f"sr_d64 inpainting, {steps} steps, graph={graph}: rel-L2 vs restatement = {err:.3e}")
        assert err < 2e-3
    e = rel_l2(outs[True], outs[False])
    print(f"sr_d64 inpainting: graph vs eager rel-L2 = {e:.3e}")
    assert e < 1e-5


@pytest.mark.gpu
def test_cached_graph_follows_new_image_and_mask(native):
    """A second inpainting call of the same signature replays the cached graph; its static image and mask are refreshed,
    so the result equals the eager loop on the new inputs."""
    outs = {}
    for graph in (True, False):
        im, g = _tiny_base("cuda", graph)
        bank = NoiseBank(41)
        im.noise_fn = bank
        kw = dict(text_embeds=g["text_embeds"].cuda(), text_masks=g["text_mask"].cuda(), cond_scale=g["cond_scale"],
                  inpaint_resample_times=2)
        first = im.sample(inpaint_images=known_image(2, 64, 42).cuda(), inpaint_masks=blob_mask(2, 64, 43).cuda(), **kw)
        second = im.sample(inpaint_images=known_image(2, 64, 44).cuda(), inpaint_masks=blob_mask(2, 64, 45).cuda(), **kw)
        if graph:
            assert len(im._graphs) == 1
        outs[graph] = (first, second)
    e = rel_l2(outs[True][1], outs[False][1])
    effect = rel_l2(outs[False][1], outs[False][0])
    print(f"cached inpainting graph, new image and mask: rel-L2 vs eager = {e:.3e} (inputs change the output by {effect:.3e})")
    assert e < 1e-5 and effect > 1e-2


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_sharding_invariance_on_device(native, graph):
    full, parts = run_sharded("cuda", graph)
    err = rel_l2(parts, full)
    print(f"inpainting batch 4 vs two shards of 2 (graph={graph}): rel-L2 = {err:.3e}")
    assert err < 1e-5
