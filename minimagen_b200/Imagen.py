"""Cascaded text-to-image diffusion sampler, B200-native (reference: minimagen/Imagen.py).

Same class surface as the reference's `Imagen` (constructor `Imagen.py:27-42`, `.sample` `:424-433`, `.forward` `:575-582`,
`.device`, `.unets`, `.noise_schedulers`, `.lowres_noise_schedule`, `state_dict` / `load_state_dict` overrides), same
asserts and messages.  The reverse-diffusion step is executed by the fused step kernels (csrc/step.cu): CFG combine,
x0 prediction, EXACT per-image dynamic-threshold quantile (radix select), posterior mean and noise add; the whole step
(both U-Net passes + epilogue) is optionally replayed from a CUDA graph so the ~10^3 kernel launches per step cost
nothing on the host.

Three additions that the reference does not have (all optional, defaults reproduce the reference):
  * `noise_fn(kind, shape, step)`  -- inject the Gaussian draws (x_T, per-step noise, low-res augmentation noise) so that
    a CPU oracle and this GPU path consume identical numbers (CPU mt19937 and CUDA Philox streams differ);
  * data-parallel sampling over `torch.distributed` ranks: the batch is sharded, each rank runs the whole cascade on
    its shard, ONE NCCL all-gather assembles the finished images (`sample(..., distributed=True)`);
  * text-guided inpainting (`sample(..., inpaint_images=, inpaint_masks=, inpaint_resample_times=)`, the keywords of
    imagen-pytorch): the masked pixels are kept from the given images, the rest is generated, with RePaint resampling;
    the blend and the resample counter run on the device inside the captured step (csrc/step.cu, DESIGN.md 4.6).
"""
from contextlib import contextmanager
from typing import Callable, List, Literal, Tuple, Union

import torch
import torch.nn.functional as F
from torch import nn

from .Unet import Unet
from .diffusion_model import GaussianDiffusion
from .helpers import (cast_tuple, default, eval_decorator, exists, identity, maybe, module_device,
                      normalize_neg_one_to_one, null_context, resize_image_to, unnormalize_zero_to_one)
from . import _native as N
from .ops import get_ops
from .t5 import get_encoded_dim, t5_encode_text

F32 = torch.float32


def quantile_rank(n: int, q: float):
    """(rank_lo, rank_hi, weight) exactly as torch.quantile derives them: the rank q*(n-1) is computed in FP32
    (ATen quantile_compute: `q * (n - 1)` on an fp32 tensor), e.g. n = 3*1024*1024, q = 0.9 -> weight 0.25, not 0.3."""
    rank = torch.tensor(q, dtype=torch.float32) * (n - 1)
    lo = torch.floor(rank)
    hi = torch.ceil(rank)
    return int(lo.item()), int(hi.item()), float((rank - lo).item())


class _StepGraph:
    """One captured denoising step (U-Net pass(es) + step epilogue) over STATIC buffers:
         x      [B, C, s, s]  the image, updated IN PLACE by every replay (x_t -> x_{t-1});
         t      [B] int64     the timestep, decremented (floor 0) at the end of every replay;
         noise  [B, C, s, s]  the step's Gaussian draw: drawn INSIDE the graph (graph-safe Philox) unless the caller
                              injects noise, in which case it is copied here before each replay;
         cond   static copies of text_embeds / text_mask / lowres_cond_img / lowres_noise_times (`set_cond` refreshes them).
    A whole sampling loop is then `set x, t; replay() * T` -- no per-step host-side tensor ops.
    An inpainting step graph adds the RePaint blend and its counter after the step:
         known  [B, C, s, s]  the normalised image to keep; mask uint8 [B, mh, mw] (nonzero = known), both refreshed by
                              `set_cond`;
         z_known, z_renoise   the blend's two Gaussian draws (in-graph, or copied in like `noise`);
         u      [1] int32     the resample round at t, advanced with t by mi_inpaint_advance."""

    def __init__(self):
        self.graph = None
        self.x = self.t = self.noise = None
        self.known = self.mask = self.z_known = self.z_renoise = self.u = None
        self.cond = {}
        self.inject_noise = False
        self.unet = None

    def set_cond(self, known=None, mask=None, **tensors):
        for k, v in tensors.items():
            if v is not None:
                self.cond[k].copy_(v)
        if known is not None:
            self.known.copy_(known)
        if mask is not None:
            self.mask.copy_(mask)
        self.refresh_static()

    def refresh_static(self):
        """Step-invariant conditioning of the static buffers (eager, once per sampling loop): the text projection."""
        te = self.cond.get('text_embeds')
        if self.unet is not None and te is not None and te.dtype == F32:
            self.unet.register_static_text(te)

    def release(self):
        te = self.cond.get('text_embeds')
        if self.unet is not None and te is not None:
            self.unet.unregister_static_text(te)

    def replay(self):
        self.graph.replay()


class Imagen(nn.Module):
    def __init__(
            self,
            unets: Union[Unet, List[Unet], Tuple[Unet, ...]],
            *,
            text_encoder_name: str,
            image_sizes: Union[int, List[int], Tuple[int, ...]],
            text_embed_dim: int = None,
            channels: int = 3,
            timesteps: Union[int, List[int], Tuple[int, ...]] = 1000,
            cond_drop_prob: float = 0.1,
            loss_type: Literal["l1", "l2", "huber"] = 'l2',
            lowres_sample_noise_level: float = 0.2,
            auto_normalize_img: bool = True,
            dynamic_thresholding_percentile: float = 0.9,
            only_train_unet_number: int = None
    ):
        super().__init__()
        self.loss_type = loss_type
        self.loss_fn = self._set_loss_fn(loss_type)
        self.channels = channels

        unets = cast_tuple(unets)
        num_unets = len(unets)
        self.noise_schedulers = self._make_noise_schedulers(num_unets, timesteps)
        # NB like the reference (Imagen.py:78) this takes `timesteps` as is, i.e. it must be an int
        self.lowres_noise_schedule = GaussianDiffusion(timesteps=timesteps)

        self.text_encoder_name = text_encoder_name
        self.text_embed_dim = default(text_embed_dim, lambda: get_encoded_dim(text_encoder_name))
        self.unet_being_trained_index = -1
        self.only_train_unet_number = only_train_unet_number

        # first U-Net is the base model (no low-res conditioning), the others are super-resolution models; U-Nets whose
        # settings disagree are re-instantiated with fresh weights (Imagen.py:91-103)
        self.unets = nn.ModuleList([])
        for ind, one_unet in enumerate(unets):
            assert isinstance(one_unet, Unet)
            one_unet = one_unet._cast_model_parameters(
                lowres_cond=not (ind == 0), text_embed_dim=self.text_embed_dim, channels=self.channels,
                channels_out=self.channels)
            self.unets.append(one_unet)

        self.image_sizes = cast_tuple(image_sizes)
        assert num_unets == len(self.image_sizes), \
            f'you did not supply the correct number of u-nets ({len(self.unets)}) for resolutions {image_sizes}'
        self.sample_channels = cast_tuple(self.channels, num_unets)
        self.lowres_sample_noise_level = lowres_sample_noise_level

        self.cond_drop_prob = cond_drop_prob
        self.can_classifier_guidance = cond_drop_prob > 0.

        self.normalize_img = normalize_neg_one_to_one if auto_normalize_img else identity
        self.unnormalize_img = unnormalize_zero_to_one if auto_normalize_img else identity
        self.input_image_range = (0. if auto_normalize_img else -1., 1.)
        self.auto_normalize_img = auto_normalize_img
        self.dynamic_thresholding_percentile = dynamic_thresholding_percentile

        self.register_buffer('_temp', torch.tensor([0.]), persistent=False)
        self.to(next(self.unets.parameters()).device)

        # B200 additions (not part of the reference surface)
        self.use_cuda_graph = True       # replay each denoising step from a captured CUDA graph
        self.noise_fn: Callable = None   # see module docstring
        self.cfg_batched = False         # classifier-free guidance as ONE 2B-sample forward (not yet measured on B200)
        self._graphs = {}
        self.max_cached_graphs = 4

    # -------------------------------------------------------------------------------------------- bookkeeping
    @property
    def device(self):
        return self._temp.device

    @staticmethod
    def _set_loss_fn(loss_type):
        if loss_type == 'l1':
            return F.l1_loss
        if loss_type == 'l2':
            return F.mse_loss
        if loss_type == 'huber':
            return F.smooth_l1_loss
        raise NotImplementedError()

    @staticmethod
    def _make_noise_schedulers(num_unets, timesteps):
        timesteps = cast_tuple(timesteps, num_unets)
        return nn.ModuleList([GaussianDiffusion(timesteps=ts) for ts in timesteps])

    def _get_unet(self, unet_number):
        """Select the U-Net to train; like the reference (Imagen.py:180-203) the others are parked on the CPU."""
        assert 0 < unet_number <= len(self.unets)
        index = unet_number - 1
        if isinstance(self.unets, nn.ModuleList):
            unets_list = [unet for unet in self.unets]
            delattr(self, 'unets')
            self.unets = unets_list
        if index != self.unet_being_trained_index:
            for unet_index, unet in enumerate(self.unets):
                unet.to(self.device if unet_index == index else 'cpu')
        self.unet_being_trained_index = index
        return self.unets[index]

    def _reset_unets_all_one_device(self, device=None):
        device = default(device, self.device)
        self.unets = nn.ModuleList([*self.unets])
        self.unets.to(device)
        self.unet_being_trained_index = -1

    def state_dict(self, *args, **kwargs):
        self._reset_unets_all_one_device()
        return super().state_dict(*args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self._reset_unets_all_one_device()
        return super().load_state_dict(*args, **kwargs)

    @contextmanager
    def _one_unet_in_gpu(self, unet_number=None, unet=None):
        """Reference behaviour (Imagen.py:235-259) moves every other U-Net to the CPU for the duration of a stage.
        With 180 GB of HBM per B200 all U-Nets of the cascade stay resident (cfg 5's 2.85 B-parameter SR U-Net is
        11.4 GB in fp32), so this only makes sure the requested one is on the sampling device."""
        assert exists(unet_number) ^ exists(unet)
        if exists(unet_number):
            unet = self.unets[unet_number - 1]
        if module_device(unet) != self.device:
            unet.to(self.device)
        yield

    # -------------------------------------------------------------------------------------------- one reverse step
    def _noise(self, kind, shape, step, device):
        if exists(self.noise_fn):
            return self.noise_fn(kind, shape, step).to(device=device, dtype=F32).contiguous()
        return torch.randn(shape, device=device)

    def _p_mean_variance(self, unet, x, t, *, noise_scheduler, text_embeds=None, text_mask=None, lowres_cond_img=None,
                         lowres_noise_times=None, cond_scale=1., model_output=None):
        """Reference-compatible API (Imagen.py:261-326): (posterior mean, posterior variance, clipped log variance).
        Uses the same kernels as `_p_sample` (zero noise gives the mean)."""
        zeros = torch.zeros_like(x)
        mean = self._step(unet, x, t, zeros, noise_scheduler=noise_scheduler, text_embeds=text_embeds,
                          text_mask=text_mask, lowres_cond_img=lowres_cond_img, lowres_noise_times=lowres_noise_times,
                          cond_scale=cond_scale, model_output=model_output)
        shp = (x.shape[0], *((1,) * (x.dim() - 1)))
        return (mean, noise_scheduler.posterior_variance.gather(-1, t).reshape(shp),
                noise_scheduler.posterior_log_variance_clipped.gather(-1, t).reshape(shp))

    def _step(self, unet, x, t, noise, *, noise_scheduler, text_embeds, text_mask, lowres_cond_img, lowres_noise_times,
              cond_scale, model_output=None, out=None):
        """x_{t-1} = posterior_mean(x_t, clamp-thresholded x0(x_t, eps)) + [t != 0] * sigma_t * noise.
        `out` may be `x` itself (the captured step updates the image in place)."""
        with N.device_of(x):
            return self._step_impl(unet, x, t, noise, noise_scheduler=noise_scheduler, text_embeds=text_embeds,
                                   text_mask=text_mask, lowres_cond_img=lowres_cond_img,
                                   lowres_noise_times=lowres_noise_times, cond_scale=cond_scale,
                                   model_output=model_output, out=out)

    def _step_impl(self, unet, x, t, noise, *, noise_scheduler, text_embeds, text_mask, lowres_cond_img,
                   lowres_noise_times, cond_scale, model_output=None, out=None):
        assert not (cond_scale != 1. and not self.can_classifier_guidance), \
            'imagen was not trained with conditional dropout, and thus one cannot use classifier free guidance ' \
            '(cond_scale anything other than 1)'
        ops = get_ops()
        B = x.shape[0]
        n = x[0].numel()
        sch = noise_scheduler
        kw = dict(text_embeds=text_embeds, text_mask=text_mask, lowres_cond_img=lowres_cond_img,
                  lowres_noise_times=lowres_noise_times)
        eps_null = None
        if exists(model_output):
            eps = model_output.to(F32).contiguous()
        else:
            if cond_scale != 1 and self.cfg_batched:
                # conditional and unconditional pass as ONE batch of 2B (per-sample keep mask instead of two forwards)
                two = lambda v: torch.cat((v, v), dim=0) if exists(v) else None
                keep = torch.cat((torch.ones(B, dtype=torch.uint8, device=x.device),
                                  torch.zeros(B, dtype=torch.uint8, device=x.device)))
                both = unet._forward_impl(two(x), two(t), cond_keep=keep, **{k: two(v) for k, v in kw.items()})
                eps, eps_null = both[:B], both[B:]
            else:
                eps = unet.forward(x, t, **kw)
                if cond_scale != 1:
                    eps_null = unet.forward(x, t, cond_drop_prob=1., **kw)
        x = x.contiguous()
        lo, hi, w = quantile_rank(n, self.dynamic_thresholding_percentile)
        if out is None:
            out = torch.empty_like(x)
        # ONE kernel: CFG combine + x0 + exact dynamic-threshold quantile + clamp/divide + posterior mean + noise
        # (mi_step_epilogue; images too large for its register-resident select take the three-kernel form inside the ABI)
        ops.step_epilogue(x, eps, eps_null, cond_scale, t, sch.sqrt_recip_alphas_cumprod, sch.sqrt_recipm1_alphas_cumprod,
                          sch.posterior_mean_coef1, sch.posterior_mean_coef2, sch.sigma, noise, B, n, lo, hi, w, 1.0, out)
        return out

    @torch.no_grad()
    def _p_sample(self, unet, x, t, *, noise_scheduler, text_embeds=None, text_mask=None, lowres_cond_img=None,
                  lowres_noise_times=None, cond_scale=1., noise=None):
        """One reverse-diffusion step (reference Imagen.py:328-370).  `noise` defaults to a fresh N(0,1) draw, which --
        like the reference -- is drawn at every step, t == 0 included."""
        noise = default(noise, lambda: self._noise('step', x.shape, int(t[0].item()), x.device))
        return self._step(unet, x, t, noise.contiguous(), noise_scheduler=noise_scheduler, text_embeds=text_embeds,
                          text_mask=text_mask, lowres_cond_img=lowres_cond_img, lowres_noise_times=lowres_noise_times,
                          cond_scale=cond_scale)

    # -------------------------------------------------------------------------------------------- sampling loop
    def _graph_key(self, unet, shape, noise_scheduler, text_embeds, text_mask, lowres_cond_img, lowres_noise_times,
                   cond_scale, inpaint=None):
        sig = lambda v: None if v is None else (tuple(v.shape), str(v.dtype))
        p0 = next(unet.parameters())
        inpaint_sig = None if inpaint is None else (tuple(inpaint[1].shape), int(inpaint[2]))   # (mask shape, U)
        return (id(unet), tuple(shape), float(cond_scale), bool(self.cfg_batched), exists(self.noise_fn),
                noise_scheduler.num_timesteps, sig(text_embeds), sig(text_mask), sig(lowres_cond_img),
                sig(lowres_noise_times), p0.data_ptr(), sum(p._version for p in unet.parameters()),
                self.dynamic_thresholding_percentile, inpaint_sig)

    def clear_graphs(self):
        """Drop the captured step graphs (and the activation memory their pools hold)."""
        for g in getattr(self, "_graphs", {}).values():
            g.release()
        self._graphs = {}
        self.max_cached_graphs = 4

    def _step_graph(self, unet, shape, *, noise_scheduler, text_embeds, text_mask, lowres_cond_img,
                    lowres_noise_times, cond_scale, inpaint=None):
        """The captured step for this (unet, shape, conditioning signature, weights version): captured once, then reused by
        every later sampling loop of the same signature; the conditioning tensors are refreshed in its static buffers.
        `inpaint` = (known, mask uint8, U) captures the inpainting step instead: step, RePaint blend, advance of (t, u)."""
        device = self.device
        key = self._graph_key(unet, shape, noise_scheduler, text_embeds, text_mask, lowres_cond_img,
                              lowres_noise_times, cond_scale, inpaint)
        cond = dict(text_embeds=text_embeds, text_mask=text_mask, lowres_cond_img=lowres_cond_img,
                    lowres_noise_times=lowres_noise_times)
        known, mask, U = inpaint if inpaint is not None else (None, None, None)
        g = self._graphs.get(key)
        if g is not None:
            g.set_cond(known=known, mask=mask, **cond)
            return g
        if len(self._graphs) >= self.max_cached_graphs:
            self._graphs.pop(next(iter(self._graphs))).release()
        g = _StepGraph()
        g.unet = unet
        g.inject_noise = exists(self.noise_fn)
        g.x = torch.zeros(shape, dtype=F32, device=device)
        g.noise = torch.zeros(shape, dtype=F32, device=device)
        g.t = torch.zeros((shape[0],), dtype=torch.long, device=device)
        g.cond = {k: v.clone() for k, v in cond.items() if v is not None}
        kw = dict(noise_scheduler=noise_scheduler, cond_scale=cond_scale,
                  **{k: g.cond.get(k) for k in cond})
        g.refresh_static()
        ops = get_ops()
        if inpaint is not None:
            g.known, g.mask = known.clone(), mask.clone()
            g.z_known = torch.zeros(shape, dtype=F32, device=device)
            g.z_renoise = torch.zeros(shape, dtype=F32, device=device)
            g.u = torch.zeros((1,), dtype=torch.int32, device=device)
            sa, sb = noise_scheduler.inpaint_tables(device)

        def body():
            if not g.inject_noise:
                g.noise.normal_()                       # the reference's randn_like(x) (Imagen.py:361), graph-safe Philox
                if inpaint is not None:
                    g.z_renoise.normal_()
                    g.z_known.normal_()
            self._step(unet, g.x, g.t, g.noise, out=g.x, **kw)
            if inpaint is None:
                ops.step_advance_t(g.t, shape[0])       # t <- max(t - 1, 0): the next loop iteration's timestep
            else:
                ops.inpaint_blend(g.x, g.known, g.mask, g.z_known, g.z_renoise, g.t, g.u, U, 0,
                                  noise_scheduler.sqrt_alphas_cumprod, noise_scheduler.sqrt_one_minus_alphas_cumprod, sa, sb)
                ops.inpaint_advance(g.t, g.u, U, shape[0])   # (t, u) of the next replay

        # warm-up on a side stream (packs weights, sizes the caching allocator), then capture
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            body()
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        g.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g.graph):
            body()
        self._graphs[key] = g
        return g

    @staticmethod
    def _inpaint_schedule(T, U):
        """(t, u) of every step of an inpainting loop: U resample rounds at each t > 0, one at t = 0."""
        return [(t, u) for t in reversed(range(T)) for u in range(U if t > 0 else 1)]

    def _inpaint_loop(self, unet, shape, img, inpaint, max_steps, kw):
        """The sampling loop with RePaint inpainting (DESIGN.md 4.6): prime the known region at T-1, then per step of the
        schedule x <- step(x, t), blend (renoise back to t and redo, or paste the known region at t-1 / at 0), advance
        (t, u).  Injected noise is drawn as ('step', key), ('renoise', key) if the step renoises, ('inpaint', key) unless
        it is the final paste, with key = t * U + u; the prime draws ('inpaint', -1)."""
        known, mask, U = inpaint
        ops = get_ops()
        sch = kw['noise_scheduler']
        T, B, device = sch.num_timesteps, shape[0], img.device
        sa, sb = sch.inpaint_tables(device)
        tabs = (sch.sqrt_alphas_cumprod, sch.sqrt_one_minus_alphas_cumprod, sa, sb)
        steps = self._inpaint_schedule(T, U)
        if exists(max_steps):
            steps = steps[:max_steps]
        renoises = lambda t, u: u < (U if t > 0 else 1) - 1
        z_prime = self._noise('inpaint', shape, -1, device)
        if self.use_cuda_graph and img.is_cuda and len(steps) > 2:
            g = self._step_graph(unet, tuple(shape), inpaint=inpaint, **kw)
            g.x.copy_(img)
            g.t.fill_(T - 1)
            g.u.zero_()
            g.z_known.copy_(z_prime)
            ops.inpaint_blend(g.x, g.known, g.mask, g.z_known, g.z_renoise, g.t, g.u, U, 1, *tabs)
            for t, u in steps:
                if g.inject_noise:
                    key = t * U + u
                    g.noise.copy_(self._noise('step', shape, key, device))
                    if renoises(t, u):
                        g.z_renoise.copy_(self._noise('renoise', shape, key, device))
                    if t > 0:
                        g.z_known.copy_(self._noise('inpaint', shape, key, device))
                g.replay()                              # x <- blend(step(x)) in place, (t, u) advanced
            return g.x
        t_dev = torch.full((B,), T - 1, dtype=torch.long, device=device)
        u_dev = torch.zeros((1,), dtype=torch.int32, device=device)
        z_known = z_renoise = z_prime                   # z_renoise is only read by a renoising blend
        x = img.contiguous().clone()                    # the prime blends in place; img may be the caller's noise_fn draw
        ops.inpaint_blend(x, known, mask, z_known, z_renoise, t_dev, u_dev, U, 1, *tabs)
        for t, u in steps:
            key = t * U + u
            x = self._step(unet, x, t_dev, self._noise('step', shape, key, device), **kw)
            if renoises(t, u):
                z_renoise = self._noise('renoise', shape, key, device)
            if t > 0:
                z_known = self._noise('inpaint', shape, key, device)
            ops.inpaint_blend(x, known, mask, z_known, z_renoise, t_dev, u_dev, U, 0, *tabs)
            ops.inpaint_advance(t_dev, u_dev, U, B)
        return x

    @torch.no_grad()
    def _p_sample_loop(self, unet, shape, *, noise_scheduler, text_embeds=None, text_mask=None, lowres_cond_img=None,
                       lowres_noise_times=None, cond_scale=1., max_steps=None, out=None, inpaint=None):
        """Reverse diffusion from x_T ~ N(0, I) to x_0 (reference Imagen.py:372-420).  `max_steps` (not in the
        reference) stops after that many iterations -- used by the benchmark / parity harness; `out` (not in the
        reference) receives the finished images (e.g. this rank's slot of the all-gather buffer).  `inpaint` (not in the
        reference) = (known [B, C, s, s] normalised fp32, mask uint8 [B, mh, mw], U) runs the inpainting loop
        (`_inpaint_loop`); `max_steps` then counts its (T - 1) * U + 1 steps."""
        device = self.device
        with N.device_of(self._temp):
            ops = get_ops()
            lowres_cond_img = maybe(self.normalize_img)(lowres_cond_img)
            if exists(lowres_cond_img):
                lowres_cond_img = lowres_cond_img.to(F32).contiguous()
            batch = shape[0]
            timesteps = noise_scheduler._get_sampling_timesteps(batch, device=device)
            if exists(max_steps):
                timesteps = timesteps[:max_steps]
            img = self._noise('init', shape, -1, device)

            kw = dict(noise_scheduler=noise_scheduler, text_embeds=text_embeds, text_mask=text_mask,
                      lowres_cond_img=lowres_cond_img, lowres_noise_times=lowres_noise_times, cond_scale=cond_scale)
            if exists(inpaint):
                img = self._inpaint_loop(unet, shape, img, inpaint, max_steps, kw)
            elif self.use_cuda_graph and img.is_cuda and len(timesteps) > 2:
                g = self._step_graph(unet, tuple(shape), **kw)
                g.x.copy_(img)
                g.t.copy_(timesteps[0])
                for i in range(len(timesteps)):
                    if g.inject_noise:
                        g.noise.copy_(self._noise('step', shape, noise_scheduler.num_timesteps - 1 - i, device))
                    g.replay()                              # x <- x_{t-1} in place, t <- t - 1
                img = g.x
            else:
                for i, times in enumerate(timesteps):
                    noise = self._noise('step', shape, noise_scheduler.num_timesteps - 1 - i, device)
                    img = self._step(unet, img, times, noise, **kw)

            if out is None:
                out = torch.empty(tuple(shape), dtype=F32, device=device)
            ops.step_finalize(img.contiguous(), img.numel(), int(self.auto_normalize_img), out)   # clamp_(-1,1); (x+1)/2
            return out

    @torch.no_grad()
    @eval_decorator
    def sample(self, texts: List[str] = None, text_masks=None, text_embeds=None, cond_scale: float = 1.,
               lowres_sample_noise_level: float = None, return_pil_images: bool = False, device=None,
               distributed: bool = False, inpaint_images=None, inpaint_masks=None, inpaint_resample_times: int = 5):
        """Generate images (reference Imagen.py:422-510).  With `distributed=True` inside an initialised
        torch.distributed (NCCL) job, rank r samples rows [r*b/G, (r+1)*b/G) of the conditioning; the last stage's
        finalize kernel writes its images straight into this rank's slot of the gather buffer and ONE in-place
        all-gather returns the full batch on every rank.
        Inpainting (not in the reference; the keywords of imagen-pytorch): `inpaint_images` float (b, channels, H, H) in
        [0, 1] and `inpaint_masks` bool (b, H, H), True = keep that pixel of the image, False = generate it.  Every stage
        keeps the known region of the image resized to its size and re-runs each timestep `inpaint_resample_times` times
        (RePaint resampling), so each stage takes (T - 1) * inpaint_resample_times + 1 steps."""
        device = torch.device(default(device, self.device))
        self._reset_unets_all_one_device(device=device)
        if self._temp.device != device:
            self.to(device)
        with N.device_of(self._temp):
            return self._sample_impl(texts, text_masks, text_embeds, cond_scale, lowres_sample_noise_level,
                                     return_pil_images, device, distributed, inpaint_images, inpaint_masks,
                                     inpaint_resample_times)

    def _check_inpaint_args(self, inpaint_images, inpaint_masks, inpaint_resample_times, batch):
        U = inpaint_resample_times
        assert isinstance(U, int) and not isinstance(U, bool) and U >= 1, \
            f'inpaint_resample_times must be an int >= 1, got {U!r}'
        assert exists(inpaint_images) == exists(inpaint_masks), \
            'inpaint_images and inpaint_masks must be given together'
        if not exists(inpaint_images):
            return
        assert torch.is_tensor(inpaint_images) and inpaint_images.is_floating_point() and inpaint_images.dim() == 4, \
            f'inpaint_images must be a float tensor (b, {self.channels}, h, h)'
        b, c, h, w = inpaint_images.shape
        assert b == batch and c == self.channels and h == w, \
            f'inpaint_images must be ({batch}, {self.channels}, h, h), got {tuple(inpaint_images.shape)}'
        assert torch.is_tensor(inpaint_masks) and inpaint_masks.dtype == torch.bool and inpaint_masks.dim() == 3 \
            and inpaint_masks.shape[0] == batch, f'inpaint_masks must be a bool tensor ({batch}, h, h)'
        assert tuple(inpaint_masks.shape[-2:]) == (h, w), \
            f'inpaint_masks size {tuple(inpaint_masks.shape[-2:])} differs from the inpaint_images size {(h, w)}'

    def _sample_impl(self, texts, text_masks, text_embeds, cond_scale, lowres_sample_noise_level, return_pil_images,
                     device, distributed, inpaint_images=None, inpaint_masks=None, inpaint_resample_times=5):
        if exists(texts) and not exists(text_embeds):
            text_embeds, text_masks = t5_encode_text(texts, name=self.text_encoder_name)
            text_embeds, text_masks = map(lambda t: t.to(device), (text_embeds, text_masks))

        assert exists(text_embeds), 'text or text encodings must be passed into Imagen'
        assert not (exists(text_embeds) and text_embeds.shape[-1] != self.text_embed_dim), \
            f'invalid text embedding dimension being passed in (should be {self.text_embed_dim})'
        self._check_inpaint_args(inpaint_images, inpaint_masks, inpaint_resample_times, text_embeds.shape[0])
        inpainting = exists(inpaint_images)

        world, rank = 1, 0
        if distributed:
            import torch.distributed as dist
            assert dist.is_available() and dist.is_initialized(), 'distributed=True needs torch.distributed'
            world, rank = dist.get_world_size(), dist.get_rank()
            full_b = text_embeds.shape[0]
            assert full_b % world == 0, f'batch {full_b} must divide evenly over {world} ranks'
            per = full_b // world
            text_embeds = text_embeds[rank * per:(rank + 1) * per]
            text_masks = text_masks[rank * per:(rank + 1) * per] if exists(text_masks) else None
            if inpainting:
                inpaint_images = inpaint_images[rank * per:(rank + 1) * per]
                inpaint_masks = inpaint_masks[rank * per:(rank + 1) * per]

        batch_size = text_embeds.shape[0]
        text_embeds = text_embeds.to(device=device, dtype=F32).contiguous()
        text_masks = text_masks.to(device).contiguous() if exists(text_masks) else None
        lowres_sample_noise_level = default(lowres_sample_noise_level, self.lowres_sample_noise_level)
        ops = get_ops()
        if inpainting:
            inpaint_images = inpaint_images.to(device=device, dtype=F32).contiguous()
            inpaint_masks = inpaint_masks.to(device=device, dtype=torch.uint8).contiguous()

        img = None
        gathered = None
        n_stages = len(self.unets)
        for unet_number, unet, channel, image_size, noise_scheduler in zip(
                range(1, n_stages + 1), self.unets, self.sample_channels, self.image_sizes,
                self.noise_schedulers):
            with self._one_unet_in_gpu(unet=unet):
                lowres_cond_img = lowres_noise_times = None
                if unet.lowres_cond:
                    sch = self.lowres_noise_schedule
                    lowres_noise_times = sch._get_times(batch_size, lowres_sample_noise_level, device=device)
                    lowres_cond_img = resize_image_to(img, image_size, pad_mode='reflect').to(F32).contiguous()
                    aug_noise = self._noise('lowres', lowres_cond_img.shape, unet_number, device)
                    noised = torch.empty_like(lowres_cond_img)
                    # NB: like the reference (Imagen.py:483 vs :393) the [0,1] image is noised BEFORE normalisation
                    ops.q_sample(lowres_cond_img, aug_noise, lowres_noise_times, sch.sqrt_alphas_cumprod,
                                 sch.sqrt_one_minus_alphas_cumprod, batch_size, lowres_cond_img[0].numel(), 1.0, 0.0,
                                 noised)
                    lowres_cond_img = noised
                shape = (batch_size, self.channels, image_size, image_size)
                inpaint = None
                if inpainting:
                    # the image to keep at this stage's size, normalised like the sampling state (once per stage)
                    known = resize_image_to(inpaint_images, image_size, pad_mode='reflect')
                    known = self.normalize_img(known).to(F32).contiguous()
                    inpaint = (known, inpaint_masks, inpaint_resample_times)
                slot = None
                if distributed and world > 1 and unet_number == n_stages:
                    # the last stage finalises straight into this rank's slot of the all-gather buffer (no staging copy)
                    gathered = torch.empty((world * batch_size, *shape[1:]), dtype=F32, device=device)
                    slot = gathered[rank * batch_size:(rank + 1) * batch_size]
                img = self._p_sample_loop(unet, shape, text_embeds=text_embeds, text_mask=text_masks,
                                          cond_scale=cond_scale, lowres_cond_img=lowres_cond_img,
                                          lowres_noise_times=lowres_noise_times, noise_scheduler=noise_scheduler,
                                          out=slot, inpaint=inpaint)

        outputs = img
        if gathered is not None:
            import torch.distributed as dist
            dist.all_gather_into_tensor(gathered, img)      # in place: `img` IS gathered[rank slot]
            outputs = gathered

        if not return_pil_images:
            return outputs
        import torchvision.transforms as T
        return list(map(T.ToPILImage(), outputs.unbind(dim=0)))

    # -------------------------------------------------------------------------------------------- training
    def _p_losses(self, unet, x_start, times, *, noise_scheduler, lowres_cond_img=None, lowres_aug_times=None,
                  text_embeds=None, text_mask=None, noise=None):
        """Forward-diffuse the training images, predict the noise with `unet` and return the loss (reference
        Imagen.py:512-573).  The U-Net call runs under autograd (minimagen_b200/train_path.py): `loss.backward()` reaches every
        parameter through the library's backward kernels."""
        ops = get_ops()
        with N.device_of(x_start):
            x_start = x_start.to(F32)
            noise = default(noise, lambda: self._noise('train_noise', x_start.shape, -1, x_start.device))
            x_start = self.normalize_img(x_start).contiguous()
            lowres_cond_img = maybe(self.normalize_img)(lowres_cond_img)
            B, n = x_start.shape[0], x_start[0].numel()
            x_noisy = torch.empty_like(x_start)
            ops.q_sample(x_start, noise.to(F32).contiguous(), times, noise_scheduler.sqrt_alphas_cumprod,
                         noise_scheduler.sqrt_one_minus_alphas_cumprod, B, n, 1.0, 0.0, x_noisy)
            lowres_noisy = None
            if exists(lowres_cond_img):
                lowres_aug_times = default(lowres_aug_times, times)
                sch = self.lowres_noise_schedule
                lowres_cond_img = lowres_cond_img.to(F32).contiguous()
                aug = self._noise('train_lowres_noise', lowres_cond_img.shape, -1, lowres_cond_img.device)
                lowres_noisy = torch.empty_like(lowres_cond_img)
                ops.q_sample(lowres_cond_img, aug, lowres_aug_times, sch.sqrt_alphas_cumprod,
                             sch.sqrt_one_minus_alphas_cumprod, B, lowres_cond_img[0].numel(), 1.0, 0.0, lowres_noisy)
            pred = unet.forward(x_noisy, times, text_embeds=text_embeds, text_mask=text_mask,
                                lowres_noise_times=lowres_aug_times, lowres_cond_img=lowres_noisy,
                                cond_drop_prob=self.cond_drop_prob)
            return self.loss_fn(pred, noise)

    def graphed_train_step(self, optimizer, images, *, text_embeds, text_masks=None, unet_number: int = None, warmup: int = 3):
        """B200-side addition (no reference counterpart): capture `loss = self(images, ...); loss.backward(); optimizer.step()`
        for this batch SHAPE in ONE CUDA graph and return `step(images, text_embeds, text_masks=None) -> loss` that copies a new
        batch into the graph's static buffers and replays it.  An eager step of this path is bound by its ~2000 host-side
        launches (b = 8: 39 ms eager vs 18.5 ms replayed, `profiles/r02_train_step_vs_torch.txt`); the timestep / noise /
        conditioning-dropout draws are in-graph RNG calls, so every replay sees fresh randomness.  `optimizer` must be
        capturable (e.g. `torch.optim.Adam(params, lr, capturable=True)`); gradients are left in `.grad` after each step.
        Drop references to losses of earlier EAGER steps first (`del loss`): a live autograd graph keeps the parameters' gradient
        accumulators bound to the default stream, and CUDA refuses to make the legacy stream wait on a capturing one."""
        assert images.is_cuda, 'graphed_train_step captures a CUDA graph: move the model and the batch to the GPU first'
        static = [images.clone(), text_embeds.clone(), text_masks.clone() if exists(text_masks) else None]

        def one(zero=True):
            if zero:
                optimizer.zero_grad(set_to_none=True)
            loss = self(static[0], text_embeds=static[1], text_masks=static[2], unet_number=unet_number)
            loss.backward()
            optimizer.step()
            return loss

        side = torch.cuda.Stream(device=images.device)
        side.wait_stream(torch.cuda.current_stream(images.device))
        with torch.cuda.stream(side):                           # warm-up off the capture stream (lazy one-time initialisations)
            for _ in range(max(warmup, 1)):
                one()
        torch.cuda.current_stream(images.device).wait_stream(side)
        torch.cuda.synchronize(images.device)
        graph = torch.cuda.CUDAGraph()
        optimizer.zero_grad(set_to_none=True)
        with torch.cuda.graph(graph):
            loss = one(zero=False)

        def step(images, text_embeds, text_masks=None):
            static[0].copy_(images, non_blocking=True)
            static[1].copy_(text_embeds, non_blocking=True)
            if exists(static[2]):
                static[2].copy_(text_masks, non_blocking=True)
            graph.replay()
            return loss.detach()

        step.graph = graph
        return step

    def forward(self, images, texts: List[str] = None, text_embeds=None, text_masks=None, unet_number: int = None):
        """Training step: noise the images and return the U-Net's noise-prediction loss (reference Imagen.py:575-650)."""
        assert not (len(self.unets) > 1 and not exists(unet_number)), \
            f'you must specify which unet you want trained, from a range of 1 to {len(self.unets)}, ' \
            f'if you are training cascading DDPM (multiple unets)'
        unet_number = default(unet_number, 1)
        assert not exists(self.only_train_unet_number) or self.only_train_unet_number == unet_number, \
            f'you can only train on unet #{self.only_train_unet_number}'

        unet_index = unet_number - 1
        unet = self._get_unet(unet_number)
        noise_scheduler = self.noise_schedulers[unet_index]
        target_image_size = self.image_sizes[unet_index]
        prev_image_size = self.image_sizes[unet_index - 1] if unet_index > 0 else None
        b, c, h, w = images.shape
        device = images.device
        assert images.dim() == 4 and c == self.channels, f'images must be (b, {self.channels}, h, w)'
        assert h >= target_image_size and w >= target_image_size

        times = noise_scheduler._sample_random_times(b, device=device)

        if exists(texts) and not exists(text_embeds):
            assert len(texts) == len(images), 'number of text captions does not match up with the number of images given'
            text_embeds, text_masks = t5_encode_text(texts, name=self.text_encoder_name)
            text_embeds, text_masks = map(lambda t: t.to(images.device), (text_embeds, text_masks))

        assert exists(text_embeds), 'text or text encodings must be passed into decoder'
        assert not (exists(text_embeds) and text_embeds.shape[-1] != self.text_embed_dim), \
            f'invalid text embedding dimension being passed in (should be {self.text_embed_dim})'

        lowres_cond_img = lowres_aug_times = None
        with N.device_of(images):
            if exists(prev_image_size):
                lowres_cond_img = resize_image_to(images, prev_image_size, clamp_range=self.input_image_range,
                                                  pad_mode='reflect')
                lowres_cond_img = resize_image_to(lowres_cond_img, target_image_size, clamp_range=self.input_image_range,
                                                  pad_mode='reflect')
                lowres_aug_time = self.lowres_noise_schedule._sample_random_times(1, device=device)
                lowres_aug_times = lowres_aug_time.repeat(b)
            images = resize_image_to(images, target_image_size)

        return self._p_losses(unet, images, times, text_embeds=text_embeds, text_mask=text_masks,
                              noise_scheduler=noise_scheduler, lowres_cond_img=lowres_cond_img,
                              lowres_aug_times=lowres_aug_times)
