"""DiffSynthSampler -- B200 drop-in for the reference sampler (model/DiffSynthSampler.py).

Same constructor, same public methods and return values:
``respace``, ``activate_classifier_free_guidance``, ``q_sample``, ``sample``, ``img_guided_sample``,
``inpaint_sample``, ``interpolate`` -> ``(imgs: list[steps+1], initial_noise)``; ``ddim_invert`` is a port extension (DDIM inversion,
no reference entry) in the same convention.

What runs where:
  * schedule tables / respacing: numpy float64 on the host, as in the reference (:55-57,169-222);
  * the per-step arithmetic (CFG combine + DDIM/DDPM update, q_sample, inpaint blend): one fused CUDA
    kernel per step (ds_ddim_step / ds_q_sample / ds_mask_blend);
  * with a ``diffusynth_b200.ConditionedUnet`` the whole step sequence -- CFG-doubled U-Net + update, for all
    steps -- is captured once in a CUDA graph and replayed; any other callable ``model(x, t, cond)`` is
    driven step by step like the reference does.
RNG contract: like the reference, noise comes from ``torch.randn`` on the sampler device under the global
generator (``seed`` -> ``torch.manual_seed``); ``noise_feed`` lets tests inject host-generated draws."""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import os

import numpy as np
import torch

from . import engine, ops
from .unet import ConditionedUnet


def _column_map(width: int, train_width: int) -> Tuple[List[int], List[int]]:
    """Column gather map of the 'repeat' noise layout (reference :97-167): which training-noise column feeds
    each output column, plus the concat points."""
    rel = int(train_width * 1.0 / 4)
    body = train_width - rel
    tail = list(range(train_width - rel, train_width))
    if width <= train_width:
        head_w = int((width - rel) / 2)
        tail_w = width - rel - head_w
        segs = [list(range(0, head_w)), list(range(body - tail_w, body)) if tail_w > 0 else list(range(0, body)), tail]
    else:
        reps, extra = (width - rel) // body, (width - rel) % body
        hw = int(body / 2)
        mid0 = (body - extra) // 2
        segs = [list(range(0, hw))] * reps + [list(range(mid0, mid0 + extra))] + [list(range(hw, body))] * reps + [tail]
    pts = [0]
    for s in segs[:-1]:
        pts.append(pts[-1] + len(s))
    return [c for s in segs for c in s], pts


class DiffSynthSampler:
    def __init__(self, timesteps, beta_start=0.0001, beta_end=0.02, device=None, mute=False, height=128, max_batchsize=16,
                 max_width=256, channels=4, train_width=64, noise_strategy="repeat"):
        if device is None:
            self.device = "cuda" if torch.cuda.is_available() else "cpu"
        else:
            self.device = device
        if torch.device(self.device).type != "cuda":
            raise RuntimeError("diffusynth_b200.DiffSynthSampler runs on a CUDA device only (there is no CPU fallback)")
        self.height, self.train_width, self.max_batchsize = height, train_width, max_batchsize
        self.max_width, self.channels = max_width, channels
        self.num_timesteps = timesteps
        self.timestep_map = list(range(timesteps))
        self.betas = np.array(np.linspace(beta_start, beta_end, timesteps), dtype=np.float64)
        self.respaced = False
        self.define_beta_schedule()
        self.CFG = 1.0
        self.unconditional_condition = None
        self.mute = mute
        self.noise_strategy = noise_strategy
        self.noise_feed: Optional[torch.Tensor] = None     # [K, >=B, C, H, train_width]; consumed in draw order
        self._feed_pos = 0
        # The reference draws the per-step noise even when eta == 0 (:340), which advances the global RNG; True reproduces that RNG
        # state after sample() at the cost of n_iter discarded randn launches (TextToTimbre leaves it on).
        self.faithful_rng = True
        self._graphs: Dict[tuple, "_GraphLoop"] = {}
        self.last_graph_launches = 0
        # Optional continuation captured in the SAME CUDA graph as the step loop (TextToTimbre: quantiser -> decoder -> iSTFT):
        # a callable ``factory(final_latent_buffer) -> object with .run() and .num_launches``; ``last_tail`` is the tail whose
        # static output buffers the last graph launch filled.  ``final_only`` skips the copy of the per-step latents.
        self.graph_tail = None
        self.last_tail = None
        self.final_only = False
        # 'repeat' strategy: the train-width noise [B,C,H,train_width] the last p_sample_loop re-laid into its initial noise
        self.last_reference_noise: Optional[torch.Tensor] = None

    # ---- schedule (host, float64) -----------------------------------------------------------
    def define_beta_schedule(self):
        assert self.respaced == False, "This schedule has already been respaced!"
        b = self.betas
        self.alphas = 1.0 - b
        ac = np.cumprod(self.alphas, axis=0)
        self.alphas_cumprod = ac
        self.alphas_cumprod_prev = np.append(1.0, ac[:-1])
        self.alphas_cumprod_next = np.append(ac[1:], 0.0)
        self.sqrt_alphas_cumprod = np.sqrt(ac)
        self.sqrt_one_minus_alphas_cumprod = np.sqrt(1.0 - ac)
        self.log_one_minus_alphas_cumprod = np.log(1.0 - ac)
        self.sqrt_recip_alphas_cumprod = np.sqrt(1.0 / ac)
        self.sqrt_recip_alphas = np.sqrt(1.0 / self.alphas)
        self.sqrt_recipm1_alphas_cumprod = np.sqrt(1.0 / ac - 1)
        self.posterior_variance = b * (1.0 - self.alphas_cumprod_prev) / (1.0 - ac)

    def activate_classifier_free_guidance(self, CFG, unconditional_condition):
        assert (not unconditional_condition is None) or CFG == 1.0, \
            "For CFG != 1.0, unconditional_condition must be available"
        self.CFG = CFG
        self.unconditional_condition = unconditional_condition

    def respace(self, use_timesteps=None):
        if use_timesteps is None:
            return
        assert self.respaced == False, "This schedule has already been respaced!"
        keep = set(int(i) for i in use_timesteps)
        last, new_betas, tmap = 1.0, [], []
        for i, a in enumerate(self.alphas_cumprod):
            if i in keep:
                new_betas.append(1 - a / last)
                last = a
                tmap.append(i)
        self.timestep_map = tmap
        self.num_timesteps = len(use_timesteps)
        self.betas = np.array(new_betas)
        self.define_beta_schedule()
        self.respaced = True

    def _coef(self, t: int, eta: float) -> List[float]:
        """Per-step scalars of :323-337, evaluated as the reference does: f64 table -> fp32 -> fp32 math."""
        at = torch.tensor(self.alphas_cumprod[t]).float()
        ap = torch.tensor(self.alphas_cumprod_prev[t]).float()
        sigma = eta * torch.sqrt((1 - ap) / (1 - at)) * torch.sqrt(1 - at / ap)
        return [float(torch.sqrt(1. - at)), float(torch.sqrt(at)), float(torch.sqrt(ap)), float(torch.sqrt(1 - ap - sigma ** 2)),
                float(sigma), float(self.CFG), 0.0, 0.0]

    # ---- noise --------------------------------------------------------------------------------
    def _draw(self, batchsize: int) -> torch.Tensor:
        if self.noise_feed is not None:
            z = self.noise_feed[self._feed_pos][:batchsize].to(self.device, torch.float32)
            self._feed_pos += 1
            return z
        return torch.randn((self.max_batchsize, self.channels, self.height, self.train_width), device=self.device)[:batchsize]

    def get_deterministic_noise_tensor_non_repeat(self, batchsize, width, reference_noise=None):
        if reference_noise is None:
            big = torch.randn((self.max_batchsize, self.channels, self.height, self.max_width), device=self.device)
        else:
            assert reference_noise.shape == (batchsize, self.channels, self.height, self.max_width), "reference_noise shape mismatch"
            big = reference_noise
        return big[:batchsize, :, :, :width], None

    def get_deterministic_noise_tensor_repeat(self, batchsize, width, reference_noise=None):
        if reference_noise is None:
            base = self._draw(batchsize)
        else:
            assert reference_noise.shape == (batchsize, self.channels, self.height, self.train_width), "reference_noise shape mismatch"
            base = reference_noise
        cols, pts = _column_map(width, self.train_width)
        if width == self.train_width:
            return base[:batchsize], pts
        idx = torch.tensor(cols, device=base.device, dtype=torch.long)
        return base[:batchsize].index_select(3, idx), pts

    def get_deterministic_noise_tensor(self, batchsize, width, reference_noise=None):
        if self.noise_strategy == "repeat":
            return self.get_deterministic_noise_tensor_repeat(batchsize, width, reference_noise=reference_noise)
        return self.get_deterministic_noise_tensor_non_repeat(batchsize, width, reference_noise=reference_noise)

    def generate_linear_noise(self, shape, variance=1.0, first_endpoint=None, second_endpoint=None):
        """Linear noise trajectories for ``interpolate`` (reference :224-269)."""
        assert shape[1] == self.channels, "shape[1] != self.channels"
        assert shape[2] == self.height, "shape[2] != self.height"
        noise = torch.empty(*shape, device=self.device)
        if first_endpoint is not None and second_endpoint is not None:
            for i in range(shape[0]):
                a = i / (shape[0] - 1)
                noise[i] = a * second_endpoint + (1 - a) * first_endpoint
            return noise
        if first_endpoint is not None:
            noise[0] = first_endpoint
        else:
            noise[0] = self.get_deterministic_noise_tensor(1, shape[3])[0][0]
        if shape[0] > 1:
            noise[1] = self.get_deterministic_noise_tensor(1, shape[3])[0][0]
        for i in range(2, shape[0]):
            noise[i] = 2 * noise[i - 1] - noise[i - 2]
        noise = noise * torch.sqrt(variance / noise.var())
        if first_endpoint is not None:
            noise += first_endpoint - noise[0]
        return noise

    # ---- single operations ------------------------------------------------------------------
    def q_sample(self, x_start, t, noise=None):
        """q(x_t | x_0) (:271-294).  ``t`` int tensor [B] (one shared value, as every caller passes)."""
        assert x_start.shape[1] == self.channels, "shape[1] != self.channels"
        assert x_start.shape[2] == self.height, "shape[2] != self.height"
        if noise is None:
            noise, _ = self.get_deterministic_noise_tensor(x_start.shape[0], x_start.shape[3])
        assert noise.shape == x_start.shape
        tv = [int(v) for v in torch.as_tensor(t).reshape(-1).tolist()]
        x0 = x_start.to(self.device, torch.float32).contiguous()
        nz = noise.to(self.device, torch.float32).contiguous()
        out = torch.empty_like(x0)
        if all(v == tv[0] for v in tv):
            coef = torch.tensor([np.float32(self.sqrt_alphas_cumprod[tv[0]]), np.float32(self.sqrt_one_minus_alphas_cumprod[tv[0]])],
                                dtype=torch.float32, device=self.device)
            ops.q_sample(x0, nz, coef, out)
        else:       # per-sample timesteps: one coefficient pair per batch element, gathered like _extract_into_tensor (:6-22)
            assert len(tv) == x0.shape[0], "t must hold one timestep per sample"
            coef = torch.tensor([[np.float32(self.sqrt_alphas_cumprod[v]), np.float32(self.sqrt_one_minus_alphas_cumprod[v])] for v in tv],
                                dtype=torch.float32, device=self.device)
            ops.q_sample(x0, nz, coef, out, per_sample=x0[0].numel())
        return out

    @torch.no_grad()
    def ddim_sample(self, model, x, t, condition=None, ddim_eta=0.0, coef=None):
        """One reverse step (:297-345) for a generic callable model; the update is the fused kernel.  ``coef``: the step's 8
        ds_ddim_step coefficients instead of _coef(t, ddim_eta), with no noise draw (sigma must be 0; ddim_invert)."""
        B = x.shape[0]
        ti = int(t.reshape(-1)[0])
        mapped = torch.full((B,), self.timestep_map[ti], device=x.device, dtype=torch.long)
        if self.CFG == 1.0:
            eps_u, eps_c = None, model(x, mapped, condition).float().contiguous()
        else:
            u = self.unconditional_condition.unsqueeze(0).repeat(*([B] + [1] * len(self.unconditional_condition.shape)))
            out = model(torch.cat([x] * 2), torch.cat([mapped] * 2), torch.cat([u.to(condition.device), condition])).float().contiguous()
            eps_u, eps_c = out[:B], out[B:]
        z = None
        if coef is None:
            z, _ = self.get_deterministic_noise_tensor(B, x.shape[3])
            z = z.contiguous()
            coef = self._coef(ti, ddim_eta)
        coef = torch.tensor(coef, dtype=torch.float32, device=x.device)
        xin = x.float().contiguous()
        nxt = torch.empty_like(xin)
        ops.ddim_step(eps_u, eps_c, xin, z, coef, nxt)
        return nxt

    def p_sample(self, model, x, t, condition=None, sampler="ddim"):
        if sampler == "ddim":
            return self.ddim_sample(model, x, t, condition=condition, ddim_eta=0.0)
        elif sampler == "ddpm":
            return self.ddim_sample(model, x, t, condition=condition, ddim_eta=1.0)
        raise NotImplementedError()

    def get_dynamic_masks(self, n_masks, shape, concat_points, mask_flexivity=0.8):
        """Shrinking freeze masks for arrangement synthesis (:365-422): 1 = keep guide, 0 = regenerate."""
        rel = int(self.train_width / 4)
        assert shape[3] == (concat_points[-1] + rel), "shape[3] != (concat_points[-1] + release_length)"
        seg = [concat_points[i + 1] - concat_points[i] for i in range(len(concat_points) - 1)]
        n_guided = int(n_masks * mask_flexivity)
        masks = []
        for i in range(n_guided):
            m = torch.zeros((shape[0], 1, shape[2], shape[3]), dtype=torch.float32, device=self.device)
            m[..., shape[3] - rel:] = 1.0
            for k, length in enumerate(seg):
                keep = int((n_guided - 1 - i) / (n_guided - 1) * length)
                if k == 0:
                    m[..., :keep] = 1.0
                elif k == len(seg) - 1:
                    if keep != 0:
                        m[..., shape[3] - keep - rel:] = 1.0
                else:
                    s = concat_points[k] + int((length - keep) / 2)
                    m[..., s:s + keep] = 1.0
            masks.append(m)
        for _ in range(n_masks - n_guided):
            m = torch.zeros((shape[0], 1, shape[2], shape[3]), dtype=torch.float32, device=self.device)
            m[..., shape[3] - rel:] = 1.0
            masks.append(m)
        masks.reverse()
        return masks

    # ---- the loop -------------------------------------------------------------------------------
    @torch.no_grad()
    def p_sample_loop(self, model, shape, initial_noise=None, start_noise_level_ratio=1.0, end_noise_level_ratio=0.0,
                      return_tensor=False, condition=None, guide_img=None, mask=None, sampler="ddim", inpaint=False,
                      use_dynamic_mask=False, mask_flexivity=0.8):
        assert shape[1] == self.channels, "shape[1] != self.channels"
        assert shape[2] == self.height, "shape[2] != self.height"
        if sampler not in ("ddim", "ddpm"):
            raise NotImplementedError()
        eta = 0.0 if sampler == "ddim" else 1.0
        self._feed_pos = 0
        shape = tuple(int(s) for s in shape)
        B, Wd = shape[0], shape[3]
        if initial_noise is not None:
            initial_noise = initial_noise.to(self.device, torch.float32)
        elif self.noise_strategy == "repeat":
            initial_noise = self._draw(B)           # the draw get_deterministic_noise_tensor_repeat would make, kept below
        self.last_reference_noise = initial_noise if self.noise_strategy == "repeat" else None
        initial_noise, _ = self.get_deterministic_noise_tensor(B, Wd, reference_noise=initial_noise)
        initial_noise = initial_noise.contiguous()
        assert tuple(initial_noise.shape) == shape, "initial_noise.shape != shape"
        start = int(self.num_timesteps * start_noise_level_ratio)
        end = int(self.num_timesteps * end_noise_level_ratio)
        assert (start_noise_level_ratio == 1.0) or (not guide_img is None), "A guide_img must be given to sample from a non-pure-noise."
        concat_points = None
        if guide_img is None:
            img = initial_noise
        else:
            guide_img, concat_points = self.get_deterministic_noise_tensor_repeat(B, Wd, reference_noise=guide_img.to(self.device, torch.float32))
            guide_img = guide_img.contiguous()
            assert tuple(guide_img.shape) == shape, "guide_img.shape != shape"
            if start > 0:
                img = self.q_sample(guide_img, torch.full((B,), start - 1, device=self.device).long(), noise=initial_noise)
            else:
                print("Zero noise added to the guidance latent representation.")
                img = guide_img
        n_iter = start - end
        if use_dynamic_mask:
            masks = self.get_dynamic_masks(n_iter, shape, concat_points, mask_flexivity)
        else:
            if inpaint and mask is not None:
                mask = ops.normalize_mask(mask, shape, self.device)       # [B,1,H,W] or [B,C,H,W], as the reference's callers pass
            masks = [mask for _ in range(n_iter)]
        steps = list(reversed(range(end, start)))

        if isinstance(model, ConditionedUnet) and condition is not None and n_iter > 0:
            imgs = self._run_graph_loop(model, shape, img, steps, eta, condition, guide_img, initial_noise, masks, inpaint)
        else:
            imgs = self._run_generic_loop(model, img, steps, eta, condition, guide_img, initial_noise, masks, inpaint, sampler)
        if not return_tensor:
            imgs = [imgs[0]] + [im.cpu().numpy() for im in imgs[1:]]
        return imgs, initial_noise

    def _run_generic_loop(self, model, img, steps, eta, condition, guide_img, initial_noise, masks, inpaint, sampler):
        imgs = [img]
        masks = list(masks)
        current_mask = None
        B = img.shape[0]
        for i in steps:
            img = self.p_sample(model, img, torch.full((B,), i, device=self.device, dtype=torch.long), condition=condition, sampler=sampler)
            if inpaint:
                if i > 0:
                    current_mask = masks.pop()
                    coef = torch.tensor([np.float32(self.sqrt_alphas_cumprod[i - 1]), np.float32(self.sqrt_one_minus_alphas_cumprod[i - 1])],
                                        dtype=torch.float32, device=self.device)
                else:
                    coef = torch.tensor([1.0, 0.0], dtype=torch.float32, device=self.device)
                ops.mask_blend(guide_img, initial_noise, ops.normalize_mask(current_mask, img.shape, self.device), coef, img)
            imgs.append(img)
        return imgs

    def _run_graph_loop(self, model, shape, img, steps, eta, condition, guide_img, initial_noise, masks, inpaint, coef=None):
        """``coef``: per-step ds_ddim_step coefficients instead of _coef(i, eta), with no per-step noise draw (ddim_invert)."""
        B, Cc, H, Wd = shape
        cfg_on = self.CFG != 1.0
        n_iter = len(steps)
        # the captured graph points at the model's packed weights: a repack (load_state_dict / .to) bumps weights_version and
        # retires every loop built on the old tensors; the loop also holds the model, so its id() cannot be recycled
        key = (id(model), model.weights_version, shape, n_iter, eta > 0, cfg_on, inpaint, id(self.graph_tail) if self.graph_tail else 0)
        loop = self._graphs.get(key)
        if loop is None:
            for k in [k for k, v in self._graphs.items() if v.model is model and k[1] != model.weights_version]:
                del self._graphs[k]
            loop = _GraphLoop(self, model, shape, n_iter, eta > 0, cfg_on, inpaint, self.graph_tail)
            self._graphs[key] = loop
        # per-call inputs (device buffers the graph reads)
        loop.imgs[0].copy_(img)
        draw_steps = coef is None
        if coef is None:
            coef = [self._coef(i, eta) for i in steps]
        loop.coef.copy_(torch.tensor(coef, dtype=torch.float32))
        loop.ttab.copy_(torch.tensor([self.timestep_map[i] for i in steps], dtype=torch.long))
        cond = condition.to(self.device, loop.cond.dtype)          # fp32 [B, L] text conditions, or int64 [B] class labels
        if cfg_on:
            u = self.unconditional_condition.to(self.device, loop.cond.dtype)
            u = u.reshape(1, -1).expand(B, -1) if cond.dim() == 2 else u.reshape(1).expand(B)       # :313-314
            loop.cond.copy_(torch.cat([u, cond]))
        else:
            loop.cond.copy_(cond)
        if draw_steps and (eta > 0 or self.faithful_rng):
            for k in range(n_iter):
                z, _ = self.get_deterministic_noise_tensor(B, Wd)
                if eta > 0:
                    loop.noise[k].copy_(z)
        if inpaint:
            ms = list(masks)
            cur = None
            ab = []
            for k, i in enumerate(steps):
                if i > 0:
                    cur = ms.pop()
                    ab.append([np.float32(self.sqrt_alphas_cumprod[i - 1]), np.float32(self.sqrt_one_minus_alphas_cumprod[i - 1])])
                else:
                    ab.append([1.0, 0.0])
                loop.masks[k].copy_(ops.normalize_mask(cur, shape, self.device).expand(B, Cc, H, Wd))
            loop.blend_coef.copy_(torch.tensor(ab, dtype=torch.float32))
            loop.guide.copy_(guide_img)
            loop.init_noise.copy_(initial_noise)
        loop.launch()               # (the step-invariant condition projections run once per call, ahead of the graph)
        self.last_graph_launches = loop.launches
        self.last_tail = loop.tail
        if self.final_only:         # (pipeline use: only imgs[0] and imgs[-1] are read)
            first, last = loop.imgs[0].clone(), loop.imgs[n_iter].clone()
            return [first] + [None] * (n_iter - 1) + [last]
        out = loop.imgs.clone()
        return [out[k] for k in range(n_iter + 1)]

    # ---- entry points ---------------------------------------------------------------------------
    def sample(self, model, shape, return_tensor=False, condition=None, sampler="ddim", initial_noise=None, seed=None):
        if not seed is None:
            torch.manual_seed(seed)
        return self.p_sample_loop(model, shape, initial_noise=initial_noise, start_noise_level_ratio=1.0, end_noise_level_ratio=0.0,
                                  return_tensor=return_tensor, condition=condition, sampler=sampler)

    def interpolate(self, model, shape, variance, first_endpoint=None, second_endpoint=None, return_tensor=False, condition=None,
                    sampler="ddim", seed=None):
        if not seed is None:
            torch.manual_seed(seed)
        linear_noise = self.generate_linear_noise(shape, variance, first_endpoint=first_endpoint, second_endpoint=second_endpoint)
        return self.p_sample_loop(model, shape, initial_noise=linear_noise, start_noise_level_ratio=1.0, end_noise_level_ratio=0.0,
                                  return_tensor=return_tensor, condition=condition, sampler=sampler)

    def _invert_coef(self, t: int) -> List[float]:
        """ds_ddim_step coefficients of inversion step t (x_t -> x_next): [sqrt(1-a_t), sqrt(a_t), sqrt(a_next), sqrt(1-a_next), 0,
        CFG, 0, 0] from alphas_cumprod / alphas_cumprod_next, evaluated as _coef is (f64 table -> fp32 -> fp32 math)."""
        at = torch.tensor(self.alphas_cumprod[t]).float()
        an = torch.tensor(self.alphas_cumprod_next[t]).float()
        return [float(torch.sqrt(1. - at)), float(torch.sqrt(at)), float(torch.sqrt(an)), float(torch.sqrt(1. - an)), 0.0,
                float(self.CFG), 0.0, 0.0]

    @torch.no_grad()
    def ddim_invert(self, model, x0, condition, return_tensor=True):
        """DDIM inversion (a port extension: the reference has no entry for it): the latents ``x0`` [B,C,H,train_width] are run
        through the respaced timesteps in ASCENDING order, step t mapping x_t to sqrt(a_next) x0_pred + sqrt(1 - a_next) eps with the
        schedule's alphas_cumprod_next (0 after the last step, so the result is the model's noise prediction), under the active
        classifier-free guidance.  With a ConditionedUnet the steps run through the same captured graph as sample() (no tail).
        Returns ``(imgs, None)``: imgs[0] = x0, imgs[k] after k steps, imgs[-1] the noise; numpy after imgs[0] unless return_tensor.
        Only the 'repeat' strategy at the train width is supported."""
        if self.noise_strategy != "repeat":
            raise NotImplementedError("ddim_invert supports the 'repeat' noise strategy only")
        shape = tuple(int(s) for s in x0.shape)
        if len(shape) != 4 or shape[1:] != (self.channels, self.height, self.train_width):
            raise ValueError(f"x0 must be [B, {self.channels}, {self.height}, {self.train_width}], got {shape}")
        if condition is None:
            raise ValueError("ddim_invert needs a condition")
        steps = list(range(0, self.num_timesteps))
        coef = [self._invert_coef(i) for i in steps]
        img = x0.to(self.device, torch.float32).contiguous()
        if isinstance(model, ConditionedUnet):
            tail, self.graph_tail = self.graph_tail, None
            try:
                imgs = self._run_graph_loop(model, shape, img, steps, 0.0, condition, None, None, None, False, coef=coef)
            finally:
                self.graph_tail = tail
        else:
            imgs = [img]
            for i, c in zip(steps, coef):
                imgs.append(self.ddim_sample(model, imgs[-1], torch.full((shape[0],), i, device=self.device, dtype=torch.long),
                                             condition=condition, coef=c))
        if not return_tensor:
            imgs = [imgs[0]] + [im.cpu().numpy() for im in imgs[1:]]
        return imgs, None

    def img_guided_sample(self, model, shape, noising_strength, guide_img, return_tensor=False, condition=None, sampler="ddim",
                          initial_noise=None, seed=None):
        if not seed is None:
            torch.manual_seed(seed)
        assert guide_img.shape[-1] == shape[-1], "guide_img.shape[:-1] != shape[:-1]"
        return self.p_sample_loop(model, shape, start_noise_level_ratio=noising_strength, end_noise_level_ratio=0.0,
                                  return_tensor=return_tensor, condition=condition, sampler=sampler, guide_img=guide_img,
                                  initial_noise=initial_noise)

    def inpaint_sample(self, model, shape, noising_strength, guide_img, mask, return_tensor=False, condition=None, sampler="ddim",
                       initial_noise=None, use_dynamic_mask=False, end_noise_level_ratio=0.0, seed=None, mask_flexivity=0.8):
        if not seed is None:
            torch.manual_seed(seed)
        return self.p_sample_loop(model, shape, start_noise_level_ratio=noising_strength, end_noise_level_ratio=end_noise_level_ratio,
                                  return_tensor=return_tensor, condition=condition, guide_img=guide_img, mask=mask, sampler=sampler,
                                  inpaint=True, initial_noise=initial_noise, use_dynamic_mask=use_dynamic_mask,
                                  mask_flexivity=mask_flexivity)


def _profiler_attached() -> bool:
    """True inside `ncu ...` (its injection library is named in the child's environment)."""
    inj = os.environ.get("CUDA_INJECTION64_PATH", "") + os.environ.get("NV_COMPUTE_PROFILER_PERFWORKS_DIR", "")
    return "nsight-compute" in inj.lower() or "nsight_compute" in inj.lower() or bool(os.environ.get("NV_COMPUTE_PROFILER_PERFWORKS_DIR"))


class _GraphLoop:
    """All steps of one sampling call -- U-Net (CFG-doubled) + fused update (+ inpaint blend) -- captured in one CUDA graph.
    Step-dependent scalars (timestep, update coefficients, masks, noise) live in device tables the graph reads, so the
    same graph serves any schedule / seed / prompt of the same shape and step count."""

    def __init__(self, sampler: DiffSynthSampler, model: ConditionedUnet, shape, n_iter: int, stochastic: bool, cfg_on: bool, inpaint: bool,
                 tail_factory=None):
        dev = sampler.device
        B, Cc, H, Wd = shape
        f32 = dict(dtype=torch.float32, device=dev)
        self.n_iter, self.cfg_on = n_iter, cfg_on
        self.model = model
        self.imgs = torch.zeros((n_iter + 1, B, Cc, H, Wd), **f32)
        self.coef = torch.zeros((n_iter, 8), **f32)
        self.ttab = torch.zeros((n_iter,), dtype=torch.long, device=dev)
        self.noise = torch.zeros((n_iter, B, Cc, H, Wd), **f32) if stochastic else None
        if inpaint:
            self.masks = torch.zeros((n_iter, B, Cc, H, Wd), **f32)      # per channel: the reference broadcasts any mask shape
            self.blend_coef = torch.zeros((n_iter, 2), **f32)
            self.guide = torch.zeros((B, Cc, H, Wd), **f32)
            self.init_noise = torch.zeros((B, Cc, H, Wd), **f32)
        N = 2 * B if cfg_on else B
        self.N, self.shape = N, (B, Cc, H, Wd)
        self.inpaint = inpaint
        self.B = B
        self._plan = None
        self.sgraph = None
        self.graph = None
        # Nsight Compute dies on the first thread-block-cluster launch inside a stream capture (ncu exit code 9, seen on 2025.x with
        # CUDA 12.9): under its injection library, or with DS_NO_GRAPH=1, the same launches run eagerly so that the profiler's launch
        # list covers every kernel of the loop and the tail.  Results are identical (tests/test_gpu_abi_engine.py); timings are not
        # bench values either way.
        use_graph = os.environ.get("DS_NO_GRAPH", "0") != "1" and not _profiler_attached()
        if getattr(model, "_engine", None) is not None and model.use_engine:
            # module-level C ABI: the plan, the capture and the replay live in the library (ds_sample_graph_build / _run)
            self.cond = torch.zeros((N,), dtype=torch.long, device=dev) if model.cfg["condition_type"] == "instrument_family" \
                else torch.zeros((N, model.cfg["label_emb_dim"]), **f32)
            self.tail = tail_factory.buffers(self.imgs[n_iter]) if tail_factory is not None else None
            b = engine.SampleBuffers()
            b.d_imgs, b.d_coef, b.d_ttab, b.d_cond = self.imgs.data_ptr(), self.coef.data_ptr(), self.ttab.data_ptr(), self.cond.data_ptr()
            b.d_noise = self.noise.data_ptr() if self.noise is not None else None
            if inpaint:
                b.d_guide, b.d_init_noise = self.guide.data_ptr(), self.init_noise.data_ptr()
                b.d_masks, b.d_blend_coef = self.masks.data_ptr(), self.blend_coef.data_ptr()
            if self.tail is not None:
                t = self.tail
                b.d_quantized, b.d_indices, b.d_spec, b.d_wave = t.q.data_ptr(), t.idx.data_ptr(), t.spec.data_ptr(), t.wave.data_ptr()
            self.sgraph = engine.SampleGraph(model._engine, tail_factory.vqgan._engine if self.tail is not None else None, b, B, H, Wd,
                                             n_iter, cfg_on, use_graph=use_graph)
            self.launches = self.sgraph.launches
            self.has_tail = self.tail is not None
            return
        # operator-level path (the other U-Net variants; A/B against the library's graph): Python plan + torch.cuda.graph
        self._plan = model.plan(N, H, Wd, x_batch_mod=B if cfg_on else 0, uniform_time=True)
        self.cond = self._plan.cond
        self.tail = tail_factory(self.imgs[n_iter]) if tail_factory is not None else None
        self.has_tail = self.tail is not None
        self.launches = n_iter * (self._plan.num_launches() + 1 + (1 if inpaint else 0)) + (self.tail.num_launches if self.tail else 0) \
            + len(self._plan.cond_ops)
        # warm-up run outside capture (lazy one-time initialisations, kernel attribute sets), then capture
        self._plan.run_cond()
        self._body(first_only=True)
        if self.tail is not None:
            self.tail.run()
        torch.cuda.synchronize()
        if use_graph:
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._body()
                if self.tail is not None:
                    self.tail.run()

    @property
    def plan(self):
        """The operator-level plan of this loop's U-Net shape (bench.py times its launches one by one); built on demand when the
        loop itself runs through the library's graph."""
        if self._plan is None:
            B = self.B
            self._plan = self.model.plan(self.N, self.shape[2], self.shape[3], x_batch_mod=B if self.cfg_on else 0, uniform_time=True)
        return self._plan

    def _body(self, first_only: bool = False):
        pl, B = self._plan, self.B
        for k in range(1 if first_only else self.n_iter):
            pl.x.copy_(self.imgs[k])
            pl.t[:1].copy_(self.ttab[k:k + 1])
            pl.run()
            eps_u = pl.eps[:B] if self.cfg_on else None
            eps_c = pl.eps[B:] if self.cfg_on else pl.eps
            ops.ddim_step(eps_u, eps_c, self.imgs[k], self.noise[k] if self.noise is not None else None, self.coef[k], self.imgs[k + 1])
            if self.inpaint:
                ops.mask_blend(self.guide, self.init_noise, self.masks[k], self.blend_coef[k], self.imgs[k + 1])

    def launch(self):
        if self.sgraph is not None:
            self.sgraph.run()
            return
        self._plan.run_cond()        # condition projections are step-invariant: once per call, outside the graph
        if self.graph is not None:
            self.graph.replay()
        else:
            self._body()
            if self.tail is not None:
                self.tail.run()
