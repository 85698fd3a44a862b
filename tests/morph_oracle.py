"""Float64 restatements of the timbre-morph pieces (TEST INFRASTRUCTURE ONLY): the linear rows of generate_linear_noise with both
endpoints (model/DiffSynthSampler.py:170-174), the spherical rows with their linear fallback, and DDIM inversion for any callable
model on the oracle's Schedule (oracle/ds_oracle.py), whose coefficients come from alphas_cumprod_next (sampler.py:92)."""
from __future__ import annotations

from typing import List, Optional

import numpy as np
import torch

from oracle import ds_oracle as O

SLERP_MIN_SIN = 1e-6          # below it (identical or antipodal endpoints) a sequence takes the linear rows


def _weights(frames: int) -> np.ndarray:
    return np.arange(frames, dtype=np.float64) / (frames - 1)


def linear_rows(e0, e1, frames: int) -> np.ndarray:
    """[P, ...] endpoints -> [P * frames, ...] rows a e1 + (1 - a) e0, a = k / (frames - 1), sequence-major, in float64."""
    e0, e1 = np.asarray(e0, np.float64), np.asarray(e1, np.float64)
    a = _weights(frames).reshape((1, frames) + (1,) * (e0.ndim - 1))
    rows = a * e1[:, None] + (1.0 - a) * e0[:, None]
    return rows.reshape((-1,) + e0.shape[1:])


def slerp_theta(e0: np.ndarray, e1: np.ndarray) -> float:
    """Angle between two endpoints, or None when slerp is undefined (a zero endpoint) or sin theta < SLERP_MIN_SIN."""
    x, y = np.asarray(e0, np.float64).ravel(), np.asarray(e1, np.float64).ravel()
    n0, n1 = float(x @ x), float(y @ y)
    if n0 <= 0.0 or n1 <= 0.0:
        return None
    th = float(np.arccos(np.clip((x @ y) / (np.sqrt(n0) * np.sqrt(n1)), -1.0, 1.0)))
    return th if np.sin(th) >= SLERP_MIN_SIN else None


def slerp_rows(e0, e1, frames: int) -> np.ndarray:
    """[P, ...] endpoints -> [P * frames, ...] rows w0 e0 + w1 e1, w0 = sin((1 - a) theta) / sin theta, w1 = sin(a theta) / sin theta,
    per sequence; a sequence without a usable angle takes linear_rows."""
    e0, e1 = np.asarray(e0, np.float64), np.asarray(e1, np.float64)
    a = _weights(frames)
    out = []
    for p in range(e0.shape[0]):
        th = slerp_theta(e0[p], e1[p])
        if th is None:
            out.append(linear_rows(e0[p:p + 1], e1[p:p + 1], frames))
            continue
        w0, w1 = np.sin((1.0 - a) * th) / np.sin(th), np.sin(a * th) / np.sin(th)
        sh = (frames,) + (1,) * (e0.ndim - 1)
        out.append(w0.reshape(sh) * e0[p][None] + w1.reshape(sh) * e1[p][None])
    return np.concatenate(out)


def alphas_cumprod_next(sch: O.Schedule) -> np.ndarray:
    return np.append(sch.alphas_cumprod[1:], 0.0)


def invert_coefficients(sch: O.Schedule, cfg_scale: float) -> np.ndarray:
    """[steps, 8] ds_ddim_step coefficients of the inversion steps, ascending: [sqrt(1-a_t), sqrt(a_t), sqrt(a_next), sqrt(1-a_next), 0,
    cfg, 0, 0], each table value rounded to fp32 and the square roots taken in fp32 (as ddim_coefficients evaluates its own)."""
    nxt = alphas_cumprod_next(sch)
    rows = []
    for t in range(sch.num_timesteps):
        at, an = torch.tensor(sch.alphas_cumprod[t]).float(), torch.tensor(nxt[t]).float()
        rows.append([float(torch.sqrt(1.0 - at)), float(torch.sqrt(at)), float(torch.sqrt(an)), float(torch.sqrt(1.0 - an)), 0.0,
                     float(cfg_scale), 0.0, 0.0])
    return np.asarray(rows, dtype=np.float64)


def ddim_invert(model, sch: O.Schedule, x0: torch.Tensor, cond: torch.Tensor, uncond: Optional[torch.Tensor], cfg_scale: float
                ) -> List[torch.Tensor]:
    """DDIM inversion x_0 -> noise over the ascending respaced steps: eps by ``model(x, t_mapped, cond)`` with classifier-free
    guidance as sample_loop forms it, then x_next = sqrt(a_next) x0_pred + sqrt(1 - a_next) eps.  Returns the latents (len steps+1)."""
    B = x0.shape[0]
    co = invert_coefficients(sch, cfg_scale)
    imgs = [x0]
    img = x0
    for t in range(sch.num_timesteps):
        t_mapped = torch.full((B,), sch.timestep_map[t], dtype=torch.long)
        if cfg_scale == 1.0:
            eps_u, eps_c = None, model(img, t_mapped, cond)
        else:
            u = uncond.unsqueeze(0).repeat(*([B] + [1] * uncond.dim()))
            out = model(torch.cat([img, img]), torch.cat([t_mapped, t_mapped]), torch.cat([u, cond]))
            eps_u, eps_c = out[:B], out[B:]
        c = dict(sqrt_one_minus_at=co[t, 0], sqrt_at=co[t, 1], sqrt_ap=co[t, 2], dir_coef=co[t, 3], sigma=0.0)
        img = O.ddim_update(img, eps_u, eps_c, cfg_scale, c, torch.zeros_like(img))
        imgs.append(img)
    return imgs
