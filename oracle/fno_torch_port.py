"""TEST INFRASTRUCTURE -- CPU PyTorch restatement ("port") of the reference FNO hot path.

Never imported by the product package; only `tests/`, `__graft_entry__.smoke()` and the
`cpu_baseline` / `--impl reference` legs of `bench.py` may use it (the reference is not part of this
repository, so this port is what those legs time).

It issues the *same library calls* the reference issues on CPU, so its speed is the reference's:
torch.fft.rfft2 -> zero-filled cfloat spectrum -> two einsum("bixy,ioxy->boxy") corner products ->
torch.fft.irfft2 (reference src/models/fno/fno2d.py:59-82), F.conv2d 1x1 + exact-erf GELU
(fno2d.py:106-112, 147), channel assembly + per-call coordinate grid (fno2d.py:195-217, 244-255),
fc1/GELU/fc2/mask (fno2d.py:228-233), MseLoss (src/models/loss.py:22-37), feed-back rollout
(fno2d.py:257-295).  Parameters are a plain dict with the reference's state_dict keys.

`round_fn` (optional) is applied to every hidden activation the CUDA path stores between kernels
(lift output and each block output).  With `round_fn = lambda t: t.bfloat16().float()` this is the
"bf16-boundary oracle" of SURVEY.md 7.

Pinning: validated bit-for-bit against the imported reference module by `oracle/make_golden.py`
(run in the build container) and against `tests/golden/*.npz` by `tests/test_oracle.py`.
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np
import torch
import torch.nn.functional as F


def params_from_numpy(sd: dict, requires_grad: bool = False) -> dict:
    out = {}
    for k, v in sd.items():
        t = torch.from_numpy(np.ascontiguousarray(v)).clone()
        out[k] = t.requires_grad_(requires_grad)
    return out


def depth_of(p: dict) -> int:
    return 1 + max(int(k.split(".")[1]) for k in p if k.startswith("blocks."))


def spectral_conv(x: torch.Tensor, w1: torch.Tensor, w2: torch.Tensor) -> torch.Tensor:
    m1, m2 = w1.shape[-2:]
    spec = torch.fft.rfft2(x)
    out = torch.zeros(x.shape[0], w1.shape[1], x.shape[-2], x.shape[-1] // 2 + 1,
                      dtype=torch.cfloat, device=x.device)
    out[:, :, :m1, :m2] = torch.einsum("bixy,ioxy->boxy", spec[:, :, :m1, :m2], w1)
    out[:, :, -m1:, :m2] = torch.einsum("bixy,ioxy->boxy", spec[:, :, -m1:, :m2], w2)
    return torch.fft.irfft2(out, s=(x.shape[-2], x.shape[-1]))


def coords(b: int, h: int, w: int) -> torch.Tensor:
    gx = torch.tensor(np.linspace(0, 1, h), dtype=torch.float).reshape(1, 1, h, 1).repeat(b, 1, 1, w)
    gy = torch.tensor(np.linspace(0, 1, w), dtype=torch.float).reshape(1, 1, 1, w).repeat(b, 1, h, 1)
    return torch.cat([gx, gy], dim=1)


def forward(p: dict, inputs: torch.Tensor, case_params: torch.Tensor,
            mask: Optional[torch.Tensor] = None, label: Optional[torch.Tensor] = None,
            normalize: bool = True, round_fn: Optional[Callable] = None,
            return_acts: bool = False) -> dict:
    b, _, h, w = inputs.shape
    if mask is None:
        mask = torch.ones(b, 1, h, w)
    elif mask.dim() == 3:
        mask = mask.unsqueeze(1)
    rf = round_fn if round_fn is not None else (lambda t: t)
    feats = torch.cat([inputs, mask, coords(b, h, w),
                       case_params[:, :, None, None].repeat(1, 1, h, w)], dim=1)
    a = rf(F.conv2d(feats, p["fc0.weight"], p["fc0.bias"]))
    acts = [a]
    for l in range(depth_of(p)):
        s = spectral_conv(a, p[f"blocks.{l}.conv0.weights1"], p[f"blocks.{l}.conv0.weights2"])
        a = rf(F.gelu(s + F.conv2d(a, p[f"blocks.{l}.w0.weight"], p[f"blocks.{l}.w0.bias"])))
        acts.append(a)
    hid = F.gelu(F.conv2d(a, p["fc1.weight"], p["fc1.bias"]))
    preds = F.conv2d(hid, p["fc2.weight"], p["fc2.bias"]) * mask
    out = {"preds": preds}
    if label is not None:
        out["loss"] = mse_loss(preds, label * mask, normalize)
    if return_acts:
        out["acts"] = acts
    return out


def mse_loss(preds: torch.Tensor, labels: torch.Tensor, normalize: bool = True) -> dict:
    mse = F.mse_loss(preds, labels)
    res = {"mse": mse, "rmse": torch.sqrt(mse), "mae": F.l1_loss(preds, labels)}
    if normalize:
        res["nmse"] = mse / torch.square(labels).mean()
    return res


def rollout(p: dict, inputs: torch.Tensor, case_params: torch.Tensor, mask: torch.Tensor,
            steps: int, round_fn: Optional[Callable] = None) -> list:
    if inputs.dim() == 3:
        inputs, case_params, mask = inputs[None], case_params[None], mask[None]
    cur, outs = inputs, []
    for _ in range(steps):
        cur = forward(p, cur, case_params, mask, round_fn=round_fn)["preds"]
        outs.append(cur)
    return outs


def train_step(p: dict, opt: torch.optim.Optimizer, batch: dict) -> float:
    """fwd -> loss["nmse"].backward() -> Adam.step -> zero_grad -> .item()
    (reference src/train_auto.py:233-260)."""
    out = forward(p, batch["inputs"], batch["case_params"], batch["mask"], batch["label"])
    out["loss"]["nmse"].backward()
    opt.step()
    opt.zero_grad()
    return out["loss"]["nmse"].item()


def bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.bfloat16().float()


def bf16_round_ste(t: torch.Tensor) -> torch.Tensor:
    """bf16 rounding with a straight-through gradient: what the CUDA training path does when activations are stored
    as bf16 (the next layer consumes the rounded value, the backward pass differentiates the unrounded expression)."""
    return t + (t.bfloat16().float() - t).detach()
