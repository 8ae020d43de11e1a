"""Float64 restatement of the prober path and the pooler's exact promise -- TEST INFRASTRUCTURE ONLY.

  prober_logits_f64   OracleImprovedProbe (oracle/prober_oracle.py) evaluated in float64 from the same state_dicts:
                      LN_in -> fc1 -> SiLU -> LN1 -> fc2 -> SiLU -> LN2 -> fc3, prober p applied to x[:, p]
  gate_f64            oracle/prober_oracle.gate on float64 logits: probsum = sum over probers >= ablation of
                      softmax, retrieve = NOT (probsum0 + theta < probsum1); NaN rows retrieve (a failed comparison)
  pool_call           what pr_pool_accumulate promises for one call, bit for bit: per activation row the tokens summed in
                      fp32 in token order starting from 0, that sum then added once to the accumulator row
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

LN_EPS = 1e-5      # nn.LayerNorm's default, which ImprovedProbe uses


def state_f64(sd: dict) -> dict:
    return {k: v.detach().to("cpu", torch.float64) for k, v in sd.items()}


def probe_logits_f64(sd64: dict, x: torch.Tensor) -> torch.Tensor:
    """One prober: x[B, d] (any float dtype, widened exactly) -> logits f64 [B, 2]."""
    h = x.to(torch.float64)
    h = F.layer_norm(h, h.shape[-1:], sd64["layer_norm_input.weight"], sd64["layer_norm_input.bias"], LN_EPS)
    h = F.silu(F.linear(h, sd64["fc1.weight"], sd64["fc1.bias"]))
    h = F.layer_norm(h, h.shape[-1:], sd64["layer_norm1.weight"], sd64["layer_norm1.bias"], LN_EPS)
    h = F.silu(F.linear(h, sd64["fc2.weight"], sd64["fc2.bias"]))
    h = F.layer_norm(h, h.shape[-1:], sd64["layer_norm2.weight"], sd64["layer_norm2.bias"], LN_EPS)
    return F.linear(h, sd64["fc3.weight"], sd64["fc3.bias"])


@torch.no_grad()
def prober_logits_f64(sds64, x: torch.Tensor) -> torch.Tensor:
    """x[B, P, d] -> logits f64 [B, P, 2]; sds64 from state_f64."""
    return torch.stack([probe_logits_f64(sd, x[:, i]) for i, sd in enumerate(sds64)], dim=1)


def gate_f64(logits: torch.Tensor, theta: float = 0.0, ablation: int = 0):
    """(probs f64 [B, P, 2], probsum f64 [B, 2], retrieve bool [B])."""
    probs = torch.softmax(logits.to(torch.float64), dim=-1)
    psum = probs[:, ablation:].sum(dim=1)
    retrieve = ~(psum[:, 0] + theta < psum[:, 1])
    return probs, psum, retrieve


def pool_call(acc: np.ndarray, slot: int, act: np.ndarray, row_map=None) -> None:
    """acc f32 [n_acc_rows, P, d] += token sums of act [R, T, d] (f32 / bf16-as-f32 / f16), in place.
    row_map: None (identity) or int [R]; negative entries skip the row."""
    assert acc.dtype == np.float32
    a = np.asarray(act, dtype=np.float32)
    s = np.zeros((a.shape[0], a.shape[2]), dtype=np.float32)
    for t in range(a.shape[1]):
        s += a[:, t]                     # one rounded f32 add per token, in token order
    dst = np.arange(a.shape[0]) if row_map is None else np.asarray(row_map, dtype=np.int64)
    for r, d in enumerate(dst.tolist()):
        if d >= 0:
            acc[d, slot] += s[r]
