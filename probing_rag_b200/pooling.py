"""On-device pooling of the probed layers' hidden states (SURVEY 8f-3).

The reference registers one forward hook per probed layer (/root/reference/exp_rag.py:317-329) that
appends `activations.detach().cpu()` to `cache[layer]` on every forward call -- six device->host
syncs per decode step -- and later concatenates `cache[layer][1:]` (the prefill entry is dropped),
copies it back to the device and sums over the token axis (exp_rag.py:385-386).  `HiddenStatePooler`
keeps the same hook signature `hook_fn(activations, hook, layer)` but adds the activations straight
into the prober input matrix X[n_rows, n_probers, d_model] on the device (pr_pool_accumulate), so
`pooler.X` feeds `ProberGate` with no copy at all.

    pooler = HiddenStatePooler(n_rows=B, layers=[f'blocks.{l}.hook_resid_post' for l in range(6, 17, 2)])
    for name in pooler.layers:
        model.add_hook(name, functools.partial(pooler.hook_fn, layer=name))     # exp_rag.py:323-329
    pooler.reset()                  # where the reference writes `cache = {}` (exp_rag.py:397, 423)
    model.generate(...)
    out = gate(pooler.X)            # exp_rag.py:406-415
"""
from __future__ import annotations

import torch

from . import _lib

_DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


class HiddenStatePooler:
    def __init__(self, n_rows: int, layers, d_model: int = 2048, device="cuda"):
        dev = torch.device(device)
        if dev.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("HiddenStatePooler needs a CUDA device: the pooling path has no CPU fallback")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.layers = list(layers)
        if not 1 <= len(self.layers) <= _lib.PR_PROBER_MAX:
            raise ValueError(f"between 1 and {_lib.PR_PROBER_MAX} probed layers")
        if d_model % 4:
            raise ValueError("d_model must be a multiple of 4")
        self._slot = {name: i for i, name in enumerate(self.layers)}
        self.n_rows, self.d_model, self.device = int(n_rows), int(d_model), dev
        self.X = torch.zeros((self.n_rows, len(self.layers), self.d_model), dtype=torch.float32, device=dev)
        self._calls = [0] * len(self.layers)

    def reset(self) -> None:
        """Start of a generation: the reference's `cache = {}` (exp_rag.py:397, 423)."""
        self.X.zero_()
        self._calls = [0] * len(self.layers)

    def calls(self, layer) -> int:
        return self._calls[self._slot[layer]]

    def add(self, layer, activations: torch.Tensor, row_map: torch.Tensor | None = None) -> None:
        """Add sum_t activations[r, t, :] to X[row, slot(layer), :] (row = row_map[r] or r).  A negative row_map
        entry skips the row; the others must be distinct and below n_rows, else ValueError (two activation rows
        into one accumulator row would race in the kernel).  The check reads row_map on the host: a row_map on
        the device costs a synchronisation."""
        slot = self._slot[layer]
        a = activations.detach()
        if a.dim() == 2:
            a = a.unsqueeze(1)
        if a.dim() != 3 or a.shape[2] != self.d_model:
            raise ValueError(f"activations must be [rows, tokens, {self.d_model}], got {tuple(activations.shape)}")
        if a.device != self.device:
            raise ValueError("activations must live on the pooler's device")
        if a.dtype not in _DTYPES:
            a = a.float()
        if a.stride(2) != 1 or a.stride(0) % 4 or a.stride(1) % 4 or a.data_ptr() % (4 * a.element_size()):
            a = a.contiguous()
        rm = None
        if row_map is not None:
            rm = row_map.to("cpu", torch.int64).flatten()
            if rm.numel() != a.shape[0]:
                raise ValueError("row_map needs one entry per activation row")
            live = rm[rm >= 0]
            if live.numel() and (int(live.max()) >= self.n_rows or live.unique().numel() != live.numel()):
                raise ValueError(f"row_map: non-negative entries must be distinct and below {self.n_rows}")
            rm = rm.to(self.device, torch.int32)
        elif a.shape[0] > self.n_rows:
            raise ValueError(f"{a.shape[0]} activation rows for {self.n_rows} accumulator rows")
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().pr_pool_accumulate(
                self.X.data_ptr(), self.n_rows, len(self.layers), slot, self.d_model, a.data_ptr(), _DTYPES[a.dtype],
                a.shape[0], a.shape[1], a.stride(0), a.stride(1), rm.data_ptr() if rm is not None else None,
                torch.cuda.current_stream(self.device).cuda_stream))

    def hook_fn(self, activations, hook=None, layer=None, row_map=None):
        """Drop-in for the reference's `hook_fn(activations, hook, layer)` (exp_rag.py:317-321): the first
        call after reset() is the prefill and is dropped like `cache[layer][0]`; every later call is summed."""
        slot = self._slot[layer]
        if self._calls[slot] > 0:
            self.add(layer, activations, row_map)
        self._calls[slot] += 1
        return activations
