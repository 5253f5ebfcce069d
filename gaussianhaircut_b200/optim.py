"""Fused multi-group Adam over the Gaussian parameters ("next" row 2 of SURVEY.md 8f).

Same arithmetic and hyper-parameter surface as the reference's `torch.optim.Adam(l, lr=0.0,
eps=1e-15)` with per-group learning rates (src/scene/gaussian_model.py:431-448); the reference's
NaN guard (src/train_gaussians.py:174-181, seven blocking `.isnan().any()` syncs per step) becomes a
device-side flag.  One kernel launch per step for all groups, through `gh_adam_step` of the C ABI.

State handling follows torch.optim so that the reference's densification code works on it unchanged
(src/scene/gaussian_model.py:581-680: `optimizer.state.get(param)`, `del optimizer.state[param]`,
`group["params"][0] = nn.Parameter(...)`, `optimizer.state[new_param] = stored_state`):
`state` is a dict keyed by the parameter TENSOR (so a parameter that was replaced can never be paired
with another tensor's moments through a recycled `id()`), entries hold `exp_avg` / `exp_avg_sq` (and
a `step` tensor for torch compatibility), missing entries are created lazily in `step()`, and every
tensor handed to the kernel is validated against the parameter's element count.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Iterable, List, Optional, Sequence

import torch

from . import _capi

MAX_GROUPS = 8   # GH_ADAM_MAX_GROUPS


class FusedAdam:
    """`param_groups` like torch (dicts with 'params', 'lr', optional 'name'), `.state`, `.step()`,
    `.zero_grad()`, `.state_dict()` / `.load_state_dict()`.  All tensors float32 CUDA contiguous."""

    def __init__(self, param_groups: Iterable[Dict], betas=(0.9, 0.999), eps: float = 1e-15, nan_guard: bool = True,
                 lr: float = 0.0):
        self.param_groups: List[Dict] = []
        for g in param_groups:
            g = dict(g)
            g["params"] = list(g["params"])
            g.setdefault("lr", lr)
            self.param_groups.append(g)
        self.defaults = {"lr": lr, "betas": betas, "eps": eps}
        self.betas, self.eps = betas, eps
        self.state: Dict[torch.Tensor, Dict[str, torch.Tensor]] = {}
        flat = self._params()
        if not flat:
            raise ValueError("FusedAdam needs at least one parameter")
        if len(flat) > MAX_GROUPS:
            raise ValueError("at most 8 parameter tensors (GH_ADAM_MAX_GROUPS)")
        for p in flat:
            self._check_param(p)
        dev = flat[0].device
        self.nan_flag = torch.zeros(1, dtype=torch.int32, device=dev) if nan_guard else None
        self.step_state = torch.zeros(2, dtype=torch.int32, device=dev)   # [steps taken, scratch], device resident
        self._keep = None

    # ------------------------------------------------------------------------------------------ helpers
    def _params(self) -> List[torch.Tensor]:
        return [p for g in self.param_groups for p in g["params"]]

    @staticmethod
    def _check_param(p: torch.Tensor) -> None:
        if p.dtype != torch.float32 or not p.is_cuda or not p.is_contiguous():
            raise ValueError("FusedAdam needs contiguous float32 CUDA parameters")

    def _state_for(self, p: torch.Tensor) -> Dict[str, torch.Tensor]:
        st = self.state.get(p)
        if st is None or "exp_avg" not in st:       # lazily, like torch (also after `del optimizer.state[p]`)
            st = {"step": torch.zeros((), dtype=torch.float32, device=p.device),
                  "exp_avg": torch.zeros_like(p, memory_format=torch.contiguous_format),
                  "exp_avg_sq": torch.zeros_like(p, memory_format=torch.contiguous_format)}
            self.state[p] = st
        return st

    @property
    def step_count(self) -> int:
        """Steps taken (host sync: the count lives on the device so that skipped steps are not counted)."""
        return int(self.step_state[0].item())

    def zero_grad(self, set_to_none: bool = True):
        for g in self.param_groups:
            for p in g["params"]:
                if set_to_none:
                    p.grad = None
                elif p.grad is not None:
                    p.grad.zero_()

    # ------------------------------------------------------------------------------------------ step
    def step(self, grads: Optional[Sequence[Optional[torch.Tensor]]] = None,
             skip_flags: Sequence[torch.Tensor] = (), nan_flag_in: Optional[torch.Tensor] = None):
        """Update every parameter that has a gradient (`grads` overrides `.grad`, in parameter order).

        `skip_flags`: device int32/uint32 tensors (1 element each; at most one is passed to the kernel, the
        others are OR-ed on the device first): the step is skipped when one is non-zero, e.g.
        `PeerAllReduce.error_flag`.  `nan_flag_in`: a NaN verdict already computed by the producer of the
        gradients (`PeerAllReduce.nan_flag`): replaces this optimizer's own scan of the gradients."""
        lib = _capi.load()
        ps, gs, ms, vs, ns, lrs = [], [], [], [], [], []
        it = iter(grads) if grads is not None else None
        if len(self._params()) > MAX_GROUPS:
            raise ValueError("at most 8 parameter tensors (GH_ADAM_MAX_GROUPS)")
        for g in self.param_groups:
            for p in g["params"]:
                gr = next(it) if it is not None else p.grad
                if gr is None:
                    continue
                self._check_param(p)
                st = self._state_for(p)
                gr = gr.contiguous()
                n = p.numel()
                for name, t in (("gradient", gr), ("exp_avg", st["exp_avg"]), ("exp_avg_sq", st["exp_avg_sq"])):
                    if t.numel() != n or t.dtype != torch.float32 or t.device != p.device or not t.is_contiguous():
                        raise RuntimeError(f"FusedAdam: {name} of parameter group '{g.get('name', '?')}' has {t.numel()} "
                                           f"elements ({t.dtype}, {t.device}), the parameter has {n}: optimizer state "
                                           "and parameter went out of sync (densification must replace both)")
                if n == 0:
                    continue      # nothing to update, and a tensor without elements has no storage to hand to the kernel
                ps.append(p); gs.append(gr); ms.append(st["exp_avg"]); vs.append(st["exp_avg_sq"])
                ns.append(n); lrs.append(float(g["lr"]))
        if not ps:
            return
        n = len(ps)
        arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])   # noqa: E731
        dev = ps[0].device
        skip = None
        flags = [f for f in skip_flags if f is not None]
        if nan_flag_in is not None:
            flags.append(nan_flag_in)
        if len(flags) == 1:
            skip = flags[0]
        elif len(flags) > 1:
            skip = torch.stack([f.reshape(-1)[0].to(torch.int32) for f in flags]).amax().reshape(1).contiguous()
        own_nan = self.nan_flag if nan_flag_in is None else None
        with torch.cuda.device(dev):
            _capi.check(lib.gh_adam_step(
                n, arr(ps), arr(gs), arr(ms), arr(vs), (C.c_ulonglong * n)(*ns), (C.c_float * n)(*lrs),
                float(self.betas[0]), float(self.betas[1]), float(self.eps), 0,
                C.c_void_p(self.step_state.data_ptr()),
                C.c_void_p(own_nan.data_ptr()) if own_nan is not None else None,
                C.c_void_p(skip.data_ptr()) if skip is not None else None,
                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        if nan_flag_in is not None:
            nan_flag_in.zero_()       # consumed: ready for the next iteration's backward (stream-ordered after the update)
        self._keep = (ps, gs, skip)   # keep the tensors alive until the kernels have run

    # ------------------------------------------------------------------------------------------ (de)serialisation
    def state_dict(self) -> Dict:
        """torch.optim-shaped: {'state': {index: {...}}, 'param_groups': [{..., 'params': [indices]}]} plus the
        device-resident step count."""
        index = {}
        groups = []
        for g in self.param_groups:
            ids = []
            for p in g["params"]:
                index.setdefault(p, len(index))
                ids.append(index[p])
            groups.append({**{k: v for k, v in g.items() if k != "params"}, "params": ids})
        state = {index[p]: {k: v.clone() for k, v in st.items()} for p, st in self.state.items() if p in index}
        return {"state": state, "param_groups": groups, "steps_taken": self.step_count}

    def load_state_dict(self, sd: Dict) -> None:
        params = self._params()
        saved_groups = sd["param_groups"]
        if len(saved_groups) != len(self.param_groups) or \
                any(len(a["params"]) != len(b["params"]) for a, b in zip(saved_groups, self.param_groups)):
            raise ValueError("loaded state dict has a different number of parameter groups / parameters")
        for g, sg in zip(self.param_groups, saved_groups):
            for k, v in sg.items():
                if k != "params":
                    g[k] = v
        order = [i for sg in saved_groups for i in sg["params"]]
        self.state = {}
        for p, i in zip(params, order):
            st = sd["state"].get(i)
            if st is None:
                continue
            for k in ("exp_avg", "exp_avg_sq"):
                if st[k].numel() != p.numel():
                    raise ValueError(f"loaded {k} has {st[k].numel()} elements, the parameter has {p.numel()}")
            self.state[p] = {k: (v.to(device=p.device, dtype=torch.float32).contiguous().clone() if isinstance(v, torch.Tensor) else v)
                             for k, v in st.items()}
        self.step_state.zero_()
        self.step_state[0] = int(sd.get("steps_taken", 0))
