"""Fused Adam with ``torch.optim.Adam``'s constructor, semantics and ``state_dict`` layout
(ref:ssp_vit2spn_tiny.py:173,216; fine-tune: ref:octmnist_ft_vit2spn.py:192 with L2 weight decay).

Parameters that are views of a vit2spn flat buffer (every parameter of ``DualStreamNetwork`` /
``ViTModel``) are updated by ONE flat-range kernel launch per optimizer step (v2s_adam_step*);
any other parameter is updated by the same kernel, one range per tensor.  Tensors whose ``.grad``
is None are skipped, exactly as torch does (SURVEY D6: final LayerNorm + pooler).

``torch.amp.GradScaler`` (the reference's fp16 recipe, ref:175,216-217) is supported the way torch's own fused Adam
supports it: ``_step_supports_amp_scaling`` makes ``scaler.step(optimizer)`` hand over its scale and found-inf tensors,
and the kernel unscales / skips on the device (v2s_adam_step_amp) — no host synchronisation, step counts kept on the
device.  ``capturable=True`` selects that device-resident path without a scaler (CUDA-graph capture of the step).
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import Range, lib, check, stream_ptr
from .modules import _STORES


class FusedAdam(torch.optim.Optimizer):
    _step_supports_amp_scaling = True       # torch.amp.GradScaler: pass grad_scale / found_inf tensors, do not unscale

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, capturable=False):
        if lr < 0 or eps < 0 or not (0 <= betas[0] < 1) or not (0 <= betas[1] < 1) or weight_decay < 0:
            raise ValueError("invalid Adam hyper-parameter")
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=False, maximize=False,
                        foreach=None, capturable=bool(capturable), differentiable=False, fused=None,
                        decoupled_weight_decay=False)
        super().__init__(params, defaults)
        self._flat_state = {}      # id(store) -> [store, exp_avg_flat, exp_avg_sq_flat, host step | None, device state8 | None]
        self._dev_steps = {}       # id(param) -> device state8 of a parameter outside the flat stores
        self._psets = {}
        self._member = {}          # (group, store, #params) -> does the store hold parameters of the group
        self._all_ids = None
        self.grad_multiplier = 1.0  # multiplies every gradient inside the kernel (1/world_size of the data-parallel mean)

    # -- state bookkeeping ---------------------------------------------------------------------------------------
    def _state_for(self, p, m_view=None, v_view=None):
        st = self.state[p]
        if len(st) == 0:
            st["step"] = torch.tensor(0.0, dtype=torch.float32)
            st["exp_avg"] = m_view if m_view is not None else torch.zeros_like(p, memory_format=torch.preserve_format)
            st["exp_avg_sq"] = v_view if v_view is not None else torch.zeros_like(p, memory_format=torch.preserve_format)
        return st

    @staticmethod
    def _active(store):
        return [(p, o) for p, o in zip(store.params, store.offsets) if o < store.active_numel]

    def _store_plan(self, store, pset):
        """[store, m_flat, v_flat, step, state8] if the whole active range of the store can be updated as ONE flat
        range: every tensor in it is trainable, belongs to this parameter group and shares one step count; else None
        (per-tensor path — frozen tensors inside the range must not be touched, e.g. by weight decay)."""
        active = self._active(store)
        if not active or any((not p.requires_grad) or id(p) not in pset for p, _ in active):
            return None
        if store.flat is None or not store.flat.is_cuda or store.active_numel % 4:
            return None
        key = id(store)
        ent = self._flat_state.get(key)
        if ent is None or ent[1].device != store.flat.device:
            m = torch.zeros(store.numel, dtype=torch.float32, device=store.flat.device)
            v = torch.zeros(store.numel, dtype=torch.float32, device=store.flat.device)
            ent = [store, m, v, None, None]
            self._flat_state[key] = ent
        _, m, v, step, state8 = ent
        if step is None and state8 is None:
            steps = set()
            for p, o in active:
                mv, vv = m[o:o + p.numel()].view(p.shape), v[o:o + p.numel()].view(p.shape)
                st = self._state_for(p, mv, vv)
                if st["exp_avg"].data_ptr() != mv.data_ptr():      # e.g. after load_state_dict
                    mv.copy_(st["exp_avg"]); st["exp_avg"] = mv
                if st["exp_avg_sq"].data_ptr() != vv.data_ptr():
                    vv.copy_(st["exp_avg_sq"]); st["exp_avg_sq"] = vv
                steps.add(float(st["step"]))
            if len(steps) != 1:
                return None                                          # inconsistent history: per-tensor path
            ent[3] = int(steps.pop())
        return ent

    def _release_store(self, store):
        """The store leaves the flat path (a tensor was frozen, .grad detached, ...): hand its step count back to the
        per-parameter state so that the per-tensor path continues the same history."""
        ent = self._flat_state.get(id(store))
        if ent is None:
            return
        self._sync_entry(ent)
        ent[3], ent[4] = None, None

    def _sync_entry(self, ent):
        store, _, _, step, state8 = ent
        if state8 is not None:
            step = int(round(float(state8[0].item())))       # device-resident count (amp / capturable path): one sync
        if step is None:
            return
        for p, _ in self._active(store):
            if p in self.state:
                self.state[p]["step"] = torch.tensor(float(step), dtype=torch.float32)

    def _all_param_ids(self):
        n = sum(len(g["params"]) for g in self.param_groups)
        if self._all_ids is None or len(self._all_ids) != n:
            self._all_ids = {id(p) for g in self.param_groups for p in g["params"]}
        return self._all_ids

    def _sync_steps(self):
        """Write the step counters back into the per-parameter state (state_dict layout of torch)."""
        for ent in self._flat_state.values():
            self._sync_entry(ent)
        for group in self.param_groups:
            for p in group["params"]:
                s8 = self._dev_steps.get(id(p))
                if s8 is not None and p in self.state:
                    self.state[p]["step"] = torch.tensor(float(round(float(s8[0].item()))), dtype=torch.float32)

    def state_dict(self):
        self._sync_steps()
        return super().state_dict()

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        for ent in self._flat_state.values():
            ent[3], ent[4] = None, None             # re-derive the flat views and step counters from the loaded state
        self._dev_steps.clear()

    def zero_grad(self, set_to_none: bool = True):
        """Flat-buffer fast path: ONE memset per store, ``.grad`` views stay attached (they read as zeros
        instead of None).  Parameters outside vit2spn stores follow torch's semantics."""
        handled = set()
        mine = self._all_param_ids()
        for store in list(_STORES):
            # only stores whose trainable parameters all belong to this optimizer
            if store.flat_grad is None or not all(id(p) in mine for p in store.params if p.requires_grad):
                continue
            if store.zero_grads_fast():
                handled.update(id(p) for p in store.params)
        for group in self.param_groups:
            for p in group["params"]:
                if id(p) in handled or p.grad is None:
                    continue
                if set_to_none:
                    p.grad = None
                else:
                    p.grad.detach_(); p.grad.zero_()

    # -- the step ------------------------------------------------------------------------------------------------
    @staticmethod
    def _scalar_ptr(t, dev, what):
        if t is None:
            return None, None
        if not isinstance(t, torch.Tensor) or t.numel() != 1:
            raise RuntimeError(f"FusedAdam: {what} must be a one-element tensor")
        t = t.detach().to(device=dev, dtype=torch.float32).reshape(1)
        return t, t.data_ptr()

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        # set by torch.amp.GradScaler.step() for optimizers with _step_supports_amp_scaling (deleted again afterwards)
        amp_scale = getattr(self, "grad_scale", None)
        amp_inf = getattr(self, "found_inf", None)
        for group in self.param_groups:
            lr, (b1, b2), eps, wd = group["lr"], group["betas"], group["eps"], group["weight_decay"]
            if group.get("amsgrad") or group.get("maximize"):
                raise NotImplementedError("FusedAdam: amsgrad/maximize are not used by the reference")
            on_device = bool(group.get("capturable")) or amp_scale is not None or amp_inf is not None
            params = group["params"]
            pset = self._psets.get(id(group))
            if pset is None or len(pset) != len(params):
                pset = {id(p) for p in params}
                self._psets[id(group)] = pset
            host_launches = {}     # (step, lp_fmt) -> [Range]
            dev_launches = {}      # (id(state8), lp_fmt) -> (state8, [Range]); one shared state8 per step count
            fresh8 = {}            # (device, step) -> state8 created in this call
            covered, keep = set(), []
            dev_of = {}            # Range.params address -> device (host-path launches run with that device current)

            def new_state8(dev, step):
                s8 = fresh8.get((dev, step))
                if s8 is None:
                    s8 = torch.zeros(8, dtype=torch.float32, device=dev)
                    s8[0] = float(step)
                    fresh8[(dev, step)] = s8
                return s8

            for store in list(_STORES):
                mkey = (id(group), id(store), len(params))
                member = self._member.get(mkey)
                if member is None:
                    member = self._member[mkey] = any(id(p) in pset for p in store.params)
                if not member:
                    continue
                ent = None
                if store.flat_grad is not None and store.grads_attached():
                    ent = self._store_plan(store, pset)
                if ent is None:
                    self._release_store(store)
                    continue
                _, m, v, step, state8 = ent
                lp = store.flat_lp
                if lp is not None and store.active_numel != store.numel and not getattr(store, "_lp_tail_ok", None) == store.lp_fmt:
                    # the kernel refreshes only the trained prefix of the 16-bit shadow; the never-trained tail
                    # (final LN, pooler) is constant, so one full cast makes every later refresh complete
                    store.lp(refresh=True)
                    store._lp_tail_ok = store.lp_fmt
                rng = Range(store.flat.data_ptr(), store.flat_grad.data_ptr(), m.data_ptr(), v.data_ptr(),
                            lp.data_ptr() if lp is not None else None, store.active_numel)
                if on_device or state8 is not None:
                    if state8 is None:
                        state8 = new_state8(store.flat.device, step)
                        ent[3], ent[4] = None, state8
                    dev_launches.setdefault((id(state8), store.lp_fmt), (state8, []))[1].append(rng)
                else:
                    host_launches.setdefault((step + 1, store.lp_fmt, store.flat.device), []).append(rng)
                    dev_of[rng.params] = store.flat.device
                    ent[3] = step + 1
                if lp is not None:
                    store.mark_lp_fresh()
                covered.update(id(p) for p, _ in self._active(store))
            if len(covered) != len(params):
                for p in params:
                    if id(p) in covered or p.grad is None:
                        continue
                    if not p.is_cuda:
                        raise RuntimeError("FusedAdam: parameter on CPU — vit2spn has no CPU fallback")
                    if p.grad.is_sparse or p.dtype != torch.float32 or not p.is_contiguous():
                        raise RuntimeError("FusedAdam supports dense contiguous fp32 parameters only")
                    st = self._state_for(p)
                    g = p.grad.contiguous()
                    keep.append(g)
                    rng = Range(p.data_ptr(), g.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), None,
                                p.numel())
                    s8 = self._dev_steps.get(id(p))
                    if on_device or s8 is not None:
                        if s8 is None:
                            s8 = new_state8(p.device, int(float(st["step"])))
                            self._dev_steps[id(p)] = s8
                        dev_launches.setdefault((id(s8), _lib.LP_BF16), (s8, []))[1].append(rng)
                    else:
                        step = int(float(st["step"]))
                        st["step"] += 1
                        host_launches.setdefault((step + 1, _lib.LP_BF16, p.device), []).append(rng)
                        dev_of[rng.params] = p.device
            for (step, fmt, _dev), rs in host_launches.items():
                for i in range(0, len(rs), 4):
                    chunk = rs[i:i + 4]
                    arr = (Range * len(chunk))(*chunk)
                    with torch.cuda.device(dev_of[chunk[0].params]):
                        check(lib.v2s_adam_step(arr, len(chunk), int(step), float(lr), float(b1), float(b2), float(eps),
                                                float(wd), float(self.grad_multiplier), int(fmt), stream_ptr()), "adam_step")
            advanced = set()
            for (sid, fmt), (state8, rs) in dev_launches.items():
                dev = state8.device
                st_, sp = self._scalar_ptr(amp_scale, dev, "grad_scale")
                ft_, fp = self._scalar_ptr(amp_inf, dev, "found_inf")
                keep += [st_, ft_]
                for i in range(0, len(rs), 4):
                    chunk = rs[i:i + 4]
                    arr = (Range * len(chunk))(*chunk)
                    with torch.cuda.device(dev):
                        check(lib.v2s_adam_step_amp(arr, len(chunk), state8.data_ptr(), float(lr), float(b1), float(b2),
                                                    float(eps), float(wd), float(self.grad_multiplier), sp, fp, int(fmt),
                                                    0 if sid in advanced else 1, stream_ptr()), "adam_step_amp")
                    advanced.add(sid)
        return loss
