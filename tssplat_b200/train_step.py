"""One graph-replayable step of the reference's geometry loop (``trainer.py:71-132``): the fused energy + gradient
launch, an optional external gradient (the image loss's ``tet_v.grad``) and ``AdamUniform``, with every per-step
scalar -- the coefficient multiplier of ``coeff_scheduler``, the learning rate of the LR scheduler, the Adam bias
corrections and the ``grad_limit`` value -- read from a schedule table on the device.  A device-side step counter
selects the row, so a sequence of steps is captured once into a CUDA graph and replayed without Python in between.

    step = GeometryStep(energy, tet_v, n_steps, lr=0.2, grad_limit=True, grad_limit_values=[0.01, 0.01],
                        grad_limit_iters=[1500], lr_scheduler=lambda o: CosineAnnealingLR(o, n_steps, eta_min=1e-4))
    step.run(n_steps)                 # graph replays of ``graph_steps`` steps, the remainder eagerly
    loss = step.history()[:, 0]       # per-step reg_loss, on the device

C ABI: ``tsb_train_step`` (``include/tssplat_b200.h``).  Single GPU only: ``AdamUniform``'s maximum runs over the
whole parameter, so a sharded step would need an all-reduce inside the step.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _capi
from . import tet_spheres_ext as _ext

__all__ = ["coeff_multiplier", "build_schedule", "GeometryStep"]


def coeff_multiplier(it: int) -> float:
    """The factor ``SmoothnessBarrierEnergy.coeff_scheduler`` applies to both coefficients at iteration ``it``
    (``energies/smooth_barrier.py:50-54``): ``2 ** (4 |sin(min(it/2400 * pi, pi/2))|)``, in [1, 16]."""
    return math.pow(2, abs(math.sin(min(it / 300.0 / 4 * 0.5 * math.pi, 0.5 * math.pi))) * 4)


def build_schedule(n_steps, *, coeff_multiplier=coeff_multiplier, increase_order_iter, lr, betas=(0.9, 0.999),
                   grad_limit=False, grad_limit_values=(0.05, 0.01), grad_limit_iters=(4000,), lr_scheduler=None,
                   forward_per_iter=1):
    """Per-step table of ``tsb_train_step``: returns ``(table, orders)``, float32 ``[n_steps, 5]`` rows
    ``(m, lr, 1/(1-b1^t), 1/(1-b2^t), grad_limit)`` and the int32 barrier order of every step.  CPU only.

    Step ``k`` belongs to the trainer iteration ``it = k // forward_per_iter`` (``trainer.py:71-72``), which sets
    ``m = coeff_multiplier(it)`` and the order (4 once ``it > increase_order_iter``, ``smooth_barrier.py:61-63``).
    ``lr`` is the learning rate of step ``k`` as ``lr_scheduler`` (a factory ``optimizer -> scheduler``, e.g.
    ``lambda o: CosineAnnealingLR(o, T_max, eta_min=1e-4)``, ``trainer.py:57-58``) sets it when stepped once per
    step over an optimizer with base rate ``lr``; constant without one.  The bias corrections use ``t = k + 1`` and
    the ``grad_limit`` value follows ``AdamUniform``'s ``grad_limit_ptr`` / ``cc`` sequence (``optimizer.py:76-81``:
    the pointer advances after the value is read, one step late); 0 disables the clamp."""
    n_steps, fpi = int(n_steps), int(forward_per_iter)
    if n_steps < 1 or fpi < 1:
        raise ValueError("build_schedule: n_steps and forward_per_iter must be >= 1")
    b1, b2 = (float(b) for b in betas)
    if not (0.0 <= b1 < 1.0 and 0.0 <= b2 < 1.0):
        raise ValueError(f"build_schedule: betas must be in [0, 1), got {betas}")
    lr = float(lr)
    if not (math.isfinite(lr) and lr > 0.0):
        raise ValueError(f"build_schedule: lr must be a positive number, got {lr}")
    table = np.zeros((n_steps, 5), dtype=np.float32)
    orders = np.zeros(n_steps, dtype=np.int32)
    for k in range(n_steps):
        it = k // fpi
        table[k, 0] = coeff_multiplier(it)
        orders[k] = 4 if it > increase_order_iter else 2
        t = float(k + 1)
        table[k, 2] = 1.0 / (1.0 - math.pow(b1, t))              # as launch_adam_uniform: double, then float
        table[k, 3] = 1.0 / (1.0 - math.pow(b2, t))
    if lr_scheduler is None:
        table[:, 1] = lr
    else:
        dummy = torch.optim.SGD([torch.zeros(1, requires_grad=True)], lr=lr)
        sched = lr_scheduler(dummy)
        for k in range(n_steps):
            table[k, 1] = dummy.param_groups[0]["lr"]            # what AdamUniform.step reads (optimizer.py:40)
            dummy.step()                                         # no gradient: a no-op that keeps the call order
            sched.step()
    if grad_limit:
        values, iters = list(grad_limit_values), list(grad_limit_iters)
        ptr = 0
        for cc in range(n_steps):
            if ptr >= len(values):
                raise ValueError(f"build_schedule: grad_limit_values has no entry {ptr} (needed at step {cc})")
            table[cc, 4] = float(values[ptr])                    # optimizer.py:77
            if ptr < len(iters) and cc >= iters[ptr]:            # optimizer.py:79-81
                ptr += 1
    if not np.all(np.isfinite(table)):
        raise ValueError("build_schedule: the schedule has non-finite entries")
    return table, orders


class GeometryStep:
    """The reference's per-step work on ``tet_v`` -- ``SmoothnessBarrierEnergy`` forward + backward, the image
    gradient if any, ``AdamUniform.step`` and the LR scheduler step -- with the optimizer state on the device.

    ``energy``: a ``tssplat_b200.energies.SmoothnessBarrierEnergy`` (its handle and ``FLAGS``: ``smooth_eng_coeff``,
    ``barrier_coeff``, ``increase_order_iter``); ``tet_v``: the float32 CUDA positions ``[n, 3]``, updated in place.
    ``lr``, ``betas``, ``grad_limit*`` as ``AdamUniform``; ``lr_scheduler`` and ``forward_per_iter`` as
    :func:`build_schedule`.  ``state["step"]``, ``state["g1"]``, ``state["g2"]`` are ``AdamUniform``'s state."""

    def __init__(self, energy, tet_v, n_steps, *, lr=0.1, betas=(0.9, 0.999), grad_limit=False,
                 grad_limit_values=(0.05, 0.01), grad_limit_iters=(4000,), lr_scheduler=None, forward_per_iter=1,
                 graph_steps=32):
        sp = energy.tet_sp
        flags = energy.FLAGS
        if not isinstance(tet_v, torch.Tensor) or tet_v.dtype != torch.float32 or not tet_v.is_cuda \
                or not tet_v.is_contiguous() or tet_v.numel() != sp.n3 or tet_v.device != sp.device:
            raise RuntimeError(f"GeometryStep: tet_v must be a contiguous float32 tensor of {sp.n3} entries on {sp.device}")
        if int(graph_steps) < 1:
            raise ValueError("GeometryStep: graph_steps must be >= 1")
        table, self.orders = build_schedule(
            n_steps, increase_order_iter=flags.increase_order_iter, lr=lr, betas=betas, grad_limit=grad_limit,
            grad_limit_values=grad_limit_values, grad_limit_iters=grad_limit_iters, lr_scheduler=lr_scheduler,
            forward_per_iter=forward_per_iter)
        self.n_steps = int(n_steps)
        self.graph_steps = int(graph_steps)
        self.tet_sp, self.tet_v = sp, tet_v
        self.c1, self.c2 = float(flags.smooth_eng_coeff), float(flags.barrier_coeff)   # coeff_scheduler scales both by m
        dev = sp.device
        self.schedule = torch.from_numpy(table).to(dev)
        self.state = {"step": 0, "g1": torch.zeros_like(tet_v), "g2": torch.zeros_like(tet_v)}
        self._grad = torch.zeros(sp.n3, dtype=torch.float32, device=dev)
        self._energy = torch.zeros(4, dtype=torch.float32, device=dev)
        self._history = torch.zeros((self.n_steps, 4), dtype=torch.float32, device=dev)
        self._step = torch.zeros(1, dtype=torch.int32, device=dev)
        self._work = torch.zeros(8, dtype=torch.float32, device=dev)
        b1, b2 = betas
        self._st = _capi.tsb_train_state_t(
            g1=self.state["g1"].data_ptr(), g2=self.state["g2"].data_ptr(), grad=self._grad.data_ptr(),
            energy=self._energy.data_ptr(), schedule=self.schedule.data_ptr(), history=self._history.data_ptr(),
            step=self._step.data_ptr(), work=self._work.data_ptr(), n_steps=self.n_steps, beta1=float(b1), beta2=float(b2))
        self._graphs = {}          # (order, grad_ext pointer) -> (CUDAGraph, grad_ext kept alive)

    # ------------------------------------------------------------------------------------------------------------
    def _check_ext(self, grad_ext):
        if grad_ext is None:
            return None
        sp = self.tet_sp
        if not isinstance(grad_ext, torch.Tensor) or grad_ext.dtype != torch.float32 or grad_ext.device != sp.device \
                or not grad_ext.is_contiguous() or grad_ext.numel() != sp.n3:
            raise RuntimeError(f"GeometryStep: grad_ext must be a contiguous float32 tensor of {sp.n3} entries on {sp.device}")
        return grad_ext

    def _launch(self, order, grad_ext):
        rc = _capi.lib.tsb_train_step(self.tet_sp._h, self.tet_v.data_ptr(),
                                      grad_ext.data_ptr() if grad_ext is not None else None, self.c1, self.c2,
                                      int(order), C.byref(self._st), _ext._stream_ptr(self.tet_sp.device))
        if rc:
            _capi.check(rc, self.tet_sp._h, "GeometryStep")

    def _reserve(self, k):
        if int(k) != k or k < 0:
            raise ValueError(f"GeometryStep: step count must be a non-negative integer, got {k}")
        if self.state["step"] + k > self.n_steps:
            raise RuntimeError(f"GeometryStep: {k} more steps would run past the schedule "
                               f"({self.state['step']} of {self.n_steps} taken)")

    def step(self, grad_ext=None):
        """One step, eagerly: the launches of ``tsb_train_step`` on the current stream, no host sync."""
        grad_ext = self._check_ext(grad_ext)
        self._reserve(1)
        self._launch(self.orders[self.state["step"]], grad_ext)
        self.state["step"] += 1
        _ext.note_parameters_changed()              # tet_v changed through its data pointer

    def _graph(self, order, grad_ext):
        key = (int(order), grad_ext.data_ptr() if grad_ext is not None else 0)
        entry = self._graphs.get(key)
        if entry is None:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):                # captures only: the counter does not move
                for _ in range(self.graph_steps):
                    self._launch(order, grad_ext)
            entry = self._graphs[key] = (g, grad_ext)
        return entry[0]

    def run(self, k, grad_ext=None):
        """``k`` steps: replays of a captured ``graph_steps``-step graph (one per barrier order, captured on first
        use), split at the order switch, and the rest eagerly -- the same kernels either way.  ``grad_ext`` is a
        fixed buffer used by every one of the ``k`` steps; a graph keeps its address, so rewrite its contents
        between calls rather than passing a new tensor each time."""
        grad_ext = self._check_ext(grad_ext)
        self._reserve(k)
        left = int(k)
        G = self.graph_steps
        while left > 0:
            s = self.state["step"]
            order = self.orders[s]
            same = int(np.argmax(self.orders[s:] != order)) or (self.n_steps - s)   # steps until the order switch
            todo = min(left, same)
            for _ in range(todo // G):
                self._graph(order, grad_ext).replay()
                self.state["step"] += G
            for _ in range(todo % G):
                self._launch(order, grad_ext)
                self.state["step"] += 1
            left -= todo
        _ext.note_parameters_changed()

    def reset(self):
        """Back to step 0 with zero moments and history (``AdamUniform.reset``, ``utils/optimizer.py:27-35``), in
        place, so captured graphs stay valid.  ``tet_v`` is the caller's to restore."""
        for t in (self.state["g1"], self.state["g2"], self._history, self._step, self._work):
            t.zero_()
        self.state["step"] = 0

    def history(self):
        """``[steps taken, 4]`` device tensor: per step ``reg_loss`` (the energy the step's gradient belongs to, with
        the scheduled coefficients), smoothness term, barrier term, coefficient multiplier ``m``."""
        return self._history[:self.state["step"]]

    def schedule_overrun(self) -> bool:
        """True if a step ever ran with the device counter past the schedule (it then changed nothing).  Syncs."""
        return bool(self._work.view(torch.int32)[3].item() != 0)
