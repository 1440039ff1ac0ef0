"""build_schedule (tssplat_b200.train_step): the per-step table of tsb_train_step against the reference's own
formulas -- coeff_scheduler's multiplier and the order switch (energies/smooth_barrier.py:47-63), torch's LR
scheduler, AdamUniform's bias corrections and grad_limit sequence (utils/optimizer.py:55-86) -- as exact float32
equality.  CPU only."""
import math

import numpy as np
import pytest
import torch

from tssplat_b200.train_step import build_schedule


def _m_ref(it):
    return np.float32(math.pow(2, abs(math.sin(min(it / 300.0 / 4 * 0.5 * math.pi, 0.5 * math.pi))) * 4))


@pytest.mark.parametrize("fpi", [1, 3])
def test_multiplier_and_order_switch(fpi):
    n = 1250 * fpi
    table, orders = build_schedule(n, increase_order_iter=700, lr=0.2, forward_per_iter=fpi)
    assert table.dtype == np.float32 and table.shape == (n, 5) and orders.shape == (n,)
    for k in range(n):
        it = k // fpi
        assert table[k, 0] == _m_ref(it), k
        assert orders[k] == (4 if it > 700 else 2), k
    assert table[0, 0] == 1.0 and table[1200 * fpi, 0] == 16.0 and orders[701 * fpi - 1] == 2 and orders[701 * fpi] == 4
    assert np.all(table[:, 1] == np.float32(0.2))        # no scheduler: constant lr
    assert np.all(table[:, 4] == 0.0)                    # grad_limit off


def test_cosine_annealing_lr_matches_torch():
    n, T = 2000, 1500
    table, _ = build_schedule(n, increase_order_iter=10, lr=0.2,
                              lr_scheduler=lambda o: torch.optim.lr_scheduler.CosineAnnealingLR(o, T, eta_min=1e-4))
    p = torch.nn.Parameter(torch.zeros(3))
    opt = torch.optim.Adam([p], lr=0.2)                  # any optimizer: the scheduler only touches param_groups
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T, eta_min=1e-4)
    want = []
    for _ in range(n):
        want.append(opt.param_groups[0]["lr"])
        opt.step()
        sched.step()
    assert np.array_equal(table[:, 1], np.asarray(want, dtype=np.float64).astype(np.float32))
    assert table[0, 1] == np.float32(0.2) and table[T, 1] == np.float32(1e-4)


def test_bias_corrections():
    b1, b2 = 0.9, 0.999
    table, _ = build_schedule(500, increase_order_iter=10, lr=0.1, betas=(b1, b2))
    for k in range(500):
        t = k + 1
        assert table[k, 2] == np.float32(1.0 / (1.0 - math.pow(b1, float(t))))     # launch_adam_uniform
        assert table[k, 3] == np.float32(1.0 / (1.0 - math.pow(b2, float(t))))
        assert table[k, 2] == np.float32(1.0 / (1 - b1 ** t))                       # utils/optimizer.py:67-68


@pytest.mark.parametrize("values,iters", [([0.05, 0.01], [4]), ([0.5, 0.2, 0.1, 0.05], [0, 1, 7]),
                                          ([0.3, 0.2, 0.1], [3, 3])])
def test_grad_limit_sequence_with_its_lag(values, iters):
    n = 20
    table, _ = build_schedule(n, increase_order_iter=10, lr=0.1, grad_limit=True, grad_limit_values=values,
                              grad_limit_iters=iters)
    # utils/optimizer.py:76-86, inline: the value is read before the pointer moves
    ptr, cc, want = 0, 0, []
    for _ in range(n):
        m = values[ptr]
        if ptr < len(iters):
            if cc >= iters[ptr]:
                ptr += 1
        want.append(m)
        cc += 1
    assert np.array_equal(table[:, 4], np.asarray(want, dtype=np.float32))
    if iters == [4]:                                      # the lag: step 4 still uses values[0]
        assert table[4, 4] == np.float32(0.05) and table[5, 4] == np.float32(0.01)


def test_bad_arguments_raise():
    kw = dict(increase_order_iter=10, lr=0.1)
    with pytest.raises(ValueError):
        build_schedule(0, **kw)
    with pytest.raises(ValueError):
        build_schedule(10, forward_per_iter=0, **kw)
    with pytest.raises(ValueError):
        build_schedule(10, increase_order_iter=10, lr=-1.0)
    with pytest.raises(ValueError):
        build_schedule(10, increase_order_iter=10, lr=float("nan"))
    with pytest.raises(ValueError):
        build_schedule(10, betas=(1.0, 0.999), **kw)
    with pytest.raises(ValueError):
        build_schedule(10, betas=(0.9, -0.1), **kw)
    with pytest.raises(ValueError):                      # the pointer runs past grad_limit_values (IndexError in the reference)
        build_schedule(10, grad_limit=True, grad_limit_values=[0.05], grad_limit_iters=[2], **kw)
    with pytest.raises(ValueError):
        build_schedule(10, coeff_multiplier=lambda it: float("inf"), **kw)
