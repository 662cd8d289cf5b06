"""TEST-ONLY stand-in for makeupdiffuse_b200.ops.plms_update (mkd_plms_update of include/mkd_b200.h), in the style of
tests/fake_ops.py: upstream plms.py's own torch expressions on the CPU, so that B200PLMSSampler's host logic (the eps
ring, the two evaluations of step 0, the history order) can be tested without a GPU.  Never imported by the product."""
import torch

import fake_ops


def plms_update(x, eps, x_prev, *, mode, history=(), e_store=None, sqrt_one_minus_at, sqrt_at, sqrt_a_prev, dir_coef,
                pred_x0=None, cfg_scale=None, peer_ptrs=None):
    """upstream plms.py's own torch expressions (p_sample_plms), evaluated in its order"""
    assert peer_ptrs is None, "peer stores need real GPUs"
    assert len(history) == (0, 1, 1, 2, 3)[mode]
    f = lambda v: torch.tensor(v, dtype=torch.float32)  # noqa: E731
    e = eps
    if cfg_scale is not None:
        eu, ec = eps.chunk(2)
        e = eu + f(cfg_scale) * (ec - eu)
    o = history
    if mode == 0:
        ep = e
    elif mode == 1:
        ep = (o[0] + e) / 2
    elif mode == 2:
        ep = (3 * e - o[0]) / 2
    elif mode == 3:
        ep = (23 * e - 16 * o[0] + 5 * o[1]) / 12
    else:
        ep = (55 * e - 59 * o[0] + 37 * o[1] - 9 * o[2]) / 24
    p0 = (x - f(sqrt_one_minus_at) * ep) / f(sqrt_at)
    xp = f(sqrt_a_prev) * p0 + f(dir_coef) * ep
    # stores after every read: e_store may be the oldest history slot and x_prev may be x, as the kernel allows
    if e_store is not None:
        e_store.copy_(e)
    x_prev.copy_(xp)
    if pred_x0 is not None:
        pred_x0.copy_(p0)


def install(ops, patch=setattr):
    """replace every C-ABI wrapper of ``ops`` by its torch stand-in (patch: monkeypatch.setattr in the pytest process,
    plain setattr in a spawned worker)"""
    for name in fake_ops.ALL:
        patch(ops, name, getattr(fake_ops, name))
    patch(ops, "plms_update", plms_update)
