"""The tensor-core fused step walks a sample in strips of R rows, and a strip that continues a sample takes
the overlap rows of its hidden layers over from the previous strip instead of recomputing them (tc_carry in
nfk_fused_tc.cuh).  Every per-site operation is the same whichever strip computes it, so y and the stored
hidden layers must be bit-identical for every strip height, including an odd R (the carried h2 rows change
parity plane) and a last strip of one row; log|det J| sums in a strip-dependent order and is held to the
parity tolerance.  The strip height is forced with NFK_TC_R."""
import numpy as np
import pytest
import torch

from oracle import nf_oracle as O
from normflow__b200 import _ops, _C

pytestmark = pytest.mark.gpu

DEV = "cuda"
SHAPE = (16, 12)
STRIPS = (16, 3, 4, 5, 7, 15)      # 16: one strip per sample, nothing carried (the reference)


def _close(got, ref, tol=1e-5):
    got = got.detach().double().cpu().numpy()
    err = np.abs(got - ref)
    bound = tol * np.maximum(np.abs(ref), 1.0)
    assert np.all(err <= bound), f"max excess {np.max(err / bound):.3g} (abs err {err.max():.3g})"


def _inputs(kind, K, B, seed):
    g = torch.Generator('cpu').manual_seed(seed)
    P = 2 if kind == 0 else 3 * K - 2
    rnd = lambda *s, scale=1.0: (torch.randn(*s, generator=g, device='cpu') * scale).to(DEV)
    w = [rnd(8, 1, 3, 3, scale=0.3), rnd(8, 8, 3, 3, scale=0.5 / 72 ** 0.5), rnd(P, 8, 3, 3, scale=0.5 / 72 ** 0.5)]
    b = [rnd(8, scale=0.1), rnd(8, scale=0.1), rnd(P, scale=0.1)]
    x = rnd(B, *SHAPE, scale=1.3).clamp(-4.7, 4.7)
    prm = _C.RqsParams(K, -5.0, 5.0, -5.0, 5.0, 1, 1) if kind == 1 else None
    return w, b, x, prm


def _oracle(x, w, b, kind, parity, inverse, mask_parity):
    mask = O.evenodd_mask(SHAPE, parity=mask_parity)
    layers = [(t.double().cpu().numpy(), bb.double().cpu().numpy()) for t, bb in zip(w, b)]
    kw = dict(xlim=(-5, 5), ylim=(-5, 5), extrap=dict(left='linear', right='linear')) if kind == 1 else {}
    step = O.make_convact_step('rqs' if kind == 1 else 'affine', layers, ['tanh', 'tanh', None], mask, **kw)
    ident = lambda xa, xf, p, l0, inv: (xa, l0)
    steps = [step] if parity == 0 else [ident, step]
    return O.coupling_forward(x.double().cpu().numpy(), np.zeros(x.shape[0]), mask, steps, inverse=inverse)


@pytest.mark.parametrize("kind,K", [(0, 2), (1, 4), (1, 5), (1, 6), (1, 8), (1, 10)])
def test_strip_height_does_not_change_the_step(kind, K, monkeypatch):
    w, b, x, prm = _inputs(kind, K, B=5, seed=23)
    monkeypatch.setenv('NFK_FUSED_TC', '1')
    for parity, mask_parity, inverse in ((0, 0, False), (1, 1, True), (1, 0, False)):
        yo, lo = _oracle(x, w, b, kind, parity, inverse, mask_parity)
        ys = {}
        for R in STRIPS:
            monkeypatch.setenv('NFK_TC_R', str(R))
            with torch.no_grad():
                y, lj = _ops.fused2d_step(x, w, b, kind, prm, mask_parity, parity, 0, inverse)
            _close(y, yo)
            _close(lj, lo)
            ys[R] = y
        for R in STRIPS[1:]:
            assert torch.equal(ys[R], ys[STRIPS[0]]), f"R = {R}"


@pytest.mark.parametrize("kind,K", [(0, 2), (1, 4), (1, 10)])
def test_training_forward_stores_every_row_for_every_strip_height(kind, K, monkeypatch):
    """The rows a continuing strip takes over are stored by the strip that computed them: with the
    outputs poisoned with NaN, h1 and h2 come back complete and equal to the one-strip run."""
    B = 3
    w, b, x, prm = _inputs(kind, K, B, seed=29)
    if prm is None:
        prm = _C.RqsParams(2, 0.0, 1.0, 0.0, 1.0, 0, 0)
    P = w[2].shape[0]
    L0, L1 = SHAPE
    nan = float('nan')
    res = {}
    for R in STRIPS:
        monkeypatch.setenv('NFK_TC_R', str(R))
        y = torch.full_like(x, nan)
        log_out = torch.full((B,), nan, device=DEV)
        h1 = torch.full((B, 8, L0, L1), nan, device=DEV)
        h2 = torch.full((B, 8, L0, L1), nan, device=DEV)
        out = torch.full((B, P, L0, L1), nan, device=DEV)
        _C.check(_C.lib().nfk_fused2d_step_train(
            _C.dev(x), _C.dev(w[0]), _C.dev(b[0]), _C.dev(w[1]), _C.dev(b[1]), _C.dev(w[2]), _C.dev(b[2]),
            8, kind, prm, 0, 1, _C.dev(None), _C.dev(y), _C.dev(log_out), _C.dev(h1), _C.dev(h2), _C.dev(out),
            L0, L1, B, _C.stream()), "fused2d_step_train")
        torch.cuda.synchronize()
        assert not torch.isnan(h1).any() and not torch.isnan(h2).any() and not torch.isnan(y).any(), f"R = {R}"
        res[R] = (y, log_out, h1, h2, out)
    ref = res[STRIPS[0]]
    for R in STRIPS[1:]:
        for got, want in zip(res[R][:1] + res[R][2:], ref[:1] + ref[2:]):
            torch.testing.assert_close(got, want, rtol=0, atol=0, equal_nan=True, msg=f"R = {R}")
        _close(res[R][1], ref[1].double().cpu().numpy())
