"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol
the header declares, the Python mirror of the reference API builds the same objects
(masks bit-exact, state_dict keys), the host Metropolis / resampling helpers match the
reference's golden outputs, the product path refuses to run without CUDA, and the
multi-rank gradient averaging works over gloo with world_size 2."""

import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden

import normflow__b200 as nf
from normflow__b200 import _C, Model
from normflow__b200.action import ScalarPhi4Action
from normflow__b200.lib.combo import estimate_logz, fmt_val_err
from normflow__b200.lib.stats import Resampler
from normflow__b200.mask import EvenOddMask, AlongAxesEvenOddMask
from normflow__b200.mcmc import Metropolis
from normflow__b200.nn import (ModuleList_, ConvAct, AffineCoupling_, RQSplineCoupling_, ShiftCoupling_,
                               DistConvertor_)
from normflow__b200.prior import NormalPrior


# ------------------------------------------------------------------ C ABI
def _header_symbols():
    text = open(os.path.join(ROOT, "include", "normflow_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nfk_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from normflow__b200 import _build
    lib_path = _build.build()             # no-op when up to date; nvcc cross-compiles on CPU
    declared = _header_symbols()
    assert len(declared) >= 25
    handle = ctypes.CDLL(lib_path)
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in the header but not exported"
    assert sorted(_C.declared_symbols()) == declared, "ctypes signature table out of sync with the header"
    handle.nfk_strerror.restype = ctypes.c_char_p
    assert handle.nfk_version() >= 100
    assert handle.nfk_strerror(0) == b"ok" and b"unsupported" in handle.nfk_strerror(-2)


def test_ctypes_signatures_have_the_header_arity():
    """Every prototype of include/normflow_b200.h against the argtypes the Python side binds: a drifted argument list
    would corrupt the call frame silently (the GPU tests would only show it as wrong numbers or a fault)."""
    text = open(os.path.join(ROOT, "include", "normflow_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = re.findall(r"\b(?:int|int64_t|uint64_t|void|const char\*)\s+\*?(nfk_\w+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S)
    assert len(protos) == len(_header_symbols())
    checked = 0
    for name, args in protos:
        args = args.strip()
        n = 0 if args in ("", "void") else args.count(",") + 1
        sig = _C._SIGNATURES.get(name)
        if sig is not None:
            assert len(sig) == n, f"{name}: header has {n} parameters, _C._SIGNATURES {len(sig)}"
            checked += 1
    assert checked == len(_C._SIGNATURES)


def test_library_is_sm100a_only():
    out = subprocess.run(["cuobjdump", "--list-elf", _C.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


# ------------------------------------------------------------------ no CPU fallback
_NO_CUDA = r'''
import sys
sys.path.insert(0, {root!r})
import pytest, torch
assert not torch.cuda.is_available()
from normflow__b200.action import ScalarPhi4Action
from normflow__b200.mask import EvenOddMask
from normflow__b200.nn import AffineCoupling_, ConvAct, DistConvertor_
from normflow__b200.prior import NormalPrior

act = ScalarPhi4Action(m_sq=-1.2, lambd=0.5)
with pytest.raises(RuntimeError, match="CUDA"):
    act(torch.zeros(2, 4, 4))
prior = NormalPrior(shape=(4, 4))
with pytest.raises(RuntimeError, match="CUDA"):
    prior.sample(2)
with pytest.raises(RuntimeError, match="CUDA"):
    prior.log_prob(torch.zeros(2, 4, 4))
mask = EvenOddMask(shape=(4, 4))
cpl = AffineCoupling_([ConvAct(1, 2, 3, hidden_sizes=[4], acts=['tanh', None])], mask=mask)
with pytest.raises(RuntimeError, match="CUDA"):
    cpl(torch.zeros(2, 4, 4))
with pytest.raises(RuntimeError, match="CUDA"):
    DistConvertor_(5, symmetric=True)(torch.zeros(3, 1))
print("refused")
'''


def test_hot_path_refuses_cpu_tensors(tmp_path):
    """Without a visible CUDA device the package keeps its objects on the CPU, and every kernel entry
    refuses them.  Runs in a child process with the GPUs hidden, so that it checks this on any machine."""
    script = tmp_path / "no_cuda.py"
    script.write_text(_NO_CUDA.format(root=ROOT))
    r = subprocess.run([sys.executable, str(script)], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=240)
    assert r.returncode == 0 and "refused" in r.stdout, r.stdout


# ------------------------------------------------------------------ masks (bit-exact)
def test_python_masks_bit_exact():
    g = load_golden("masks")
    for key in g.files:
        if not key.endswith("_meta"):
            continue
        tag, meta = key[:-5], g[key]
        parity, mu, shape = int(meta[0]), int(meta[1]), tuple(int(v) for v in meta[2:])
        if tag.startswith("eo_"):
            m = EvenOddMask(shape=shape, parity=parity, exclude_mu=None if mu < 0 else mu)
            assert np.array_equal(m._c_mask.cpu().numpy(), g[tag + "_cmask"])
        else:
            m = AlongAxesEvenOddMask(shape=shape, parity=parity, mu=mu)
        assert m._mask.dtype == torch.uint8
        assert np.array_equal(m._mask.cpu().numpy(), g[tag + "_mask"])


# ------------------------------------------------------------------ API surface / state_dict
def _build_model(shape=(4, 4)):
    mask = EvenOddMask(shape=shape)
    conv = dict(in_channels=1, hidden_sizes=[8, 8], kernel_size=3, conv_dim=len(shape),
                acts=('tanh', 'tanh', None), bias=False)
    net_ = ModuleList_([
        AffineCoupling_([ConvAct(out_channels=2, **conv) for _ in range(2)], mask=mask),
        RQSplineCoupling_([ConvAct(out_channels=28, **conv) for _ in range(2)], mask=mask,
                          xlim=(-5, 5), ylim=(-5, 5), extrap=dict(left='linear', right='linear')),
        DistConvertor_(10, symmetric=True),
    ])
    return Model(prior=NormalPrior(shape=shape), net_=net_, action=ScalarPhi4Action(m_sq=-1.2, lambd=0.5))


def test_state_dict_keys_follow_reference_layout():
    model = _build_model()
    keys = list(model.net_.state_dict().keys())
    assert '0.nets.0.0.weight' in keys and '0.nets.1.4.weight' in keys      # conv, act, conv, act, conv
    assert '0.mask._mask' in keys and '0.mask._c_mask' in keys               # mask buffers (mask.py:23-24)
    assert '2.1.weights_x' in keys and '2.1.weights_d' in keys               # DistConvertor_ spline layer
    assert model.net_.npar == sum(p.numel() for p in model.net_.parameters())
    # ConvAct(1->8->8->28) without bias: 9*(8 + 64 + 224) weights
    assert sum(p.numel() for p in model.net_[1].nets[0].parameters()) == 9 * (8 + 64 + 224)
    blob = model.net_.get_weights_blob()
    model.net_.set_weights_blob(blob)
    assert model.raw_dist is model.posterior and model.device_handler.nranks == 1


def test_conv4d_weight_layout_matches_reference():
    from normflow__b200.nn import Conv4d
    g = load_golden("conv")
    conv = Conv4d(1, 3, 3, bias=True)
    assert tuple(conv._conv_lower_dim.weight.shape) == tuple(g["d4_wlower0"].shape) == (9, 1, 3, 3, 3)
    with torch.no_grad():
        conv._conv_lower_dim.weight.copy_(torch.from_numpy(g["d4_wlower0"]).float())
    np.testing.assert_array_equal(conv.weight.detach().cpu().numpy(), g["d4_w0"].astype(np.float32))
    assert 'bias' in conv.state_dict() and '_conv_lower_dim.weight' in conv.state_dict()


def test_action_coefficients():
    act = ScalarPhi4Action(kappa=0.67, m_sq=-4 * 0.67, lambd=0.5)
    w0, w2, w4 = act.get_coef(2)
    assert np.isclose(w0, 0.67) and np.isclose(w2, 0.5 * (-2.68 + 4 * 0.67)) and w4 == 0.5
    w0, w2, w4 = ScalarPhi4Action(kappa=0.5, m_sq=0.3, lambd=0.2, a=0.5).get_coef(3)
    assert np.isclose(w0, 0.25) and np.isclose(w2, 0.5 * (0.3 * 0.125 + 2 * 0.25 * 3)) and np.isclose(w4, 0.025)


# ------------------------------------------------------------------ Metropolis host helpers
def test_metropolis_host_api_golden():
    g = load_golden("mcmc")
    np.random.seed(7)
    st = Metropolis.calc_accept_status(g["logqp"])
    assert st.dtype == bool and st[0] and np.array_equal(st, g["status_noref"])
    assert np.array_equal(Metropolis.calc_accept_indices(st), g["ind_noref"])
    np.random.seed(8)
    st = Metropolis.calc_accept_status(g["logqp"], logqp_ref=float(g["ref"]))
    assert np.array_equal(st, g["status_ref"])
    assert np.array_equal(Metropolis.calc_accept_indices(st), g["ind_ref"])
    # exactly one np.random.rand(B) is consumed per call
    np.random.seed(7)
    Metropolis.calc_accept_status(g["logqp"])
    after = np.random.rand()
    np.random.seed(7)
    np.random.rand(len(g["logqp"]))
    assert after == np.random.rand()


def test_estimate_logz_jackknife_closed_form():
    rs = np.random.RandomState(0)
    logqp = torch.from_numpy(rs.randn(257) * 0.7 + 0.3)
    mean, std = estimate_logz(logqp, method='jackknife')
    x = -logqp
    n = len(x)
    brute = [torch.logsumexp(torch.cat([x[:i], x[i + 1:]]), 0).item() - np.log(n) for i in range(n)]
    assert np.isclose(mean, torch.logsumexp(x, 0).item() - np.log(n))
    assert np.isclose(std, np.std(brute), rtol=1e-9)
    m2, s2 = estimate_logz(logqp, n_resamples=20, method='bootstrap')
    assert np.isclose(m2, mean) and s2 > 0


def test_resampler_and_formatting():
    data = np.arange(12.0)
    jk = list(Resampler('jackknife')(data))
    assert len(jk) == 12 and all(len(r) == 11 for r in jk) and 3.0 not in jk[3]
    sh = list(Resampler('shuffling')(torch.arange(10.0), n_resamples=3))
    assert len(sh) == 3 and all(sorted(r.tolist()) == list(range(10)) for r in sh)
    bs = list(Resampler('bootstrap')(data, n_resamples=4, binsize=2))
    assert len(bs) == 4 and all(len(r) == 12 for r in bs)
    mean, std = Resampler('jackknife').eval(data)
    assert np.isclose(mean, 5.5)
    assert fmt_val_err(1.112445, 0.000022, err_digits=2) == "1.112445(22)"
    assert fmt_val_err(0.988, 0.003, err_digits=1) == "0.988(3)"
    assert "+-" in fmt_val_err(1.0, 0.0)


def test_fitter_static_losses():
    fit = _build_model().fit
    rs = np.random.RandomState(1)
    logq, logp = torch.from_numpy(rs.randn(64)), torch.from_numpy(rs.randn(64))
    assert torch.isclose(fit.calc_kl_mean(logq, logp), (logq - logp).mean())
    assert 0 < fit.calc_ess(logq, logp) <= 1
    same = fit.calc_ess(logq, logq)
    assert torch.isclose(same, torch.tensor(1.0, dtype=same.dtype))
    assert torch.isclose(fit.calc_direct_kl_mean(logq, logq), torch.zeros((), dtype=logq.dtype), atol=1e-12)


# ------------------------------------------------------------------ data parallel over gloo, world_size 2
_WORKER = r'''
import os, sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
from normflow__b200 import Model
from normflow__b200.device._core import setup_process_group
from normflow__b200.prior import NormalPrior
from normflow__b200.action import ScalarPhi4Action
from normflow__b200.nn import DistConvertor_

rank, world, port = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
setup_process_group(rank, world, master_port=port, backend="gloo")
torch.manual_seed(100 + rank)
model = Model(prior=NormalPrior(shape=1), net_=DistConvertor_(6, symmetric=True),
              action=ScalarPhi4Action(kappa=0, m_sq=-1.2, lambd=0.5))
with torch.no_grad():
    for p in model.net_.parameters():
        p.add_(torch.randn_like(p))            # ranks start apart ...
h = model.device_handler
h.ddp_wrapper(rank, world, device=torch.device("cpu"))
ref = [p.detach().clone() for p in model.net_.parameters()]
gathered = [torch.empty_like(ref[0]) for _ in range(world)]
dist.all_gather(gathered, ref[0])
assert all(torch.equal(g, gathered[0]) for g in gathered), "... and are broadcast equal"
# every parameter's grad is a view into one flat buffer
params = list(model.net_.parameters())
assert all(p.grad is not None for p in params)
base = h._flat_grad.data_ptr()
assert params[0].grad.data_ptr() == base
# rank r contributes gradient (r + 1) everywhere -> average (1 + 2) / 2 = 1.5
h.zero_grad()
for p in params:
    p.grad += float(rank + 1)
h.sync_gradients()
assert all(torch.allclose(p.grad, torch.full_like(p, 1.5)) for p in params)
# a grad replaced behind our back is folded back into the flat buffer
params[0].grad = torch.full_like(params[0], float(rank))
h.sync_gradients()
assert torch.allclose(params[0].grad, torch.full_like(params[0], 0.5))
assert params[0].grad.data_ptr() == base
# all-gather keeps rank order; mean reduces
x = torch.arange(3.0) + 10 * rank
out = h.all_gather_into_tensor(x)
assert out.tolist() == [0, 1, 2, 10, 11, 12]
assert torch.allclose(h.all_reduce_mean(torch.tensor([float(rank)])), torch.tensor([0.5]))
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_data_parallel_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    port = 29000 + os.getpid() % 2000
    procs = [subprocess.Popen([sys.executable, str(script), str(r), "2", str(port)],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, out) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{out}"
        assert f"rank {r} ok" in out


def test_prepare_seeds():
    from normflow__b200.device._core import prepare_seeds, gen_seed
    assert prepare_seeds(3, [1, 2, 3]) == [1, 2, 3]
    seeds = prepare_seeds(4, None)
    assert len(seeds) == 4 and all(0 <= s < 2 ** 32 for s in seeds)
    with pytest.raises(AssertionError):
        prepare_seeds(2, [1])
    assert isinstance(gen_seed(), int)


def test_fused2d_supported_mirrors_kernel_dispatch():
    """Which lattices take the single-kernel coupling step (nfk_fused.cu / nfk_fused_tc.cu dispatch)."""
    from normflow__b200 import _ops
    ok = _ops.fused2d_supported
    assert ok(64, 64, 10) and ok(16, 16, None) and ok(2, 2, 6) and ok(6, 10, 5)      # tensor-core kernel: even sides
    assert ok(7, 8, 10) and ok(5, 12, 16)                                            # CUDA-core kernel: L1 % 4 == 0
    assert not ok(7, 10, 10)            # odd rows and L1 % 4 != 0: neither kernel
    assert not ok(64, 64, 12) or 12 in _ops.FUSED2D_KNOTS                            # K = 12 only on the CUDA-core kernel
    assert ok(64, 64, 12) and not ok(6, 10, 12)
    assert not ok(64, 64, 7) and not ok(64, 64, -1)
    assert not ok(3, 3, None)


# ------------------------------------------------------------------ blocked MCMC host logic (CPU)
def test_blocked_mcmc_host_logic_replays_reference_chain():
    """BlockedMCMCSampler's control flow (sweeps, restore on reject, reuse of the accepted proposal, chain state
    across calls) with the numerics supplied by the oracle on the host: replaying the reference's recorded block
    proposals and np.random stream must reproduce its accept flags bit for bit and its chain to rounding."""
    from oracle import nf_oracle as O
    from test_oracle_rank4 import blocked_setup
    from normflow__b200.mcmc import BlockedMCMCSampler
    from normflow__b200.prior.prior import BlockUpdater

    g = load_golden("blocked_mcmc")
    evaluate, inverse = blocked_setup(g)
    lens, flat = g["draw_lens"], g["draws"]
    offs = np.concatenate([[0], np.cumsum(lens)])
    draws = iter([torch.from_numpy(flat[offs[i]:offs[i + 1]].reshape(1, -1).copy()) for i in range(len(lens))])
    lat = tuple(int(v) for v in g["lat"])

    class Chopped:
        def sample(self, batch_size=1):
            return next(draws)

    class HostPrior:
        shape, nvar = lat, int(np.prod(lat))

        def sample(self, batch_size=1):
            return torch.from_numpy(g["x0"].copy())

        def setup_blockupdater(self, block_len):
            self.blockupdater = BlockUpdater(Chopped(), block_len)

        def log_prob(self, x):
            return torch.from_numpy(O.normal_log_prob(x.double().numpy()))

    class HostNet:
        def __call__(self, x, log0=0):
            self.last = evaluate(x.double().numpy())
            y, logq, _ = self.last
            return torch.from_numpy(y), torch.from_numpy(O.normal_log_prob(x.double().numpy()) - logq)

        def backward(self, y, log0=0):
            return torch.from_numpy(inverse(y.double().numpy())), 0

    class HostModel:
        prior, net_ = HostPrior(), HostNet()

        def action(self, y):
            return torch.from_numpy(-self.net_.last[2])

    sampler = BlockedMCMCSampler(HostModel())
    np.random.seed(9)
    for call in range(3):
        B, nb = (int(v) for v in g[f"call{call}_shape"])
        cfgs, logq, logp = sampler.sample__(batch_size=B, n_blocks=nb, bookkeeping=True)
        assert np.array_equal(sampler.history.accept_seq[-1], g[f"call{call}_accept_seq"])
        np.testing.assert_allclose(cfgs.numpy(), g[f"call{call}_cfgs"], rtol=2e-6, atol=2e-6)
        np.testing.assert_allclose(logq.numpy(), g[f"call{call}_logq"], rtol=2e-6, atol=2e-5)
        np.testing.assert_allclose(logp.numpy(), g[f"call{call}_logp"], rtol=2e-6, atol=2e-5)
        assert abs(sampler.history.accept_rate[-1] - float(g[f"call{call}_accept_rate"])) < 1e-12
    assert next(draws, None) is None
