"""Pins the oracle: restatement vs the committed fixtures generated from the reference's own modules.  CPU only."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import rel_errs
from oracle import cases, weights
from oracle import estimator_ref as R

# fp32 CPU kernels vs the same kernels: only summation-order noise is expected
TOL = 2e-5

_STATE = {}


def state_for(n_mel):
    if n_mel not in _STATE:
        _STATE[n_mel] = weights.make_state(cases.WEIGHT_SEED, n_mel)
    return _STATE[n_mel]


def test_param_inventory():
    st = state_for(80)
    assert len(st) == 116                                     # SURVEY.md §8a
    assert sum(v.numel() for v in st.values()) == 20_174_928
    assert sum(v.numel() for v in state_for(128).values()) == 20_347_008


@pytest.mark.parametrize("name", list(cases.ESTIMATOR_CASES))
def test_estimator_vs_golden(name, golden_dir):
    cs = cases.ESTIMATOR_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    st = state_for(cs["n_mel"])
    assert abs(weights.checksum(st) - float(g["weight_checksum"])) < 1e-6 * abs(float(g["weight_checksum"])) + 1e-9, "RNG drift"
    inp = weights.make_inputs(cs["seed"], cs["lengths"], cs["T"], cs["n_mel"],
                              t_per_sample=cs.get("t_per_sample", False), t_value=cs.get("t_value", 0.37))
    with torch.inference_mode():
        out = R.estimator_forward(st, inp["t"], inp["x"], inp["mask"], inp["mu"], inp["c"])
    ref = torch.from_numpy(g["out"])
    assert out.shape == ref.shape
    e_max, e_l2 = rel_errs(out, ref)
    assert e_max < TOL and e_l2 < TOL, (e_max, e_l2)
    # estimator output is exactly zero at masked frames (SURVEY.md §8a a4)
    assert float((out * (1 - inp["mask"])).abs().max()) == 0.0


@pytest.mark.parametrize("name", list(cases.SOLVE_CASES))
def test_solve_vs_golden(name, golden_dir):
    cs = cases.SOLVE_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    st = state_for(cs["n_mel"])
    inp = weights.make_inputs(cs["seed"], cs["lengths"], cs["T"], cs["n_mel"])
    fs, fc = weights.make_cfg_params(cases.CFG_SEED, cs["n_mel"])
    cfg = None if cs["cfg"] is None else dict(fake_speaker=fs, fake_content=fc, cfg_strength=cs["cfg"])
    torch.manual_seed(cs["seed"] + 1000)
    z = torch.randn_like(inp["mu"])                          # models/flow_matching.py:45, temperature 1
    out = R.cfm_forward(st, inp["mu"], inp["mask"], cs["steps"], z, inp["c"], cs["method"], cfg)
    e_max, e_l2 = rel_errs(out, torch.from_numpy(g["out"]))
    assert e_max < 1e-4 and e_l2 < 1e-4, (e_max, e_l2)


def test_live_reference_modules(golden_dir):
    """The restatement against the reference's Decoder and RotaryPositionalEmbeddings called on the same weights and
    inputs (oracle/make_golden_modules.py records their outputs)."""
    from oracle.make_golden_modules import DECODER_CALL as cs, ROPE_DIMS, rope_query
    g = np.load(os.path.join(golden_dir, "decoder_rope.npz"))
    st = state_for(80)
    with open(os.path.join(golden_dir, "reference_state_dicts.json")) as f:        # what load_state_dict(strict=True) checks
        assert [[k, list(v.shape)] for k, v in st.items()] == json.load(f)["Decoder"]
    inp = weights.make_inputs(cs["seed"], cs["lengths"], cs["T"], 80, t_per_sample=cs["t_per_sample"])
    with torch.inference_mode():
        out = R.estimator_forward(st, inp["t"], inp["x"], inp["mask"], inp["mu"], inp["c"])
    assert rel_errs(out, torch.from_numpy(g["decoder_out"]))[0] < TOL
    # RoPE restatement is bit-exact against the module (SURVEY.md §8a a10)
    q = rope_query()
    assert abs(weights.checksum([q]) - float(g["rope_q_checksum"])) < 1e-6 * abs(float(g["rope_q_checksum"])), "RNG drift"
    assert torch.equal(R.rope_partial(q, ROPE_DIMS), torch.from_numpy(g["rope_out"]))


def test_padding_is_not_inert():
    """SURVEY.md fact 4: values of x in the padded region leak into valid frames."""
    st = state_for(80)
    inp = weights.make_inputs(5, [40], 48, 80)
    x2 = inp["x"].clone()
    x2[:, :, 40:] = 7.0
    with torch.inference_mode():
        a = R.estimator_forward(st, inp["t"], inp["x"], inp["mask"], inp["mu"], inp["c"])
        b = R.estimator_forward(st, inp["t"], x2, inp["mask"], inp["mu"], inp["c"])
    assert float((a - b)[:, :, :40].abs().max()) > 1e-3


@pytest.mark.parametrize("name", ["loss_b3_ragged", "loss_b1", "loss_b2_mel128"])
def test_cfm_loss_restatement_vs_reference_golden(name, golden_dir):
    """oracle.cfm_loss against fixtures produced by the unmodified reference compute_loss (make_golden_loss.py)"""
    from oracle.make_golden_loss import LOSS_CASES, loss_draws
    cs = LOSS_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    st = weights.make_state(cases.WEIGHT_SEED, cs["n_mel"])
    inp = weights.make_inputs(cs["seed"], cs["lengths"], cs["T"], cs["n_mel"])
    x1 = inp["x"] * inp["mask"]
    u, z = loss_draws(cs["seed"], len(cs["lengths"]), cs["n_mel"], cs["T"])
    assert abs(weights.checksum([x1, inp["mu"], inp["c"], u, z]) - float(g["input_checksum"])) < 1e-6 * max(1.0, abs(float(g["input_checksum"])))
    loss, y = R.cfm_loss(st, x1, inp["mask"], inp["mu"], inp["c"], u, z)
    assert abs(float(loss) - float(g["loss"])) <= 2e-5 * abs(float(g["loss"]))
    assert np.abs(y.numpy() - g["y"]).max() <= 1e-6


def test_fixed_grid_solvers_have_their_published_order():
    """torchdiffeq is absent, so the fixed-grid stepping of the oracle driver is pinned by what its tableaux must
    deliver: on y' = -y + sin(3t) (closed form) halving the step divides the error by ~2^p with p = 1 (euler),
    2 (midpoint), 4 (rk4, the 3/8 rule), 5 (dopri5 on a fixed grid); and the 3/8-rule weights are (1,3,3,1)/8."""
    import math
    f = lambda t, y: -y + torch.sin(3 * t)
    exact = math.exp(-1) * 1.3 + (math.sin(3) - 3 * math.cos(3)) / 10
    y0 = torch.ones(1, dtype=torch.float64)

    def err(method, n):
        ts = torch.linspace(0, 1, n + 1, dtype=torch.float64)
        return abs(float(R.odeint_fixed(f, y0, ts, method)[0]) - exact)

    for method, p, n in [("euler", 1, 64), ("midpoint", 2, 32), ("rk4", 4, 16), ("dopri5_fixed", 5, 16)]:   # asymptotic range
        ratio = err(method, n) / err(method, 2 * n)
        assert 0.8 * 2 ** p < ratio < 1.25 * 2 ** p, (method, ratio)
    # one 3/8-rule step on y' = 1, y' = t, y' = t^2, y' = t^3 integrates exactly (a 4th-order quadrature)
    for k in range(4):
        g = lambda t, y, k=k: t ** k + 0 * y
        out = R.odeint_fixed(g, torch.zeros(1, dtype=torch.float64), torch.tensor([0.0, 1.0], dtype=torch.float64), "rk4")
        assert abs(float(out[0]) - 1.0 / (k + 1)) < 1e-12


def test_cfg_needs_four_pad_frames_for_crop_invariance():
    """ADVICE r1 / shard.bucketed_solve's default min_pad: without CFG an utterance followed by >= 3 pad frames is
    insensitive to further padding; WITH CFG the unconditional branch broadcasts a non-zero fake_content over the pad
    frames, the last valid frame sees cond_proj at frame L which reaches mu[L+3], so a crop needs >= 4 pad frames."""
    from oracle import weights as W
    st = W.make_state(0, 80)
    L = 20
    inp = W.make_inputs(5, [L], L + 12)
    x = inp["x"].clone(); x[:, :, L:] = 0
    fs, fc = W.make_cfg_params(7)
    t = torch.tensor(0.4)

    def run(pad, cfg):
        Tp = L + pad
        a = (x[:, :, :Tp], inp["mask"][:, :, :Tp], inp["mu"][:, :, :Tp], inp["c"])
        with torch.inference_mode():
            o = R.cfg_estimator(st, t, *a, fs, fc, 3.0) if cfg else R.estimator_forward(st, t, *a)
        return o[:, :, :L]

    for cfg in (False, True):
        full = run(12, cfg)
        err = {p: float((run(p, cfg) - full).abs().max() / full.abs().max()) for p in (2, 3, 4, 6)}
        assert err[4] < 5e-6 and err[6] < 5e-6, (cfg, err)
        if cfg:
            assert err[3] > 5e-6, err                 # three pad frames are NOT enough under CFG
        else:
            assert err[3] < 5e-6 and err[2] > 5e-6, err
