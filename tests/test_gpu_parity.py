"""-m gpu parity tests: the CUDA path (through the drop-in modules → ctypes → C ABI) against the
reference-generated golden fixtures and the oracle.  Tolerance 1e-3 on max|d|/max|ref| and
||d||2/||ref||2 (BASELINE.json north_star: "within 1e-3 rel-fp32"); the fp32 SIMT engine is held
to 5e-5."""
import os

import numpy as np
import pytest
import torch

from conftest import rel_errs
from oracle import cases, weights
from oracle import estimator_ref as R

pytestmark = pytest.mark.gpu

TOL = {"tcgen05": 1e-3, "simt": 5e-5}
ENGINES = ["simt", "tcgen05"]


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as g
    g.build()
    return torch.device("cuda:0")


_MODELS = {}


def model_for(n_mel, engine, dev):
    from stabletts_b200 import CFMDecoder
    key = (n_mel, engine)
    if key not in _MODELS:
        m = CFMDecoder(n_mel, n_mel, 256, n_mel, 1024, 4, 6, 3, 0.1, 256).eval()
        m.estimator.load_state_dict(weights.make_state(cases.WEIGHT_SEED, n_mel), strict=True)
        m = m.to(dev)
        m.estimator.set_engine(engine)
        _MODELS[key] = m
    return _MODELS[key]


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", list(cases.ESTIMATOR_CASES))
def test_estimator_vs_golden(name, engine, dev, golden_dir):
    cs = cases.ESTIMATOR_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    m = model_for(cs["n_mel"], engine, dev)
    inp = weights.make_inputs(cs["seed"], cs["lengths"], cs["T"], cs["n_mel"],
                              t_per_sample=cs.get("t_per_sample", False), t_value=cs.get("t_value", 0.37))
    out = m.estimator(inp["t"].to(dev), inp["x"].to(dev), inp["mask"].to(dev), inp["mu"].to(dev), inp["c"].to(dev))
    ref = torch.from_numpy(g["out"])
    e_max, e_l2 = rel_errs(out, ref)
    assert e_max < TOL[engine] and e_l2 < TOL[engine], (name, engine, e_max, e_l2)
    assert float((out.cpu() * (1 - inp["mask"])).abs().max()) == 0.0      # exact zeros at masked frames
    assert torch.isfinite(out).all()


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", list(cases.SOLVE_CASES))
def test_solve_vs_golden(name, engine, dev, golden_dir):
    cs = cases.SOLVE_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    m = model_for(cs["n_mel"], engine, dev)
    inp = weights.make_inputs(cs["seed"], cs["lengths"], cs["T"], cs["n_mel"])
    fs, fc = weights.make_cfg_params(cases.CFG_SEED, cs["n_mel"])
    kw = None if cs["cfg"] is None else dict(fake_speaker=fs.to(dev), fake_content=fc.to(dev), cfg_strength=cs["cfg"])
    torch.manual_seed(cs["seed"] + 1000)
    z = torch.randn_like(inp["mu"])                     # same CPU draw the golden generator consumed
    out = m(inp["mu"].to(dev), inp["mask"].to(dev), cs["steps"], 1.0, inp["c"].to(dev), cs["method"], kw, z=z.to(dev))
    e_max, e_l2 = rel_errs(out, torch.from_numpy(g["out"]))
    tol = TOL[engine] * (2.0 if engine == "simt" else 1.0)
    assert e_max < tol and e_l2 < tol, (name, engine, e_max, e_l2)


@pytest.mark.parametrize("engine", ENGINES)
def test_kernel_gemm_and_conv(engine, dev):
    """conv-GEMM engine in isolation vs torch fp64 on the device."""
    import ctypes as C
    from stabletts_b200 import _lib
    m = model_for(80, engine, dev)
    m.estimator._prepare(torch.zeros(1, device=dev), 1, 8, 0)
    lib, h = _lib.load_library(), m.estimator._handle
    s = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device="cpu").manual_seed(5)
    for (Rr, K, N, silu) in [(300, 256, 256, 0), (129, 80, 1024, 1), (1000, 1024, 256, 0), (77, 256, 80, 0), (5, 256, 768, 0)]:
        A = torch.randn(Rr, K, generator=g).to(dev); W = (torch.randn(N, K, generator=g) / K ** 0.5).to(dev)
        b = torch.randn(N, generator=g).to(dev); out = torch.empty(Rr, N, device=dev)
        _lib.check(lib, h, lib.st_test_gemm(h, A.data_ptr(), W.data_ptr(), b.data_ptr(), out.data_ptr(), Rr, K, N, silu, s), "st_test_gemm")
        ref = A.double() @ W.double().T + b.double()
        if silu:
            ref = torch.nn.functional.silu(ref)
        e_max, e_l2 = rel_errs(out, ref)
        assert e_max < 5e-5 and e_l2 < 5e-5, (engine, Rr, K, N, e_max, e_l2)
    for (B, Cin, Cout, T, k) in [(2, 256, 1024, 300, 3), (3, 1024, 256, 131, 3), (1, 80, 1024, 1, 3), (2, 512, 256, 2, 3), (2, 256, 256, 64, 1)]:
        x = torch.randn(B, Cin, T, generator=g).to(dev); w = (torch.randn(Cout, Cin, k, generator=g) / (Cin * k) ** 0.5).to(dev)
        b = torch.randn(Cout, generator=g).to(dev); out = torch.empty(B, Cout, T, device=dev)
        _lib.check(lib, h, lib.st_test_conv(h, x.data_ptr(), w.data_ptr(), b.data_ptr(), out.data_ptr(), B, Cin, Cout, T, k, s), "st_test_conv")
        ref = torch.nn.functional.conv1d(x.double(), w.double(), b.double(), padding=k // 2)
        e_max, e_l2 = rel_errs(out, ref)
        assert e_max < 5e-5 and e_l2 < 5e-5, (engine, B, Cin, Cout, T, k, e_max, e_l2)


@pytest.mark.parametrize("engine", ENGINES)
def test_kernel_attention(engine, dev):
    """masked RoPE attention vs the oracle's restatement of models/diffusion_transformer.py:58-79."""
    from stabletts_b200 import _lib
    m = model_for(80, engine, dev)
    m.estimator._prepare(torch.zeros(1, device=dev), 1, 8, 0)
    lib, h = _lib.load_library(), m.estimator._handle
    s = torch.cuda.current_stream().cuda_stream
    g = torch.Generator().manual_seed(9)
    for lens, T in [([300, 211], 300), ([1], 1), ([33, 0, 40], 40), ([129], 129), ([1000, 517], 1000), ([64, 63, 65], 70)]:
        B = len(lens)
        qkv = torch.randn(B, T, 768, generator=g)
        mask = (torch.arange(T)[None] < torch.tensor(lens)[:, None]).float()
        out = torch.empty(B, T, 256, device=dev)
        _lib.check(lib, h, lib.st_test_attention(h, qkv.to(dev).data_ptr(), mask.to(dev).data_ptr(), out.data_ptr(), B, T, s), "st_test_attention")
        q, k, v = [t.view(B, T, 4, 64).transpose(1, 2).double() for t in qkv.split(256, dim=-1)]
        q, k = R.rope_partial(q, 32), R.rope_partial(k, 32)
        am = mask[:, None, :, None] * mask[:, None, None, :]
        am = torch.zeros_like(am).masked_fill(am == 0, -torch.finfo(torch.float32).max).double()
        ref = torch.nn.functional.scaled_dot_product_attention(q, k, v, attn_mask=am).transpose(1, 2).reshape(B, T, 256)
        ref = ref * mask[:, :, None]
        e_max, e_l2 = rel_errs(out, ref)
        tol = 2e-5 if engine == "simt" else 1e-4
        assert e_max < tol and e_l2 < tol, (engine, lens, e_max, e_l2)


def test_properties_at_benchmark_shape(dev):
    """Size-independent properties at BASELINE cfg1's per-utterance shape (T=1000), small batch:
    batch-permutation equivariance, exact zeros at masked frames, CFG strength 1 == no CFG,
    and >=3 pad frames vs more padding agree (SURVEY.md fact 4)."""
    m = model_for(80, "tcgen05", dev)
    T = 1000
    inp = weights.make_inputs(77, [1000, 640, 873, 1000], T)
    d = {k: v.to(dev) for k, v in inp.items()}
    out = m.estimator(d["t"], d["x"], d["mask"], d["mu"], d["c"])
    perm = torch.tensor([2, 0, 3, 1], device=dev)
    out_p = m.estimator(d["t"], d["x"][perm], d["mask"][perm], d["mu"][perm], d["c"][perm])
    assert rel_errs(out_p, out[perm])[0] < 1e-5
    assert float((out * (1 - d["mask"])).abs().max()) == 0.0
    fs, fc = weights.make_cfg_params(7)
    z = d["x"]
    a = m(d["mu"], d["mask"], 2, 1.0, d["c"], "euler", None, z=z)
    b = m(d["mu"], d["mask"], 2, 1.0, d["c"], "euler", dict(fake_speaker=fs.to(dev), fake_content=fc.to(dev), cfg_strength=1.0), z=z)
    assert rel_errs(b, a)[0] < 1e-4
    # padding: utterance of 640 frames padded to 643 vs 700 (noise in the pad region differs → use zeros there)
    one = weights.make_inputs(78, [640], 700)
    x0 = one["x"].clone(); x0[:, :, 640:] = 0
    o700 = m.estimator(one["t"].to(dev), x0.to(dev), one["mask"].to(dev), one["mu"].to(dev), one["c"].to(dev))
    o643 = m.estimator(one["t"].to(dev), x0[:, :, :643].contiguous().to(dev), one["mask"][:, :, :643].contiguous().to(dev),
                       one["mu"][:, :, :643].contiguous().to(dev), one["c"].to(dev))
    assert rel_errs(o643[:, :, :640], o700[:, :, :640])[0] < 1e-4


def test_graph_replay_and_host_entry(dev, golden_dir):
    """Small solves are replayed as a CUDA graph from the 2nd identical call on: the 1st (direct), 2nd
    (capture + launch) and 3rd (replay) results must be bit-identical; st_solve_host (host buffers,
    copies inside the call) must agree too."""
    import ctypes as C
    from stabletts_b200 import _lib
    cs = cases.SOLVE_CASES["solve_euler10_cfg"]
    m = model_for(cs["n_mel"], "tcgen05", dev)
    inp = weights.make_inputs(cs["seed"], cs["lengths"], cs["T"], cs["n_mel"])
    fs, fc = weights.make_cfg_params(cases.CFG_SEED, cs["n_mel"])
    kw = dict(fake_speaker=fs.to(dev), fake_content=fc.to(dev), cfg_strength=cs["cfg"])
    torch.manual_seed(cs["seed"] + 1000)
    z = torch.randn_like(inp["mu"])
    outs = [m(inp["mu"].to(dev), inp["mask"].to(dev), cs["steps"], 1.0, inp["c"].to(dev), "euler", kw, z=z.to(dev)).cpu() for _ in range(3)]
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2])
    g = np.load(os.path.join(golden_dir, "solve_euler10_cfg.npz"))
    assert rel_errs(outs[2], torch.from_numpy(g["out"]))[0] < 1e-3
    # host-buffer entry point of the C ABI
    lib, h = _lib.load_library(), m.estimator._handle
    B, M, T = z.shape
    zh = z.clone().contiguous(); muh = inp["mu"].contiguous(); mk = inp["mask"].reshape(B, T).contiguous(); ch = inp["c"].contiguous()
    fch, fsh = fc.reshape(-1).contiguous(), fs.reshape(-1).contiguous()
    tspan = (C.c_float * (cs["steps"] + 1))(*torch.linspace(0, 1, cs["steps"] + 1).tolist())
    rc = lib.st_solve_host(h, zh.data_ptr(), muh.data_ptr(), mk.data_ptr(), ch.data_ptr(), fch.data_ptr(), fsh.data_ptr(),
                           C.c_float(cs["cfg"]), tspan, cs["steps"], _lib.ST_EULER, B, T, torch.cuda.current_stream().cuda_stream)
    _lib.check(lib, h, rc, "st_solve_host")
    assert rel_errs(zh, outs[0])[0] < 1e-6


def test_general_binary_mask_and_weight_update(dev):
    """(a) a NON-prefix 0/1 mask (holes inside the utterance): keys with mask 0 are excluded, rows with mask 0
    are exact zeros — the reference supports it through its mask products and so must the kernels;
    (b) an in-place parameter update is picked up (the packed copy is refreshed from the version counter)."""
    st = weights.make_state(cases.WEIGHT_SEED, 80)
    m = model_for(80, "tcgen05", dev)
    inp = weights.make_inputs(123, [200, 150], 200)
    mask = inp["mask"].clone()
    mask[0, 0, 37:49] = 0.0
    mask[0, 0, 130] = 0.0
    mask[1, 0, 0:5] = 0.0                                   # hole at the very start: key 0 is NOT valid
    mu = inp["mu"] * mask
    with torch.inference_mode():
        ref = R.estimator_forward(st, inp["t"], inp["x"], mask, mu, inp["c"])
    out = m.estimator(inp["t"].to(dev), inp["x"].to(dev), mask.to(dev), mu.to(dev), inp["c"].to(dev))
    e = rel_errs(out, ref)
    assert max(e) < 1e-3, e
    assert float((out.cpu() * (1 - mask)).abs().max()) == 0.0
    # (b) weight update
    from stabletts_b200 import CFMDecoder
    m2 = CFMDecoder(80, 80, 256, 80, 1024, 4, 6, 3, 0.1, 256).eval()
    m2.estimator.load_state_dict(st, strict=True)
    m2 = m2.to(dev)
    small = weights.make_inputs(5, [40], 40)
    args = [small[k].to(dev) for k in ("t", "x", "mask", "mu", "c")]
    a = m2.estimator(*args)
    with torch.no_grad():
        m2.estimator.final_proj.weight.mul_(2.0)
        m2.estimator.final_proj.bias.mul_(2.0)
    b = m2.estimator(*args)
    assert rel_errs(b, 2.0 * a)[0] < 1e-5


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", ["loss_b3_ragged", "loss_b1", "loss_b2_mel128"])
def test_compute_loss_vs_reference_golden(name, engine, dev, golden_dir):
    """CFMDecoder.compute_loss (eval, forward value) against the unmodified reference's compute_loss on the same
    injected draws (oracle/make_golden_loss.py): y to fp32 rounding, loss to 1e-3 (measured ~1e-5)."""
    from oracle.make_golden_loss import LOSS_CASES, loss_draws, inject_draws
    cs = LOSS_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    m = model_for(cs["n_mel"], engine, dev)
    inp = weights.make_inputs(cs["seed"], cs["lengths"], cs["T"], cs["n_mel"])
    x1 = inp["x"] * inp["mask"]
    u, z = loss_draws(cs["seed"], len(cs["lengths"]), cs["n_mel"], cs["T"])
    with inject_draws(u, z):
        loss, y = m.compute_loss(x1.to(dev), inp["mask"].to(dev), inp["mu"].to(dev), inp["c"].to(dev))
    assert loss.dim() == 0 and y.shape == x1.shape
    assert np.abs(y.cpu().numpy() - g["y"]).max() <= 2e-6
    assert abs(float(loss) - float(g["loss"])) <= TOL[engine] * abs(float(g["loss"])), (float(loss), float(g["loss"]))
    with pytest.raises(NotImplementedError):
        m.train().compute_loss(x1.to(dev), inp["mask"].to(dev), inp["mu"].to(dev), inp["c"].to(dev))
    m.eval()


def test_long_and_wide_shapes_vs_oracle(dev):
    """BASELINE cfg3's longest bucket (T = 2000, ragged) and the reference's own n_mel = 128 at T = 1000, against the
    oracle computed on the host in the same test (a few seconds of CPU): the maximum sizes of the path, not only
    size-independent properties."""
    for n_mel, lengths, T, seed in [(80, [2000, 1337], 2000, 91), (128, [1000, 777], 1000, 92)]:
        st = weights.make_state(cases.WEIGHT_SEED, n_mel)
        m = model_for(n_mel, "tcgen05", dev)
        inp = weights.make_inputs(seed, lengths, T, n_mel, t_per_sample=True)
        with torch.inference_mode():
            ref = R.estimator_forward(st, inp["t"], inp["x"], inp["mask"], inp["mu"], inp["c"])
        out = m.estimator(inp["t"].to(dev), inp["x"].to(dev), inp["mask"].to(dev), inp["mu"].to(dev), inp["c"].to(dev))
        e = rel_errs(out, ref)
        assert max(e) < 1e-3, (n_mel, T, e)
        assert float((out.cpu() * (1 - inp["mask"])).abs().max()) == 0.0


def test_split_k_small_problems_vs_oracle(dev):
    """Latency-bound small problems run their long-K GEMMs (FFN conv_2, long-skip and cond convs) as split-K slices plus a
    reduce kernel; the factor follows the tile count: T = 300 alone -> 4, two utterances at T = 1316 -> 3 (the case whose
    stale factor once left an empty K slice and hung), four utterances at T = 1000 -> 2.  Each against the oracle, and bit-identical when
    repeated (the slices are summed in a fixed order)."""
    st = weights.make_state(cases.WEIGHT_SEED, 80)
    m = model_for(80, "tcgen05", dev)
    for lengths, T, seed in [([300], 300, 71), ([1316, 1207], 1316, 72), ([1000, 990, 700, 512], 1000, 73)]:
        inp = weights.make_inputs(seed, lengths, T, 80, t_per_sample=True)
        with torch.inference_mode():
            ref = R.estimator_forward(st, inp["t"], inp["x"], inp["mask"], inp["mu"], inp["c"])
        args = [inp[k].to(dev) for k in ("t", "x", "mask", "mu", "c")]
        out = m.estimator(*args)
        e = rel_errs(out, ref)
        assert max(e) < 1e-3, (lengths, e)
        assert torch.equal(out, m.estimator(*args))
    # graph replay of a split-K solve stays valid while other small shapes use the (fixed, never re-allocated) partial buffer
    a = weights.make_inputs(74, [300], 300)
    b = weights.make_inputs(75, [700, 650], 700)
    solve = lambda i: m(i["mu"].to(dev), i["mask"].to(dev), 3, 1.0, i["c"].to(dev), "euler", None, z=i["x"].to(dev)).cpu()
    first = [solve(a) for _ in range(3)]                     # direct, capture, replay
    other = solve(b)
    again = solve(a)                                        # replay after another shape ran in between
    assert all(torch.equal(first[0], o) for o in first[1:] + [again])
    assert torch.equal(other, solve(b))


def test_empty_and_zero_length_inputs(dev):
    """Edge cases: an empty batch and zero frames return empty tensors like the reference's modules do; an utterance
    of length 0 inside a batch (all-zero mask row) yields exact zeros for that row and leaves the others untouched."""
    m = model_for(80, "tcgen05", dev)
    e = m.estimator(torch.tensor(0.3, device=dev), torch.zeros(0, 80, 16, device=dev), torch.zeros(0, 1, 16, device=dev),
                    torch.zeros(0, 80, 16, device=dev), torch.zeros(0, 256, device=dev))
    assert e.shape == (0, 80, 16)
    s0 = m(torch.zeros(2, 80, 0, device=dev), torch.zeros(2, 1, 0, device=dev), 3, 1.0, torch.zeros(2, 256, device=dev), "euler")
    assert s0.shape == (2, 80, 0)
    st = weights.make_state(cases.WEIGHT_SEED, 80)
    inp = weights.make_inputs(55, [70, 0, 33], 70)
    assert float(inp["mask"][1].sum()) == 0.0
    with torch.inference_mode():
        ref = R.estimator_forward(st, inp["t"], inp["x"], inp["mask"], inp["mu"], inp["c"])
    out = m.estimator(inp["t"].to(dev), inp["x"].to(dev), inp["mask"].to(dev), inp["mu"].to(dev), inp["c"].to(dev)).cpu()
    assert torch.isfinite(out).all()
    assert float(out[1].abs().max()) == 0.0
    assert max(rel_errs(out, ref)) < 1e-3


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs[2..4] at (or near) their full per-utterance sizes — VERDICT r1 "configs without a parity record"
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_solve_rows(st, inp, rows, steps, method, kw):
    """Per-utterance oracle solves (utterances are independent on this path, SURVEY.md §8e)."""
    outs = []
    for i in rows:
        sl = slice(i, i + 1)
        outs.append(R.cfm_forward(st, inp["mu"][sl], inp["mask"][sl], steps, inp["x"][sl], inp["c"][sl], method, kw))
    return torch.cat(outs, dim=0)


def test_cfg2_25_step_dormand_prince_T500(dev):
    """BASELINE cfg2's solver at its full depth: 25 fixed Dormand-Prince steps = 150 estimator evaluations at T = 500
    (B = 4, one ragged row) against the oracle — error accumulation over 150 evaluations is where a 1e-5-per-call path
    could drift; the bar stays 1e-3."""
    st = weights.make_state(cases.WEIGHT_SEED, 80)
    m = model_for(80, "tcgen05", dev)
    inp = weights.make_inputs(201, [500, 500, 387, 500], 500)
    with torch.inference_mode():
        ref = R.cfm_forward(st, inp["mu"], inp["mask"], 25, inp["x"], inp["c"], "dopri5_fixed", None)
    out = m(inp["mu"].to(dev), inp["mask"].to(dev), 25, 1.0, inp["c"].to(dev), "dopri5_fixed", None, z=inp["x"].to(dev))
    e = rel_errs(out, ref)
    assert max(e) < 1e-3, e
    assert torch.isfinite(out).all()


def test_cfg3_bucketed_solve_vs_per_utterance_oracle(dev):
    """BASELINE cfg3's plumbing: a seeded U{200..2000} batch solved through shard.bucketed_solve (sorted, cut into cost
    buckets, each cropped to its own maximum + 4 pad frames) against PER-UTTERANCE oracle solves at each utterance's own
    padded length — with CFG (the case ADVICE r1 flagged: the unconditional branch makes pad >= 4 necessary) and without."""
    from stabletts_b200 import shard
    st = weights.make_state(cases.WEIGHT_SEED, 80)
    m = model_for(80, "tcgen05", dev)
    g = torch.Generator().manual_seed(303)
    lens = sorted(int(v) for v in torch.randint(200, 2001, (10,), generator=g))
    T = max(lens)
    inp = weights.make_inputs(304, lens, T)
    fs, fc = weights.make_cfg_params(cases.CFG_SEED)
    for kw_cpu in (None, dict(fake_speaker=fs, fake_content=fc, cfg_strength=3.0)):
        kw = None if kw_cpu is None else dict(fake_speaker=fs.to(dev), fake_content=fc.to(dev), cfg_strength=3.0)
        solve_one = lambda mu, mask, c, z: m(mu, mask, 3, 1.0, c, "euler", kw, z=z)
        out = shard.bucketed_solve(solve_one, inp["mu"].to(dev), inp["mask"].to(dev), inp["c"].to(dev), inp["x"].to(dev),
                                   lens, n_buckets=3).cpu()
        pad = (1 - inp["mask"]).bool().expand_as(out)
        assert torch.equal(out[pad], inp["x"][pad])             # padded frames keep the (unmasked) initial noise, as in the reference
        for i in (0, 4, 9):                                     # shortest, middle, longest: alone, padded to the batch T
            sl = slice(i, i + 1)
            with torch.inference_mode():
                ref = R.cfm_forward(st, inp["mu"][sl], inp["mask"][sl], 3, inp["x"][sl], inp["c"][sl], "euler", kw_cpu)
            L = lens[i]
            e = rel_errs(out[sl, :, :L], ref[:, :, :L])
            assert max(e) < 1e-3, (kw_cpu is not None, i, L, e)


def test_cfg4_doubled_batch_256_spot_check(dev):
    """BASELINE cfg4's per-GPU shape: B = 128 at T = 1000 with CFG = a doubled batch of 256 rows inside the library
    (row b and row 128+b share a sample).  Two Euler steps on the device, utterances {0, 63, 127} re-solved by the
    oracle: a tile-index or batch-offset error in the later rows of the big batch would show here."""
    st = weights.make_state(cases.WEIGHT_SEED, 80)
    m = model_for(80, "tcgen05", dev)
    B, T = 128, 1000
    lens = [T] * B
    lens[63], lens[127] = 811, 977
    inp = weights.make_inputs(405, lens, T)
    fs, fc = weights.make_cfg_params(cases.CFG_SEED)
    kw = dict(fake_speaker=fs.to(dev), fake_content=fc.to(dev), cfg_strength=3.0)
    out = m(inp["mu"].to(dev), inp["mask"].to(dev), 2, 1.0, inp["c"].to(dev), "euler", kw, z=inp["x"].to(dev)).cpu()
    assert torch.isfinite(out).all()
    with torch.inference_mode():
        ref = _oracle_solve_rows(st, inp, (0, 63, 127), 2, "euler", dict(fake_speaker=fs, fake_content=fc, cfg_strength=3.0))
    e = rel_errs(out[[0, 63, 127]], ref)
    assert max(e) < 1e-3, e
    del out
    torch.cuda.empty_cache()


def test_two_devices_in_one_process():
    """Per-device kernel attributes (cudaFuncAttributeMaxDynamicSharedMemorySize is per device): a second module on
    cuda:1 in the same process must launch the >48 KB-smem kernels too, and calling it must not change the caller's
    current device.  Needs >= 2 GPUs (skipped on a 1-GPU machine)."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import __graft_entry__ as g
    g.build()
    from stabletts_b200 import CFMDecoder
    st = weights.make_state(cases.WEIGHT_SEED, 80)
    inp = weights.make_inputs(11, [300, 251], 300)
    outs = []
    for idx in (0, 1):
        d = torch.device("cuda", idx)
        m = CFMDecoder(80, 80, 256, 80, 1024, 4, 6, 3, 0.1, 256).eval()
        m.estimator.load_state_dict(st, strict=True)
        m = m.to(d)
        torch.cuda.set_device(0)
        outs.append(m.estimator(inp["t"].to(d), inp["x"].to(d), inp["mask"].to(d), inp["mu"].to(d), inp["c"].to(d)).cpu())
        assert torch.cuda.current_device() == 0          # the library restored the caller's device
    with torch.inference_mode():
        ref = R.estimator_forward(st, inp["t"], inp["x"], inp["mask"], inp["mu"], inp["c"])
    assert max(rel_errs(outs[0], ref)) < 1e-3 and max(rel_errs(outs[1], ref)) < 1e-3
    assert torch.equal(outs[0], outs[1])


def test_text_encoder_rejects_out_of_range_ids_and_empty_inputs(dev):
    from stabletts_b200.text_encoder import TextEncoder
    enc = TextEncoder(50, 80, 256, 1024, 4, 3, 3, 0.1, 256).eval().to(dev)
    c = torch.zeros(1, 256, device=dev)
    with pytest.raises(IndexError):
        enc(torch.tensor([[1, 2, 50]], device=dev), c, torch.tensor([3], device=dev))
    x, mu, mask = enc(torch.zeros(0, 5, dtype=torch.long, device=dev), torch.zeros(0, 256, device=dev), torch.zeros(0, dtype=torch.long, device=dev))
    assert x.shape == (0, 256, 5) and mu.shape == (0, 80, 5) and mask.shape == (0, 1, 5)


def test_ffn_fp16x2_precision_mode(dev):
    """The two precision modes (st_set_precision / Decoder.set_precision): 'bf16x3' (three passes everywhere) and 'ffn_fp16x2'
    (the default: fp16 activations against fp16 hi / lo weights in conv_1 / conv_2).  At a shape that runs on the 2-CTA kernel (20 x 1024 frames) it must stay inside the
    1e-3 bar, be measurably less exact than the default (proof that the mode is active), leave the default results
    bit-identical after switching back; a 10-step CFG Euler solve at 24 x 512 must stay inside the bar as well."""
    from stabletts_b200 import CFMDecoder
    st = weights.make_state(cases.WEIGHT_SEED, 80)
    m = CFMDecoder(80, 80, 256, 80, 1024, 4, 6, 3, 0.1, 256).eval()
    m.estimator.load_state_dict(st, strict=True)
    m = m.to(dev)
    lens = [1024] * 20
    lens[7], lens[19] = 700, 1001
    big = weights.make_inputs(4, lens, 1024, 80)
    args = [big[k].to(dev) for k in ("t", "x", "mask", "mu", "c")]
    rows = [0, 7, 19]
    with torch.inference_mode():
        ref = R.estimator_forward(st, big["t"], big["x"][rows], big["mask"][rows], big["mu"][rows], big["c"][rows])
    m.estimator.set_precision("bf16x3")
    base = m.estimator(*args).cpu()
    e_def = max(rel_errs(base[rows], ref))
    m.estimator.set_precision("ffn_fp16x2")
    out16 = m.estimator(*args).cpu()
    e_16 = max(rel_errs(out16[rows], ref))
    assert e_16 < 1e-3, e_16
    assert e_16 > 2 * e_def, (e_16, e_def)                     # the mode is on: fp16 activations cost accuracy
    assert float((out16 * (1 - big["mask"])).abs().max()) == 0.0
    # a full solve in the mode
    inp = weights.make_inputs(9, [512] * 23 + [401], 512, 80)
    fs, fc = weights.make_cfg_params(cases.CFG_SEED)
    kw = dict(fake_speaker=fs.to(dev), fake_content=fc.to(dev), cfg_strength=3.0)
    sol = m(inp["mu"].to(dev), inp["mask"].to(dev), 10, 1.0, inp["c"].to(dev), "euler", kw, z=inp["x"].to(dev)).cpu()
    with torch.inference_mode():
        rs = _oracle_solve_rows(st, inp, (0, 23), 10, "euler", dict(fake_speaker=fs, fake_content=fc, cfg_strength=3.0))
    e_solve = max(rel_errs(sol[[0, 23]], rs))
    assert e_solve < 1e-3, e_solve
    print(f"ffn_fp16x2: estimator call {e_16:.2e} (default {e_def:.2e}), 10-step CFG Euler solve {e_solve:.2e}")
    m.estimator.set_precision("bf16x3")
    again = m.estimator(*args).cpu()
    assert torch.equal(again, base)


def test_ffn_fp16x2_margin_at_maximum_sizes(dev):
    """Evidence for the precision decision (VERDICT r1 item 3): the two-pass FFN mode at the path's maximum sizes, at batch
    sizes where the 2-CTA kernel (and therefore the mode) is active — T = 2000 ragged, n_mel = 128 at T = 1000, and the
    150-evaluation Dormand-Prince solve of BASELINE cfg2 at T = 500 — each against the oracle on two utterances.  The mode
    is the library default BECAUSE every one of these stays <= 5e-4 (2x margin under the 1e-3 bar; measured 2.4e-4 / 2.9e-4 /
    4.1e-5, profiles/r2p_margin.log): if this test ever fails, the default has to go back to 'bf16x3'."""
    from stabletts_b200 import CFMDecoder
    errs = {}
    for name, n_mel, lens, T, seed in [("T2000_ragged", 80, [2000] * 9 + [1337], 2000, 91), ("mel128_T1000", 128, [1000] * 19 + [777], 1000, 92)]:
        st = weights.make_state(cases.WEIGHT_SEED, n_mel)
        m = CFMDecoder(n_mel, n_mel, 256, n_mel, 1024, 4, 6, 3, 0.1, 256).eval()
        m.estimator.load_state_dict(st, strict=True)
        m = m.to(dev)
        m.estimator.set_precision("ffn_fp16x2")
        inp = weights.make_inputs(seed, lens, T, n_mel, t_per_sample=True)
        rows = [0, len(lens) - 1]
        with torch.inference_mode():
            ref = R.estimator_forward(st, inp["t"][rows], inp["x"][rows], inp["mask"][rows], inp["mu"][rows], inp["c"][rows])
        out = m.estimator(inp["t"].to(dev), inp["x"].to(dev), inp["mask"].to(dev), inp["mu"].to(dev), inp["c"].to(dev)).cpu()
        errs[name] = max(rel_errs(out[rows], ref))
        del m
        torch.cuda.empty_cache()
    st = weights.make_state(cases.WEIGHT_SEED, 80)
    m = CFMDecoder(80, 80, 256, 80, 1024, 4, 6, 3, 0.1, 256).eval()
    m.estimator.load_state_dict(st, strict=True)
    m = m.to(dev)
    m.estimator.set_precision("ffn_fp16x2")
    inp = weights.make_inputs(93, [500] * 39 + [387], 500)
    with torch.inference_mode():
        ref = _oracle_solve_rows(st, inp, (0, 39), 25, "dopri5_fixed", None)
    out = m(inp["mu"].to(dev), inp["mask"].to(dev), 25, 1.0, inp["c"].to(dev), "dopri5_fixed", None, z=inp["x"].to(dev)).cpu()
    errs["cfg2_150nfe_T500"] = max(rel_errs(out[[0, 39]], ref))
    print("ffn_fp16x2 margin:", {k: f"{v:.2e}" for k, v in errs.items()})
    assert max(errs.values()) < 5e-4, errs          # the condition under which this mode is allowed to be the default
