"""Row f2 (SURVEY.md §8f): TextEncoder on the estimator's kernels.  CPU: oracle vs reference-generated
fixtures; state_dict inventory of the drop-in vs the reference module's.  GPU: CUDA path vs fixtures (1e-3)."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import rel_errs
from oracle import text_encoder_ref as T


@pytest.mark.parametrize("name", list(T.CASES))
def test_oracle_vs_golden(name, golden_dir):
    cs = T.CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    st = T.make_state(3, out_channels=cs["out_channels"])
    ids, c, lens = T.make_inputs(cs["seed"], cs["lens"], cs["T"])
    with torch.inference_mode():
        x, mu, m = T.text_encoder_forward(st, ids, c, lens)
    assert rel_errs(x, torch.from_numpy(g["x"]))[0] < 2e-5 and rel_errs(mu, torch.from_numpy(g["mu"]))[0] < 2e-5
    assert torch.equal(m, torch.from_numpy(g["mask"]))


def test_drop_in_inventory(golden_dir):
    import __graft_entry__ as ge
    ge.build()
    from stabletts_b200 import TextEncoder
    m = TextEncoder(401, 80, 256, 1024, 4, 3, 3, 0.1, 256)
    assert list(m.state_dict().keys()) == list(T.param_shapes().keys())
    m.load_state_dict(T.make_state(3), strict=True)
    with open(os.path.join(golden_dir, "reference_state_dicts.json")) as f:       # the reference's TextEncoder, same sizes
        assert [[k, list(v.shape)] for k, v in m.state_dict().items()] == json.load(f)["TextEncoder"]
    ids, c, lens = T.make_inputs(1, [4], 4)
    with pytest.raises(NotImplementedError):                   # train() mode + autograd: no silent detached output
        m(ids, c, lens)
    with pytest.raises(RuntimeError, match="CUDA"):
        m.eval()(ids, c, lens)


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
@pytest.mark.parametrize("name", list(T.CASES))
def test_cuda_vs_golden(name, engine, golden_dir):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from stabletts_b200 import TextEncoder
    dev = torch.device("cuda:0")
    cs = T.CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    m = TextEncoder(401, cs["out_channels"], 256, 1024, 4, 3, 3, 0.1, 256).eval()
    m.load_state_dict(T.make_state(3, out_channels=cs["out_channels"]), strict=True)
    m = m.to(dev)
    m.set_engine(engine)
    ids, c, lens = T.make_inputs(cs["seed"], cs["lens"], cs["T"])
    x, mu, mask = m(ids.to(dev), c.to(dev), lens.to(dev))
    tol = 1e-3 if engine == "tcgen05" else 5e-5
    ex, emu = rel_errs(x, torch.from_numpy(g["x"])), rel_errs(mu, torch.from_numpy(g["mu"]))
    assert max(ex) < tol and max(emu) < tol, (name, engine, ex, emu)
    assert torch.equal(mask.cpu(), torch.from_numpy(g["mask"]))
