"""Row f4 (SURVEY.md §8f): the vocoder hand-off.  CPU: state_dict inventory of the drop-in against the oracle's restated
inventory and the unmodified reference Vocos's (as recorded in tests/golden).  GPU: the CUDA path through the C ABI against
the fixtures generated from the unmodified reference (tests/golden/vocos_*.npz, 1e-3) and against the oracle at sizes that
reach the 2-CTA GEMM kernel; size-independent properties (batch independence, frame-count scaling of the output)."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import rel_errs
from oracle import vocoder_ref as V


def test_drop_in_inventory_matches_reference_keys(golden_dir):
    import __graft_entry__ as ge
    ge.build()
    from stabletts_b200 import Vocos
    m = Vocos()
    want = V.param_shapes()
    got = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert list(got) == list(want) and got == dict(want)
    m.load_state_dict(V.make_state(), strict=True)
    with open(os.path.join(golden_dir, "reference_state_dicts.json")) as f:     # Vocos(VocosConfig(), MelConfig())
        assert [(k, tuple(v)) for k, v in json.load(f)["Vocos"]] == list(got.items())
    with pytest.raises(RuntimeError, match="CUDA"):
        m.eval()(torch.zeros(1, 128, 4))


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as g
    g.build()
    return torch.device("cuda:0")


def _model(dev, engine="tcgen05", **dims):
    from stabletts_b200 import Vocos
    d = dict(V.DIMS); d.update(dims)
    m = Vocos(**d).eval()
    m.load_state_dict(V.make_state(**dims), strict=True)
    m = m.to(dev)
    m.set_engine(engine)
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
@pytest.mark.parametrize("name", list(V.CASES))
def test_vocos_vs_reference_golden(name, engine, dev, golden_dir):
    cs = V.CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    m = _model(dev, engine)
    mel = V.make_mel(cs["seed"], cs["B"], cs["T"])
    audio = m(mel.to(dev))
    ref = torch.from_numpy(g["audio"])
    assert audio.shape == ref.shape == (cs["B"], cs["T"] * 512)
    e = rel_errs(audio, ref)
    assert max(e) < (1e-3 if engine == "tcgen05" else 2e-4), (name, engine, e)
    assert torch.isfinite(audio).all()


@pytest.mark.gpu
def test_vocos_large_vs_oracle_and_properties(dev):
    """B = 6, T = 700 (4200 frames: the pwconv GEMMs reach the 2-CTA kernel) against the oracle on the host; an utterance's
    audio does not depend on its batch neighbours; n_mel = 80 (the CFM path's BASELINE width) works as input width."""
    st = V.make_state()
    m = _model(dev)
    mel = V.make_mel(77, 6, 700)
    audio = m(mel.to(dev)).cpu()
    with torch.inference_mode():
        ref = V.vocos_forward(st, mel[[0, 5]])
    e = rel_errs(audio[[0, 5]], ref)
    assert max(e) < 1e-3, e
    alone = m(mel[2:3].to(dev)).cpu()
    assert rel_errs(alone, audio[2:3])[0] < 1e-5
    m80 = _model(dev, input_channels=80)
    st80 = V.make_state(input_channels=80)
    mel80 = V.make_mel(78, 2, 130, n_mel=80)
    with torch.inference_mode():
        ref80 = V.vocos_forward(st80, mel80)
    assert max(rel_errs(m80(mel80.to(dev)), ref80)) < 1e-3
    assert m(torch.zeros(0, 128, 5, device=dev)).shape == (0, 2560)
