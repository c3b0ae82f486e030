"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol the header
declares, the drop-in modules expose the reference's parameter inventory, and there is no CPU
fallback (everything raises off-GPU)."""
import json
import os
import re

import pytest
import torch

from oracle import weights


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    from stabletts_b200 import _lib
    return _lib


def test_library_exports_header_symbols(built):
    lib = built.load_library()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "stabletts_b200.h")).read()
    declared = set(re.findall(r"\b(st_[a-z0-9_]+)\s*\(", header))
    assert declared == set(built.EXPORTS), declared ^ set(built.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.st_version() >= 100


def test_create_fails_loudly_without_gpu(built):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import ctypes as C
    lib = built.load_library()
    dims = built.StDims(80, 256, 1024, 4, 6, 3, 256)
    h = C.c_void_p()
    assert lib.st_create(C.byref(dims), 0, C.byref(h)) != 0
    assert b"no CUDA device" in lib.st_last_error(None)


def test_state_dict_matches_reference_inventory(built):
    from stabletts_b200 import CFMDecoder
    for n_mel, total in ((80, 20_174_928), (128, 20_347_008)):
        m = CFMDecoder(n_mel, n_mel, 256, n_mel, 1024, 4, 6, 3, 0.1, 256)
        sd = m.state_dict()
        ref = weights.estimator_param_shapes(n_mel)
        assert list(sd.keys()) == ["estimator." + k for k in ref]
        assert all(tuple(sd["estimator." + k].shape) == v for k, v in ref.items())
        assert sum(v.numel() for v in sd.values()) == total
        m.estimator.load_state_dict(weights.make_state(0, n_mel), strict=True)
        # adaLN-zero init of the reference (models/estimator.py:98-101)
        fresh = CFMDecoder(n_mel, n_mel, 256, n_mel, 1024, 4, 6, 3, 0.1, 256)
        assert float(fresh.state_dict()["estimator.blocks.0.block.adaLN_modulation.2.weight"].abs().max()) == 0.0


def _reference_inventory(name):
    """Ordered (key, shape) list of the reference module's state_dict (oracle/make_golden_modules.py)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "tests", "golden", "reference_state_dicts.json")) as f:
        return [(k, tuple(v)) for k, v in json.load(f)[name]]


def test_state_dict_keys_equal_live_reference(built):
    from stabletts_b200 import Decoder
    b = Decoder(80, 80, 256, 80, 1024, 0.1, 6, 4, 3, 256).state_dict()
    assert [(k, tuple(v.shape)) for k, v in b.items()] == _reference_inventory("Decoder")


def test_no_cpu_fallback(built):
    from stabletts_b200 import CFMDecoder
    m = CFMDecoder(80, 80, 256, 80, 1024, 4, 6, 3, 0.1, 256).eval()
    inp = weights.make_inputs(1, [8], 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        m.estimator(inp["t"], inp["x"], inp["mask"], inp["mu"], inp["c"])
    with pytest.raises(RuntimeError, match="CUDA"):
        m(inp["mu"], inp["mask"], 2, 1.0, inp["c"], "euler")
    with pytest.raises(RuntimeError, match="CUDA"):          # eval mode: forward value, CUDA only
        m.compute_loss(inp["x"], inp["mask"], inp["mu"], inp["c"])
    with pytest.raises(NotImplementedError):                 # train mode: dropout + backward are out of scope
        m.train().compute_loss(inp["x"], inp["mask"], inp["mu"], inp["c"])


def test_solver_names():
    from stabletts_b200.flow_matching import _method_id, ST_ADAPTIVE
    from stabletts_b200 import _lib
    assert _method_id("euler") == _lib.ST_EULER and _method_id("midpoint") == _lib.ST_MIDPOINT
    assert _method_id("rk4") == _lib.ST_RK4 and _method_id("dopri5_fixed") == _lib.ST_DOPRI5_FIXED
    assert _method_id(None) == ST_ADAPTIVE and _method_id("dopri5") == ST_ADAPTIVE     # the reference's default
    assert _method_id("bosh3") == ST_ADAPTIVE                # further adaptive tableaux (webui.py:110)
    with pytest.raises(ValueError):
        _method_id("implicit_adams")


def test_product_never_imports_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for dirpath, _, files in os.walk(os.path.join(root, "stabletts_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_drop_in_inside_reference_stabletts(built):
    """INTEGRATION.md §1: swapping the class in the reference's own StableTTS keeps its module tree and
    checkpoint keys intact (the synthesise call itself needs a GPU and is covered by the -m gpu tests).  The swap
    replaces the `decoder` subtree only, so the reference's keys stay in order exactly when its `decoder.*` keys are one
    contiguous run equal to the drop-in's, shape for shape."""
    import stabletts_b200
    ref = _reference_inventory("StableTTS")
    pos = [i for i, (k, _) in enumerate(ref) if k.startswith("decoder.")]
    assert pos and pos == list(range(pos[0], pos[-1] + 1))
    ours = stabletts_b200.CFMDecoder(80, 80, 256, 80, 1024, 4, 6, 3, 0.1, 256)     # models/model.py:40
    assert [("decoder." + k, tuple(v.shape)) for k, v in ours.state_dict().items()] == [ref[i] for i in pos]
    ckpt = {k[len("decoder."):]: torch.zeros(shape) for k, shape in (ref[i] for i in pos)}
    ours.load_state_dict(ckpt, strict=True)                          # a reference checkpoint loads unchanged


def _build_c_smoke():
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "build", "c_abi_smoke")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    cmd = ["gcc", os.path.join(root, "tests", "c_abi_smoke.c"), "-I" + os.path.join(root, "include"), "-I/usr/local/cuda/include",
           "-L" + os.path.join(root, "stabletts_b200"), "-lstabletts_b200", "-L/usr/local/cuda/lib64", "-lcudart", "-lm",
           "-Wl,-rpath," + os.path.join(root, "stabletts_b200"), "-o", exe]
    subprocess.run(cmd, check=True, capture_output=True)
    return exe


def test_pure_c_consumer_without_gpu(built):
    """A plain C program (no Python, no torch) links against the C ABI; without a GPU st_create must fail loudly."""
    import subprocess
    if torch.cuda.is_available():
        pytest.skip("GPU present (covered by the gpu test)")
    r = subprocess.run([_build_c_smoke()], capture_output=True, text=True)
    assert r.returncode == 0 and "no CUDA device" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_pure_c_consumer_on_gpu(built):
    import subprocess
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    r = subprocess.run([_build_c_smoke()], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr


def test_modules_can_be_deep_copied_and_pickled_and_refuse_training_graphs():
    """ADVICE r1: the ctypes handle / workspace / sync tags are per-process library state; copies and pickles drop them
    and re-create lazily.  In train() mode with autograd on, forward raises instead of returning a detached eval output."""
    import copy
    import pickle
    from stabletts_b200 import CFMDecoder
    m = CFMDecoder(80, 80, 256, 80, 1024, 4, 2, 3, 0.1, 256)
    m.estimator._synced["x"] = (1, 2)                 # pretend the module has been used
    m2 = copy.deepcopy(m)
    assert m2.estimator._handle is None and m2.estimator._synced == {} and m2.estimator._workspace is None
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    assert m2.estimator.final_proj.weight.data_ptr() != m.estimator.final_proj.weight.data_ptr()
    m3 = pickle.loads(pickle.dumps(m))
    assert m3.estimator._handle is None and list(m3.state_dict()) == list(m.state_dict())
    m.estimator.invalidate_weights()
    assert m.estimator._synced == {}
    m.train()
    with pytest.raises(NotImplementedError):
        m.estimator(torch.tensor(0.1), torch.zeros(1, 80, 4), torch.ones(1, 1, 4), torch.zeros(1, 80, 4), torch.zeros(1, 256))
    m.eval()
    with pytest.raises(RuntimeError, match="CUDA"):       # eval: gets as far as the no-CPU-fallback check
        m.estimator(torch.tensor(0.1), torch.zeros(1, 80, 4), torch.ones(1, 1, 4), torch.zeros(1, 80, 4), torch.zeros(1, 256))
