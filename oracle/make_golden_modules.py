"""tests/golden/reference_state_dicts.json and tests/golden/decoder_rope.npz from the UNMODIFIED reference's own module
classes (TEST INFRASTRUCTURE ONLY):

    python -m oracle.make_golden_modules <reference checkout>

reference_state_dicts.json: the ordered ``state_dict`` inventory (key -> shape) of the reference's ``Decoder``,
``StableTTS``, ``TextEncoder`` and ``Vocos`` at the sizes the tests build the drop-ins with, so that the tests can check
that a checkpoint saved by the reference loads into the drop-ins unchanged.
decoder_rope.npz: the reference ``Decoder`` on seeded weights / inputs (``oracle.weights``) and its
``RotaryPositionalEmbeddings`` on a seeded query, the two module calls the oracle's restatement is pinned against.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

from oracle import cases, weights

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# the constructor calls the tests make, in the reference's own argument order
DECODER_ARGS = (80, 80, 256, 80, 1024, 0.1, 6, 4, 3, 256)
STABLETTS_ARGS = (401, 80, 256, 1024, 4, 3, 6, 3, 0.1, 256)
TEXT_ENCODER_ARGS = (401, 80, 256, 1024, 4, 3, 3, 0.1, 256)
DECODER_CALL = dict(seed=99, lengths=[70, 45], T=70, t_per_sample=True)
ROPE_SEED, ROPE_SHAPE, ROPE_DIMS = 5, (2, 4, 37, 64), 32

# the vocoder's `models` / `config` packages shadow the TTS ones: its inventory is read in a process of its own
_VOCOS = ("import json, sys; sys.path.insert(0, sys.argv[1]);"
          "from config import MelConfig, VocosConfig; from models.model import Vocos;"
          "print(json.dumps([[k, list(v.shape)] for k, v in Vocos(VocosConfig(), MelConfig()).state_dict().items()]))")


def rope_query() -> torch.Tensor:
    return torch.randn(*ROPE_SHAPE, generator=torch.Generator().manual_seed(ROPE_SEED))


def inventory(module: torch.nn.Module) -> list:
    return [[k, list(v.shape)] for k, v in module.state_dict().items()]


def main(ref: str):
    sys.path.insert(0, ref)
    stub = types.ModuleType("torchdiffeq")                   # absent package; only imported, never called here
    stub.odeint = lambda *a, **k: None
    sys.modules["torchdiffeq"] = stub
    from models.diffusion_transformer import RotaryPositionalEmbeddings
    from models.estimator import Decoder
    from models.model import StableTTS
    from models.text_encoder import TextEncoder
    vocos = subprocess.run([sys.executable, "-c", _VOCOS, os.path.join(ref, "vocoders", "vocos")],
                           capture_output=True, text=True, check=True).stdout
    inv = {"Decoder": inventory(Decoder(*DECODER_ARGS)), "StableTTS": inventory(StableTTS(*STABLETTS_ARGS)),
           "TextEncoder": inventory(TextEncoder(*TEXT_ENCODER_ARGS)), "Vocos": json.loads(vocos)}
    with open(os.path.join(OUT, "reference_state_dicts.json"), "w") as f:          # one parameter per line
        f.write("{\n" + ",\n".join(json.dumps(name) + ": [\n" + ",\n".join(json.dumps(e) for e in entries) + "\n]"
                                     for name, entries in inv.items()) + "\n}\n")

    dec = Decoder(*DECODER_ARGS).eval()
    dec.load_state_dict(weights.make_state(cases.WEIGHT_SEED, 80), strict=True)
    c = DECODER_CALL
    inp = weights.make_inputs(c["seed"], c["lengths"], c["T"], 80, t_per_sample=c["t_per_sample"])
    q = rope_query()
    with torch.inference_mode():
        out = dec(inp["t"], inp["x"], inp["mask"], inp["mu"], inp["c"])
        rope = RotaryPositionalEmbeddings(ROPE_DIMS)(q)
    np.savez_compressed(os.path.join(OUT, "decoder_rope.npz"), decoder_out=out.numpy(), rope_out=rope.numpy(),
                        rope_q_checksum=weights.checksum([q]))
    print({k: len(v) for k, v in inv.items()}, tuple(out.shape), float(out.abs().max()))


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "models")):
        raise SystemExit("usage: python -m oracle.make_golden_modules <reference checkout>")
    main(sys.argv[1])
