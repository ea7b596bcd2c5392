"""Pin the oracle's whole generate() against a run of the UNMODIFIED reference (CPU shim) on a
trajectory the other pins do not take: dropout 2 with an absolute target label.  The reference's
result is stored as G10 in tests/golden/reference_golden.npz (tests/golden/make_golden.py)."""
import importlib.util
import os
import random

import numpy as np
import torch

from oracle import attack as OA

HERE = os.path.dirname(os.path.abspath(__file__))


def _mod():
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_generate_matches_stored_reference_run():
    """Final mask, final pattern, every log line and the numpy RNG position afterwards equal the reference's, bit for bit."""
    mg = _mod()
    G = np.load(os.path.join(HERE, "golden", "reference_golden.npz"))
    tiny = mg.TinyNet().eval()
    random.seed(1234); torch.manual_seed(1234); np.random.seed(1234)
    log = []
    m, p = OA.generate(tiny, mg.g10_input(), log=log.append, **mg.G10_KW)
    assert np.array_equal(m.numpy(), G["g10_mask"]) and np.array_equal(p.numpy(), G["g10_pattern"])
    assert log == [str(s) for s in G["g10_log"]]
    assert np.array_equal(np.random.get_state()[1][:4], G["g10_rng_np"])
