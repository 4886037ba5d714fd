"""Comparison of the oracle port with the unmodified reference on a configuration the CASES goldens do not cover
(s_val_base 2, cos_anneal 0.25, 6 outside samples).  The reference's step on these inputs is stored in
tests/golden/port_step.npz by oracle/make_golden.py: every output, the loss, a seeded sample of every parameter gradient
with the gradient's max magnitude, and the state_dict layout of the reference's modules."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import neuconw_port as port
from oracle import synth
from oracle.make_golden import PORT_CFG, PORT_RAYS, PORT_SEED, sample_index


@pytest.fixture(scope="module")
def G():
    return np.load(os.path.join(GOLDEN, "port_step.npz"))


def test_port_vs_reference_live(params, G):
    cfg = synth.PathConfig(**PORT_CFG, **synth.BRANDENBURG)
    batch = synth.make_rays(PORT_RAYS, cfg, seed=PORT_SEED)
    res_p, loss_p, grads_p = port.train_step(params, cfg, batch, perturb_overwrite=0)
    loss_r = float(G["loss"])
    assert abs(loss_r - float(loss_p)) < 1e-5 * abs(loss_r)
    assert {k for k in G.files if k.startswith("out.")} == {"out." + k for k in res_p}
    for k in res_p:
        a, b = res_p[k].detach().numpy(), G["out." + k]
        assert a.shape == b.shape, k
        if a.size:
            assert np.abs(a - b).max() <= 1e-4 * (np.abs(b).max() + 1e-12), k
    assert {k for k in G.files if k.startswith("gs.")} == {"gs." + k for k in grads_p}
    for k, g in grads_p.items():
        flat = g.reshape(-1)
        a, b = flat[sample_index(flat.numel(), k)].numpy(), G["gs." + k]
        assert np.abs(a - b).max() <= 1e-4 * (float(G["gmax." + k]) + 1e-12), k
        assert abs(float(flat.abs().max()) - float(G["gmax." + k])) <= 1e-4 * (float(G["gmax." + k]) + 1e-12), k


def test_state_dict_names_match_reference(params, G):
    """oracle.synth parameter names/shapes == reference checkpoint layout (SURVEY.md §9.4)."""
    names = {k: tuple(v) for k, v in json.loads(str(G["state_dict_layout"])).items()}
    assert names == {k: tuple(v.shape) for k, v in params.items()}
