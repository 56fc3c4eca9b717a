"""-m "not gpu": the CMP oracle against the fixture produced by the reference's own CMP module files
(oracle/make_goldens.py: make_cmp -> tests/golden/cmp_small.pt)."""
import os

import pytest
import torch

from oracle import cmp as ocmp

GOLD = os.path.join(os.path.dirname(__file__), "golden", "cmp_small.pt")


@pytest.mark.skipif(not os.path.exists(GOLD), reason="golden not generated")
def test_cmp_oracle_matches_reference_fixture():
    g = torch.load(GOLD)
    b, y, x = g["points"].unbind(1)
    sparse = torch.zeros(g["image"].shape[0], 2, *g["image"].shape[2:])
    mask = torch.zeros_like(sparse)
    sparse[b, :, y, x], mask[b, :, y, x] = g["values"], 1.0
    m = ocmp.CMP().eval()
    m.load_state_dict(ocmp.seeded_state_dict(m, seed=g["seed"]))
    with torch.no_grad():
        logits = m(g["image"] * 2 - 1, torch.cat([sparse, mask], 1))
        flow = ocmp.cmp_demo_run(m, g["image"], sparse, mask)
    assert torch.allclose(logits[:, ::9, ::4, ::4], g["logits_sub"], rtol=1e-5, atol=1e-5)
    assert torch.allclose(flow, g["flow"], rtol=1e-5, atol=1e-4)


def test_convert_flow_bins():
    # a one-hot distribution on bin k must return that bin's centre (k + 0.5) * 100/99 - 50
    nb = 99
    lo = torch.full((1, 2 * nb, 1, 1), -1e4)
    lo[0, 10], lo[0, nb + 98] = 1e4, 1e4
    f = ocmp.convert_flow(lo)
    step = 100.0 / 99
    assert abs(f[0, 0, 0, 0].item() - ((10 + 0.5) * step - 50)) < 1e-4
    assert abs(f[0, 1, 0, 0].item() - ((98 + 0.5) * step - 50)) < 1e-4
