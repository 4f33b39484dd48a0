"""CPU: the oracle against the committed reference outputs (tests/golden), the
Appendix-B table and analytic known-answer tests."""
import json
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN, golden_names, load_golden
from oracle import supcon_oracle as O


def _kw(meta):
    return dict(temperature=meta["tau"], similarity=meta["similarity"], uniformity_weight=meta["lambda_uni"],
                uniformity_t=meta["uni_t"], topk_neg=meta["topk"], alpha=meta["alpha"])


@pytest.mark.parametrize("name", golden_names())
def test_closed_form_matches_reference_fp64(name):
    meta, g = load_golden(name)
    z, y = torch.from_numpy(g["z"]), torch.from_numpy(g["labels"])
    if meta["n"] < 2:
        pytest.skip("single row: handled by the module wrapper, not the kernels")
    r = O.closed_form(z, y, **_kw(meta))
    assert r["loss"] == pytest.approx(float(g["loss64"]), rel=1e-12, abs=1e-12)
    ref = torch.from_numpy(g["dz64"])
    # ties at the K-th boundary may legitimately be broken differently by the
    # reference's unstable sort; everywhere else the gradients agree to fp64 noise
    err = (r["dz"] - ref).norm() / max(ref.norm().item(), 1e-30)
    if meta["kind"] == "ties":
        assert err < 0.5
    else:
        assert err < 1e-10


@pytest.mark.parametrize("name", golden_names())
def test_anchor_loop_port_matches_reference_fp32(name):
    meta, g = load_golden(name)
    z = torch.from_numpy(g["z"]).clone().requires_grad_(True)
    y = torch.from_numpy(g["labels"])
    loss = O.anchor_loop_loss(z, y, **_kw(meta))
    assert float(loss) == pytest.approx(float(g["loss32"]), rel=1e-6, abs=1e-7)


def test_multiclass_port():
    f = np.load(os.path.join(GOLDEN, "multiclass_n64_d32.npz"))
    z, y = torch.from_numpy(f["z"]).double(), torch.from_numpy(f["labels"])
    zz = z.clone().requires_grad_(True)
    loss = O.anchor_loop_multiclass(zz, y, 0.1)
    loss.backward()
    assert float(loss) == pytest.approx(float(f["loss64"]), rel=1e-12)
    assert torch.allclose(zz.grad, torch.from_numpy(f["dz64"]), rtol=1e-9, atol=1e-12)
    r = O.closed_form(z, y, temperature=0.1, similarity="cosine", topk_neg=0, alpha=0.0)
    assert r["loss"] == pytest.approx(float(f["loss64"]), rel=1e-12)
    assert torch.allclose(r["dz"], torch.from_numpy(f["dz64"]), rtol=1e-9, atol=1e-12)


def test_appendix_b_table():
    rows = json.load(open(os.path.join(GOLDEN, "appendix_b.json")))
    # values printed in SURVEY.md Appendix B (generated from the reference in fp64)
    survey = {(8, 4): 5.563687188701801, (256, 256): 9.435007190758588}
    for row in rows:
        x, y = O.appendix_b_inputs(row["b"], row["d"])
        z, nrm = O.normalize_fwd(x)
        r = O.closed_form(z, y, temperature=row["tau"], similarity=row["similarity"],
                          uniformity_weight=row["lambda_uni"], topk_neg=row["topk"], alpha=row["alpha"])
        assert r["loss"] == pytest.approx(row["loss"], rel=1e-12)
        dx = O.normalize_bwd(z, nrm, r["dz"])
        assert float(dx.norm()) == pytest.approx(row["dx_norm"], rel=1e-8)
        assert float(dx.sum()) == pytest.approx(row["dx_sum"], rel=1e-6, abs=1e-12)
        assert float(dx[0, 0]) == pytest.approx(row["dx_first"], rel=1e-7)
        assert float(dx[-1, -1]) == pytest.approx(row["dx_last"], rel=1e-7)
        key = (row["b"], row["d"])
        if key in survey:
            assert row["loss"] == pytest.approx(survey[key], rel=1e-14)


def test_analytic_known_answers():
    y = torch.tensor([1, 0] * 32)
    z = torch.ones(64, 8, dtype=torch.float64) / math.sqrt(8.0)
    for sim in ("cosine", "geodesic"):
        r = O.closed_form(z, y, temperature=0.07, similarity=sim, topk_neg=15, alpha=0.0, want_grad=False)
        assert r["loss"] == pytest.approx(math.log(63.0), rel=1e-9)
        r = O.closed_form(z, y, temperature=0.07, similarity=sim, topk_neg=15, alpha=1.0, want_grad=False)
        assert r["loss"] == pytest.approx(math.log(46.0), rel=1e-9)
    z = torch.eye(256, dtype=torch.float64)[:64]
    r = O.closed_form(z, y, temperature=0.07, similarity="cosine", uniformity_weight=0.05, uniformity_t=2.0,
                      want_grad=False)
    assert r["loss"] == pytest.approx(3.9431347536906003, rel=1e-12)
    z = torch.zeros(64, 4, dtype=torch.float64)
    z[:, 0] = (2 * y - 1).double()
    r = O.closed_form(z, y, temperature=0.07, similarity="cosine", want_grad=False)
    assert r["loss"] == pytest.approx(3.4339872044855504, rel=1e-12)


def test_tie_rule_lowest_index():
    z = F.normalize(torch.tensor([[1, 0], [1, 0], [0, 1], [0, 1], [0, 1], [.6, .8]], dtype=torch.float64), dim=1)
    y = torch.tensor([1, 1, 0, 0, 0, 0])
    r = O.closed_form(z, y, temperature=0.5, similarity="cosine", topk_neg=2, alpha=1.0, want_topk_idx=True)
    assert r["loss"] == pytest.approx(1.0041676759719849, rel=1e-6)  # SURVEY value is fp32
    assert sorted(r["stats"]["topk_idx"][0]) == [2, 5]
    assert sorted(r["stats"]["topk_idx"][1]) == [2, 5]
    want = torch.tensor([[-0.158372253, 0.191278547], [-0.158372253, 0.191278547],
                         [0.045940824, -0.046645738], [-0.010994585, -0.046645738],
                         [-0.010994585, -0.046645738], [0.291984826, -0.208362624]], dtype=torch.float64)
    assert torch.allclose(r["dz"], want, atol=1e-6)


def test_rowblocks_compose():
    """Two row blocks + summed partials == whole batch (the multi-rank contract)."""
    x, y = O.make_inputs(96, 32, "clustered", classes=3)
    z = F.normalize(x.double(), dim=1)
    kw = dict(tau=0.1, similarity=O.GEODESIC, topk=5, lambda_uni=0.1, uni_t=2.0)
    whole = O.closed_form(z, y, temperature=0.1, similarity="geodesic", uniformity_weight=0.1, topk_neg=5, alpha=0.3)
    s0, p0 = O.rowblock_forward(z, y, 0, 40, **kw)
    s1, p1 = O.rowblock_forward(z, y, 40, 56, **kw)
    loss, coef = O.loss_from_partials(p0 + p1, 96, alpha=0.3, lambda_uni=0.1)
    assert loss == pytest.approx(whole["loss"], rel=1e-13)
    stats = {k: torch.cat([s0[k], s1[k]]) for k in s0}
    dz1 = O.rowblock_backward(z, y, 40, 56, stats, coef, **kw)
    assert torch.allclose(dz1, whole["dz"][40:], rtol=1e-10, atol=1e-14)
