"""CPU: the C-ABI library loads and exports what include/supcon_b200.h declares;
the drop-in classes mirror the reference's interface and error behaviour."""
import ctypes
import inspect
import os
import re
import sys

import pytest
import torch

from conftest import ROOT
from oracle.ref_loader import load_reference_module, reference_available


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "supcon_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(supcon_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib_built):
    from wav2vec_contr_loss_b200 import _cabi
    lib = ctypes.CDLL(lib_built)
    names = _declared_functions()
    assert len(names) >= 10
    for name in names:
        assert hasattr(lib, name), f"{name} declared in supcon_b200.h but not exported"
    assert sorted(_cabi.EXPORTS) == names
    assert _cabi.load().supcon_abi_version() == _cabi.ABI_VERSION == 3
    # diagnostics live in the test-only library, not in the product or its public header
    assert not any("debug" in n for n in names)
    for name in ("supcon_debug_plan", "supcon_debug_tc_tile", "supcon_debug_ffma_plan"):
        assert not hasattr(lib, name)
    import debug_lib
    for name in ("supcon_debug_plan", "supcon_debug_ffma_plan", "supcon_forward_rows"):
        assert hasattr(debug_lib.load(), name)


def test_flag_constants_match_the_header():
    """every SUPCON_FLAG_* of the public header that the Python binding names carries the header's value"""
    from wav2vec_contr_loss_b200 import _cabi
    text = open(os.path.join(ROOT, "include", "supcon_b200.h")).read()
    defines = {k: int(v) for k, v in re.findall(r"#define\s+SUPCON_FLAG_([A-Z_]+)\s+(\d+)u", text)}
    assert {"FORCE_EXACT", "FORCE_TENSOR", "NO_SMALL", "UNIT_ROWS", "PEER_EXCHANGE", "CLASS_SUMS", "NO_CLASS_SUMS",
            "WS_FROM_FORWARD"} <= set(defines)
    vals = sorted(defines.values())
    assert len(set(vals)) == len(vals) and all(v & (v - 1) == 0 for v in vals)       # distinct single bits
    for name, value in defines.items():
        if hasattr(_cabi, "FLAG_" + name):
            assert getattr(_cabi, "FLAG_" + name) == value, name
    for name in ("CLASS_SUMS", "NO_CLASS_SUMS", "WS_FROM_FORWARD", "UNIT_ROWS", "PEER_EXCHANGE"):
        assert hasattr(_cabi, "FLAG_" + name), name


def test_tensor_path_workspace_is_flag_independent(lib_built):
    """the workspace of a problem does not depend on the route flags (a forward's workspace may be handed to the
    backward of the same problem with SUPCON_FLAG_WS_FROM_FORWARD set)"""
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200.functional import make_problem, with_flags
    lib = _cabi.load()
    sizes = []
    base = make_problem(4096, 256, _cabi.BF16, tau=0.07, similarity=_cabi.COSINE, flags=_cabi.FLAG_UNIT_ROWS)
    for extra in (0, _cabi.FLAG_CLASS_SUMS, _cabi.FLAG_NO_CLASS_SUMS, _cabi.FLAG_WS_FROM_FORWARD):
        nbytes = ctypes.c_size_t(0)
        prob = with_flags(base, extra)
        assert prob.flags == base.flags | extra and prob.n_total == 4096
        assert lib.supcon_workspace_bytes(ctypes.byref(prob), ctypes.byref(nbytes)) == 0
        sizes.append(nbytes.value)
    assert len(set(sizes)) == 1 and sizes[0] > 4096 * 256 * 4     # holds at least one fp32 dz record


def test_argument_validation_without_gpu(lib_built):
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200.functional import make_problem
    lib = _cabi.load()
    nbytes = ctypes.c_size_t(0)
    ok = make_problem(64, 256, _cabi.F32, tau=0.07, similarity=_cabi.COSINE)
    assert lib.supcon_workspace_bytes(ctypes.byref(ok), ctypes.byref(nbytes)) == 0 and nbytes.value >= 256
    bad = make_problem(1, 256, _cabi.F32, tau=0.07, similarity=_cabi.COSINE)
    assert lib.supcon_workspace_bytes(ctypes.byref(bad), ctypes.byref(nbytes)) == -1
    assert b"n_total" in lib.supcon_last_error()
    bad = make_problem(8, 4, _cabi.F32, tau=0.07, similarity=7)
    assert lib.supcon_workspace_bytes(ctypes.byref(bad), ctypes.byref(nbytes)) == -1
    assert b"Unknown similarity" in lib.supcon_last_error()
    bad = make_problem(8, 4, _cabi.F32, tau=0.07, similarity=0, row_offset=4, n_rows=8)
    with pytest.raises(RuntimeError, match="row block"):
        _cabi.check(lib.supcon_workspace_bytes(ctypes.byref(bad), ctypes.byref(nbytes)), "ws")


def test_dropin_interface_matches_reference():
    from wav2vec_contr_loss_b200 import loss as mine
    m = mine.SupConBinaryLoss()
    assert (m.tau, m.similarity, m.lambda_uni, m.uni_t) == (0.2, "geodesic", 0.0, 2.0)
    assert list(m.parameters()) == [] and list(m.buffers()) == []
    m = mine.SupConBinaryLoss(temperature=0.07, similarity="COSINE", uniformity_weight=0.05, uniformity_t=3)
    assert (m.tau, m.similarity, m.lambda_uni, m.uni_t) == (0.07, "cosine", 0.05, 3.0)
    with pytest.raises(ValueError, match="Unknown similarity: euclid"):
        mine.SupConBinaryLoss(similarity="euclid")
    sig = inspect.signature(mine.SupConBinaryLoss.forward)
    assert list(sig.parameters) == ["self", "z", "labels", "topk_neg", "alpha"]
    assert sig.parameters["topk_neg"].default == 32 and sig.parameters["alpha"].default == 0.0
    assert mine.SupConMultiClassLoss().tau == 0.1
    if reference_available():
        ref = load_reference_module("loss")
        for cls in ("SupConBinaryLoss", "SupConMultiClassLoss", "BCEBinaryLoss"):
            a = inspect.signature(getattr(ref, cls).__init__)
            b = inspect.signature(getattr(mine, cls).__init__)
            assert [(p.name, p.default) for p in a.parameters.values()] == \
                   [(p.name, p.default) for p in b.parameters.values()]
            a = inspect.signature(getattr(ref, cls).forward)
            b = inspect.signature(getattr(mine, cls).forward)
            assert [(p.name, p.default) for p in a.parameters.values()] == \
                   [(p.name, p.default) for p in b.parameters.values()]


def test_degenerate_batches_and_cpu_rejection():
    from wav2vec_contr_loss_b200 import loss as mine
    m = mine.SupConBinaryLoss(0.07, "cosine", 0.3)
    out = m(torch.randn(1, 8), torch.tensor([1]))
    assert out.item() == 0.0 and out.requires_grad and out.is_leaf        # reference loss.py:138-139
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(4, 8), torch.tensor([0, 1, 0, 1]))
    with pytest.raises(AssertionError, match="labels must be shape"):
        mine.SupConMultiClassLoss()(torch.randn(4, 8), torch.zeros(4, 1))


def test_bce_passthrough_and_pos_weight():
    from wav2vec_contr_loss_b200 import loss as mine
    logits, y = torch.tensor([0.3, -1.2, 2.0, 0.1]), torch.tensor([1, 0, 1, 0])
    want = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor([2.5]))(logits, y.float())
    assert torch.allclose(mine.BCEBinaryLoss(2.5)(logits, y), want)
    assert torch.allclose(mine.BCEBinaryLoss()(logits, y), torch.nn.BCEWithLogitsLoss()(logits, y.float()))

    class DS:
        data = [("a", 1), ("b", 0), ("c", 0), ("d", 0)]
    assert mine.compute_pos_weight_from_dataset(DS) == 3.0
    DS.data = [("a", 1)]
    assert mine.compute_pos_weight_from_dataset(DS) == 1.0


def test_dropin_module_name_resolves():
    path = os.path.join(ROOT, "wav2vec_contr_loss_b200", "dropin")
    saved = sys.modules.pop("loss", None)
    sys.path.insert(0, path)
    try:
        import loss
        from wav2vec_contr_loss_b200.loss import SupConBinaryLoss
        assert loss.SupConBinaryLoss is SupConBinaryLoss
    finally:
        sys.path.remove(path)
        sys.modules.pop("loss", None)
        if saved is not None:
            sys.modules["loss"] = saved
