"""CPU checks of tests/loss_reference.py: the torch restatement of normal_utils.py's losses reproduces the gradients
frozen from the executed reference, and the fp32 model of normal_loss_backward_kernel agrees with that restatement
over the whole edge matrix (norm sweep across both clamps and both overflow points, special values, degenerate
geometry, masks, upstream gradients).  Runs everywhere; the CUDA kernel itself is checked against the same
restatement in test_gpu_normal_utils_edges.py."""
import os

import numpy as np
import pytest

from tests import common as C
from tests import loss_reference as LR

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = LR.edge_cases()


def _go(case):
    m = LR.as_mask4(case["mask"]).numpy()
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.float32(LR.effective_up(case)) / np.float32(np.sum(m, dtype=np.float64))


@pytest.mark.parametrize("mode", LR.MODES)
def test_reference_reproduces_golden(mode):
    gold = np.load(os.path.join(GOLD, "golden_tiny_loss_backward.npz"))
    pred, gt, maskf, up = C.loss_inputs(3, 48, 64, seed=int(gold["seed"]))
    loss, angle, grad = LR.reference(mode, pred, gt, maskf, up)
    assert np.isclose(loss, gold[f"{mode}_loss"], rtol=2e-6, atol=0)
    assert np.isclose(angle, gold[f"{mode}_angle"], rtol=2e-6, atol=0)
    go = np.float32(up) / np.float32(maskf.sum(dtype=np.float64))
    bad = LR.grad_mismatches(mode, grad, gold[f"{mode}_grad"], pred, gt, maskf, go)
    assert not bad.any(), f"{mode}: {int(bad.sum())} gradient components off the frozen reference"
    assert np.array_equal(grad[:, 3], np.zeros_like(grad[:, 3]))
    km = LR.kernel_model(mode, pred, gt, maskf, up)
    assert not LR.grad_mismatches(mode, km, gold[f"{mode}_grad"], pred, gt, maskf, go).any()


def test_tolerance_rejects_a_dropped_term():
    """The term-scaled bar is tight enough to see a chain-rule term go missing: drop the radial term of the normalised
    L1 gradient at an ordinary pixel and the comparison must flag it."""
    pred, gt, m = LR._pixels(np.array([[0.3, -0.2, 0.5]], np.float32), np.array([[0.6, 0.8, 0.0]], np.float32))
    _, _, ref = LR.reference("l1", pred, gt, m, 1.0)
    go = np.float32(1.0) / np.float32(m.sum())
    r = pred[:, 0:3].astype(np.float64)
    direct = ref.astype(np.float64).copy()
    nr = np.sqrt((r * r).sum(1, keepdims=True))
    dn = go * np.sign(r / nr - gt) * m
    direct[:, 0:3] = dn / nr
    assert LR.grad_mismatches("l1", direct, ref, pred, gt, m, go)[0, :, 0, 0].any()


@pytest.mark.parametrize("mode", LR.MODES)
@pytest.mark.parametrize("name", sorted(CASES))
def test_kernel_model_matches_reference_on_edges(name, mode):
    case = CASES[name]
    _, _, ref = LR.reference(mode, case["pred"], case["gt"], case["mask"], case["up"], LR.outer_fn(case))
    km = LR.kernel_model(mode, case["pred"], case["gt"], case["mask"], LR.effective_up(case))
    bad = LR.grad_mismatches(mode, km, ref, case["pred"], case["gt"], case["mask"], _go(case))
    if bad.any():
        b, c, y, x = [int(v[0]) for v in np.nonzero(bad)]
        pytest.fail(f"{name}/{mode}: {int(bad.sum())} components off; first at (b={b}, c={c}, y={y}, x={x}): "
                    f"pred={case['pred'][b, :3, y, x]} model={km[b, c, y, x]} torch={ref[b, c, y, x]}")
    assert np.array_equal(km[:, 3:], ref[:, 3:])
