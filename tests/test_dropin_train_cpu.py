"""Drop-in test against the reference's OWN caller, `Lit.training_step` + `create_model` of pointcloud_vision/train.py
(train.py:19-35,71-163).  tests/golden/make_train_golden.py ran that caller unmodified, with the reference's real
PointNet2 / PointNet models and its own loss classes, and recorded per model type the batch, the model's prediction, the
loss, everything `.log` received and d loss / d prediction (tests/golden/train_golden.npz).  Here the recorded prediction
goes through the same caller protocol -- `loss_fn(prediction, y)`, `.log` assigned after construction (train.py:161), the
loss logged as 'train_loss' (train.py:34) -- into the loss classes of this package, constructed as train.py:82,100,125
constructs them.  Loss value, every logged scalar and d loss / d prediction must agree; every model parameter's gradient
is d loss / d prediction chained through the same model, so the training step is the reference's.

Without a CUDA device the three CUDA entry points of the product classes are served by the CPU oracle (the test-only
subclasses of test_sharded_cpu.py); tests/test_dropin_gpu.py replays the same vectors on the CUDA losses, plain and
wrapped in ShardedLoss."""
import inspect
import os

import numpy as np
import pytest
import torch

from helpers import CLASSES, LitProtocol
from pointcloud_b200 import cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# The module-level surface the reference's utils.py calls (INTEGRATION.md route 2): emdModule.forward and
# emdFunction.forward of pointcloud_vision/loss/emd/emd_module.py:74-79 and :33-61.
REF_EMD_MODULE_FORWARD = ["self", "input1", "input2", "eps", "iters"]
REF_EMD_FUNCTION_FORWARD = ["ctx", "xyz1", "xyz2", "eps", "iters"]


@pytest.fixture(scope="module")
def tg():
    return np.load(os.path.join(ROOT, "tests", "golden", "train_golden.npz"))


def _product_classes():
    """The product loss classes; on a host without CUDA their kernel entry points are served by the CPU oracle."""
    import pointcloud_b200 as pcl
    if torch.cuda.is_available():
        return pcl.EarthMoverDistance, pcl.SegmentingChamferDistance
    from test_sharded_cpu import CpuEMD, CpuSegmentingChamfer
    return CpuEMD, CpuSegmentingChamfer


def _batch(model_type, b, n):
    from pointcloud_b200 import synth
    if model_type == "Autoencoder":
        _, target = synth.autoencoder_batch(b, n, seed=41)        # x == y: xyz + rgb (train.py:87-94)
        return target.clone(), target
    _, target = synth.segmenter_batch(b, n, seed=42)              # y = xyz + label (train.py:105-112,128-135)
    x = torch.cat([target[:, :, :3], torch.rand(b, n, 3, generator=torch.Generator().manual_seed(1))], dim=2)
    return x, target


@pytest.mark.parametrize("model_type", [pytest.param("Autoencoder", id="Autoencoder-PointNet2"),  # id: + the reference model that
                                        pytest.param("Segmenter", id="Segmenter-PointNet"),        # made the recorded prediction
                                        pytest.param("MultiSegmenter", id="MultiSegmenter-PointNet")])
def test_training_step_of_the_reference_lit_with_the_new_losses(tg, model_type):
    emd_cls, msc_cls = _product_classes()
    if model_type == "MultiSegmenter":                                         # train.py:116-125
        loss_fn = msc_cls({n: CLASSES.index(n) for n in ("cube", "arm", "gripper")})
    else:                                                                      # train.py:82,100
        loss_fn = emd_cls(eps=cfg.emd_eps, its=cfg.emd_iterations, num_classes=None if model_type == "Autoencoder" else len(CLASSES))
        assert loss_fn.eps == 0.005 and loss_fn.iterations == 50 and loss_fn.C == (None if model_type == "Autoencoder" else 5)

    x, y = _batch(model_type, 2, 2048)
    np.testing.assert_array_equal(y.numpy(), tg[f"{model_type}_y"])            # the recorded batch is the one synth draws
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    names = [k[len(model_type) + 6:] for k in tg.files if k.startswith(f"{model_type}_pred_")]
    preds = {n: torch.from_numpy(tg[f"{model_type}_pred_{n}"]).to(dev).requires_grad_() for n in names}
    lit = LitProtocol(preds[""] if names == [""] else preds, loss_fn)
    lit.loss_fn.log = lit.log                                                  # train.py:161
    assert lit.loss_fn.log == lit.log
    loss = lit.training_step((x.to(dev), y.to(dev)), 0)                        # train.py:30-35
    assert loss.dim() == 0
    loss.backward()

    assert float(loss) == pytest.approx(float(tg[f"{model_type}_loss"]), rel=1e-5)
    want = {k[len(model_type) + 5:].replace(".", "/"): float(tg[k]) for k in tg.files if k.startswith(f"{model_type}_log_")}
    assert set(lit.logged) == set(want) and "train_loss" in want
    for k, v in want.items():
        assert lit.logged[k] == pytest.approx(v, rel=1e-5, abs=1e-9), k
    for n, p in preds.items():
        np.testing.assert_allclose(p.grad.cpu().numpy(), tg[f"{model_type}_grad_{n}"], rtol=1e-5, atol=1e-10, err_msg=n)


def test_module_level_route_names_resolve():
    """INTEGRATION.md route 2: utils.py stays, `emd_module` and `pytorch3d.loss` are re-exported from this package --
    the names and call surfaces the reference's utils.py uses must exist with the reference's signatures."""
    import pointcloud_b200.chamfer as new_p3d_loss
    import pointcloud_b200.emd_module as new_emd
    assert list(inspect.signature(new_emd.emdModule.forward).parameters) == REF_EMD_MODULE_FORWARD
    assert list(inspect.signature(new_emd.emdFunction.forward).parameters) == REF_EMD_FUNCTION_FORWARD
    sig = inspect.signature(new_p3d_loss.chamfer_distance)
    assert list(sig.parameters)[:4] == ["x", "y", "x_lengths", "y_lengths"]  # utils.py:211,228
    sig.bind("pred", "target")                                                 # ChamferDistance (utils.py:211)
    sig.bind("pred", "target", y_lengths="num_points")                         # FilteringChamferDistance (utils.py:228)
