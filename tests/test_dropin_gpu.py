"""GPU side of the drop-in contract with the reference's caller (train.py:19-35,71-163).  The vectors were recorded
from the REAL `create_model` + `Lit.training_step` with the reference's own models and losses
(tests/golden/make_train_golden.py); here the recorded prediction goes through the caller protocol --
`loss_fn(prediction, y)`, `.log` assigned after construction (train.py:161), the loss logged as 'train_loss'
(train.py:34) -- into the CUDA loss classes, plain and wrapped in ShardedLoss.
tests/test_dropin_train_cpu.py replays the same vectors on any host."""
import os

import numpy as np
import pytest
import torch

import pointcloud_b200 as pcl
from helpers import CLASSES, LitProtocol, npy

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def tg():
    return np.load(os.path.join(ROOT, "tests", "golden", "train_golden.npz"))


def _loss(model_type):
    if model_type == "Autoencoder":
        return pcl.EarthMoverDistance(eps=pcl.cfg.emd_eps, its=pcl.cfg.emd_iterations, num_classes=None)      # train.py:82
    if model_type == "Segmenter":
        return pcl.EarthMoverDistance(eps=pcl.cfg.emd_eps, its=pcl.cfg.emd_iterations, num_classes=len(CLASSES))  # train.py:100
    return pcl.SegmentingChamferDistance({n: CLASSES.index(n) for n in ("cube", "arm", "gripper")})              # train.py:116-125


@pytest.mark.parametrize("sharded", [False, True])
@pytest.mark.parametrize("model_type", ["Autoencoder", "Segmenter", "MultiSegmenter"])
def test_reference_training_step_replayed_on_the_cuda_losses(tg, model_type, sharded):
    names = [k[len(model_type) + 6:] for k in tg.files if k.startswith(f"{model_type}_pred_")]
    preds = {n: torch.from_numpy(tg[f"{model_type}_pred_{n}"]).cuda().requires_grad_() for n in names}
    prediction = preds[""] if names == [""] else preds
    loss_fn = _loss(model_type)
    lit = LitProtocol(prediction, pcl.ShardedLoss(loss_fn) if sharded else loss_fn)
    lit.loss_fn.log = lit.log                                                    # train.py:161
    y = torch.from_numpy(tg[f"{model_type}_y"]).cuda()
    loss = lit.training_step((None, y), 0)
    loss.backward()
    assert float(loss) == pytest.approx(float(tg[f"{model_type}_loss"]), rel=1e-5)
    want = {k[len(model_type) + 5:].replace(".", "/"): float(tg[k]) for k in tg.files if k.startswith(f"{model_type}_log_")}
    assert set(lit.logged) == set(want)
    for k, v in want.items():
        assert lit.logged[k] == pytest.approx(v, rel=1e-5, abs=1e-9), k
    for n, p in preds.items():
        np.testing.assert_allclose(npy(p.grad), tg[f"{model_type}_grad_{n}"], rtol=1e-5, atol=1e-10)
