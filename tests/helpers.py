"""Shared helpers of the tests."""
import numpy as np
import torch


def ref_emd_forward(ref, xyz1, xyz2, eps, iters):
    """Call the UNMODIFIED reference extension exactly like emdFunction.forward does (emd_module.py:43-58)."""
    b, n, _ = xyz1.shape
    dev = 'cuda'
    xyz1, xyz2 = xyz1.contiguous().float().cuda(), xyz2.contiguous().float().cuda()
    dist = torch.zeros(b, n, device=dev)
    assignment = torch.zeros(b, n, device=dev, dtype=torch.int32) - 1
    assignment_inv = torch.zeros(b, n, device=dev, dtype=torch.int32) - 1
    price = torch.zeros(b, n, device=dev)
    bid = torch.zeros(b, n, device=dev, dtype=torch.int32)
    bid_increments = torch.zeros(b, n, device=dev)
    max_increments = torch.zeros(b, n, device=dev)
    unass_idx = torch.zeros(b * n, device=dev, dtype=torch.int32)
    max_idx = torch.zeros(b * n, device=dev, dtype=torch.int32)
    unass_cnt = torch.zeros(512, dtype=torch.int32, device=dev)
    unass_cnt_sum = torch.zeros(512, dtype=torch.int32, device=dev)
    cnt_tmp = torch.zeros(512, dtype=torch.int32, device=dev)
    ref.forward(xyz1, xyz2, dist, assignment, price, assignment_inv, bid, bid_increments, max_increments,
                unass_idx, unass_cnt, unass_cnt_sum, cnt_tmp, max_idx, eps, iters)
    return dist, assignment


def ref_emd_backward(ref, xyz1, xyz2, graddist, assignment):
    gradxyz1 = torch.zeros(xyz1.size(), device='cuda')
    ref.backward(xyz1.contiguous().float().cuda(), xyz2.contiguous().float().cuda(), gradxyz1, graddist.contiguous(), assignment)
    return gradxyz1


class RefEmdFunction(torch.autograd.Function):
    """Restatement of the reference's emdFunction (emd_module.py:33-72) around the UNMODIFIED extension `ref` (oracle/_ref/emd.so):
    forward = 12 zero-filled scratch tensors + emd.forward, backward = 2 zero fills + emd.backward; the target gets zeros.
    Test / bench infrastructure: the reference's own emd_module.py is not available on the GPU box."""

    @staticmethod
    def forward(ctx, ref, xyz1, xyz2, eps, iters):
        dist, assignment = ref_emd_forward(ref, xyz1, xyz2, eps, iters)
        ctx.ref = ref
        ctx.save_for_backward(xyz1.contiguous().float(), xyz2.contiguous().float(), assignment)
        ctx.mark_non_differentiable(assignment)
        return dist, assignment

    @staticmethod
    def backward(ctx, graddist, gradidx):
        xyz1, xyz2, assignment = ctx.saved_tensors
        graddist = graddist.contiguous()
        gradxyz1 = torch.zeros(xyz1.size(), device='cuda').contiguous()
        gradxyz2 = torch.zeros(xyz2.size(), device='cuda').contiguous()
        ctx.ref.backward(xyz1, xyz2, gradxyz1, graddist, assignment)
        return None, gradxyz1, gradxyz2, None, None


def npy(t):
    return t.detach().cpu().numpy()


def sqdist_to_match(x1, x2, asg):
    m = np.take_along_axis(np.asarray(x2), np.asarray(asg).astype(np.int64)[..., None], 1)
    return ((np.asarray(x1, dtype=np.float64) - m) ** 2).sum(-1)


CLASSES = ['env', 'cube', 'arm', 'base', 'gripper']           # robosuite_envs/envs.py:79 (scene 'Cube')


class LitProtocol(torch.nn.Module):
    """The four lines of Lit.training_step (train.py:30-35) around a model that returns the recorded prediction."""

    def __init__(self, prediction, loss_fn):
        super().__init__()
        self.prediction, self.loss_fn, self.logged = prediction, loss_fn, {}

    def log(self, name, value):
        self.logged[name] = float(value)

    def training_step(self, batch, batch_idx):
        x, y = batch
        prediction = self.prediction
        loss = self.loss_fn(prediction, y)
        self.log('train_loss', loss)
        return loss
