"""float64 torch restatement of estimate_pointcloud_local_coord_frames (pytorch3d 0.7.2 ops/points_normals.py and
ops/utils.py:get_point_covariances as recalled [3P-memory]) from a given neighbour index: knn_gather -> mean -> central
difference -> covariance -> torch.linalg.eigh -> disambiguation -> stack((n, cross(n, z), z)).  Autograd through it is the
gradient reference of pcl_frames_bwd.  TEST INFRASTRUCTURE ONLY."""
import torch


def knn_idx(points, K, lengths=None):
    """Brute-force self-kNN in float64 on the CPU: (B,P,K) int64, the point itself first.  Rows past a cloud's length and
    clouds of at most K points are 0 (what the frames ignore).  For the CPU tests; the GPU tests take pcl_knn_fwd's idx."""
    p = points.detach().double().cpu()
    b, n, _ = p.shape
    out = torch.zeros(b, n, K, dtype=torch.int64)
    for i in range(b):
        m = n if lengths is None else int(lengths[i])
        if m <= K:
            continue
        d = torch.cdist(p[i, :m], p[i, :m])
        out[i, :m] = torch.sort(d, dim=1, stable=True).indices[:, :K]
    return out


def _gather(p, idx):
    b, n, K = idx.shape
    return p.gather(1, idx.reshape(b, n * K, 1).expand(-1, -1, 3)).view(b, n, K, 3)


def _disambiguate(df, v, K):
    """pytorch3d's _disambiguate_vector_directions with the point itself as origin: flip v where fewer than half of the
    K projections v . (p_j - p_i) are positive."""
    n_pos = ((v[:, :, None] * df).sum(3) > 0).sum(2, keepdim=True)
    return torch.where(2 * n_pos < K, -v, v)


def frames_ref(points, idx, lengths=None, disambiguate=True):
    """points (B,P,3) (any float dtype, may require grad; up-cast to float64 like .float().double()), idx (B,P,K).
    Returns (curvatures (B,P,3), frames (B,P,3,3)) in float64; rows i >= n_b and clouds with n_b <= K are 0."""
    p = points.float().double() if points.dtype != torch.float64 else points
    b, n, _ = p.shape
    idx = idx.to(p.device).long()
    K = idx.shape[2]
    nb = _gather(p, idx)
    mu = nb.mean(2, keepdim=True)
    d = nb - mu
    cov = (d.unsqueeze(4) * d.unsqueeze(3)).mean(2)
    lens = torch.full((b,), n, dtype=torch.int64) if lengths is None else lengths.cpu().clamp(max=n)
    valid = (torch.arange(n)[None, :] < lens[:, None]) & (lens[:, None] > K)
    valid = valid.to(p.device)
    # rows that are not computed get a well-separated spectrum, so that eigh's backward stays finite there
    safe = torch.diag(torch.tensor([1.0, 2.0, 3.0], dtype=p.dtype, device=p.device))
    cov = torch.where(valid[..., None, None], cov, safe)
    lam, V = torch.linalg.eigh(cov)
    if disambiguate:
        df = nb - p[:, :, None]
        nrm = _disambiguate(df, V[..., 0], K)
        z = _disambiguate(df, V[..., 2], K)
        V = torch.stack((nrm, torch.cross(nrm, z, dim=2), z), dim=3)
    zero = torch.zeros((), dtype=p.dtype, device=p.device)
    return torch.where(valid[..., None], lam, zero), torch.where(valid[..., None, None], V, zero)
