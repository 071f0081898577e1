"""Plain PyTorch fp32 restatements used as the reference for the floating-point backward kernels (test
infrastructure only; never imported by piml_b200/).  Each function follows the reference lines cited; the CPU suite
pins them against tests/golden/training_step.npz, which was produced by the unmodified reference modules.
"""
import torch
import torch.nn.functional as F


def _relu(x, name):
    return torch.relu(x)


def _mlp(sd, prefix, x, n, last_act=False, relu=_relu):
    """MLP (reference src/models/model.py:40-65): Linear + ReLU ..., Identity after the last layer.  relu(x, name) gets
    the pre-activation of Linear `name` (its state_dict prefix)."""
    for l in range(n):
        x = F.linear(x, sd[f"{prefix}.mlp.{2 * l}.weight"], sd[f"{prefix}.mlp.{2 * l}.bias"])
        if l < n - 1 or last_act:
            x = relu(x, f"{prefix}.mlp.{2 * l}")
    return x


def _count(sd, prefix):
    n = 0
    while f"{prefix}.mlp.{2 * n}.weight" in sd:
        n += 1
    return n


def pinnsf_forward_ref(sd, kind, tau, ped, obs, slf, has_obs=True, drop_ped=None, drop_obs=None, single_block=False,
                       relu=_relu):
    """PINNSF_bottleneck_multitask.forward (model.py:1185-1221, kind='pinnsf_bm'), PINNSF_multitask.forward
    (:1271-1305, 'pinnsf_m'), PINNSF_bottleneck (:1104-1135), PINNSF (:762-792), with processor_hidden_layers > 1 so
    that ResDNN(x) = dropout(2x) (model.py:115-119, SURVEY.md B-4).  sd: dict of parameter tensors.  Every ReLU goes
    through relu(pre_activation, name of its Linear)."""
    per_slot = kind in ("pinnsf_bm", "pinnsf_bottleneck")

    def mlp(prefix, x, n):
        return _mlp(sd, prefix, x, n, relu=relu)

    def branch(name, x, drop):
        e = mlp(f"{name}_encoder", x, _count(sd, f"{name}_encoder"))
        if single_block:      # ResDNN with one block: relu(W e + b) + e  (model.py:68-79, :115-119)
            key = f"{name}_processor.resnet.0.lin.mlp.0"
            e = relu(F.linear(e, sd[key + ".weight"], sd[key + ".bias"]), key) + e
        else:
            e = 2 * e
        if drop is not None:
            e = e * drop
        if per_slot:
            d = mlp(f"{name}_decoder", e, _count(sd, f"{name}_decoder"))
            msg = mlp(f"{name}_predictor", d, 1)
            return msg.sum(-2), msg, d
        d = mlp(f"{name}_decoder", e.sum(-2), _count(sd, f"{name}_decoder"))
        return mlp(f"{name}_predictor", d, 1), e, e

    acc, pmsg, phead = branch("ped", ped, drop_ped)
    out = [None, pmsg]
    if has_obs:
        acc_o, omsg, _ = branch("obs", obs, drop_obs)
        acc = acc + acc_o
        out.append(omsg)
    n = torch.norm(slf[..., :2], p=2, dim=1, keepdim=True)          # dim=1: the (C,N,7) quirk (SURVEY.md B-3)
    n_ = n.clone()
    n_[n_ == 0] = n_[n_ == 0] + 0.1
    out[0] = acc + (slf[..., -1:] * (slf[..., :2] / n_) - slf[..., 2:4]) / tau
    if kind in ("pinnsf_bm", "pinnsf_m"):
        c = mlp("ped_collision_predictor", phead, _count(sd, "ped_collision_predictor"))
        out.append(torch.sigmoid(c).squeeze())
    return out


def gathered_features_ref(pos, vel, acc, dest, obstacles, ped_idx, obs_idx):
    """Differentiable restatement of what get_relative_features returns (src/data/data.py:466-512) GIVEN the selection:
    ped_f[n,j] = (p_m - p_n, v_m - v_n, a_m - a_n) for m = ped_idx[n,j] >= 0 else 0; obs_f[n,j] = (o - p_n, -v_n, -a_n);
    dest_f = dest - p with NaN -> 0.  pos.. (B,N,2); ped_idx (B,N,kp); obs_idx (B,N,ko); obstacles (M,2)."""
    B, N, _ = pos.shape
    state = torch.cat([pos, vel, acc], -1)                           # (B,N,6)
    kp = ped_idx.shape[-1]
    valid = (ped_idx >= 0)
    gi = ped_idx.clamp_min(0).reshape(B, N * kp, 1).expand(B, N * kp, 6)
    nb = torch.gather(state, 1, gi).reshape(B, N, kp, 6)
    ped_f = torch.where(valid.unsqueeze(-1), nb - state.unsqueeze(2), torch.zeros_like(nb))
    ko = obs_idx.shape[-1]
    if ko:
        ovalid = obs_idx >= 0
        o = obstacles[obs_idx.clamp_min(0)]                          # (B,N,ko,2)
        of = torch.cat([o - pos.unsqueeze(2), (-vel).unsqueeze(2).expand(B, N, ko, 2),
                        (-acc).unsqueeze(2).expand(B, N, ko, 2)], -1)
        obs_f = torch.where(ovalid.unsqueeze(-1), of, torch.zeros_like(of))
    else:
        obs_f = torch.zeros(B, N, 0, 6)
    d = dest - pos
    dest_f = torch.where(d.isnan(), torch.zeros_like(d), d)
    return ped_f, obs_f, dest_f


def collision_detection_ref(position, threshold, real_position=None):
    """Pedestrians.collision_detection (src/data/data.py:538-601), loop-free restatement."""
    def touch(p):
        rel = p.unsqueeze(-3) - p.unsqueeze(-2)
        d = torch.norm(rel, p=2, dim=-1)
        return torch.where(d.isnan(), torch.zeros_like(d), (d < threshold).float())
    coll = touch(position)
    eye = torch.eye(position.shape[-2])
    valid_diag = (~position[..., 0].isnan()).float()
    coll = coll - eye * valid_diag.unsqueeze(-1)                     # (1 - 1) on the diagonal of present agents
    if real_position is not None:
        friends = (touch(real_position).sum(0) <= 25).float().unsqueeze(0)
    elif position.dim() == 3:
        friends = (coll.sum(0) <= 25).float().unsqueeze(0)
    else:
        friends = (1 - (coll[:, :4].sum(1) > 0).float()).unsqueeze(1)
    return coll * friends


# ---- rollout losses (reference src/models/simulators.py:169-249), plain torch ------------------------------------------
def _reduce(x, mode):
    return {"sum": torch.sum, "mean": torch.mean, "none": lambda t: t}[mode](x)


def l1_reg_loss(embeddings, weight=1e-3, mode='none'):
    """simulators.py:169-170."""
    return _reduce(weight * embeddings.abs(), mode)


def multiple_rollout_mse_loss(pred, labels, time_decay, mode='none', reverse=False):
    """simulators.py:172-195: squared error of (C,T,N,2) tensors weighted by time_decay^(T-1-t) (time_decay^t if
    `reverse`)."""
    T = pred.shape[1]
    powers = [t if reverse else T - 1 - t for t in range(T)]
    w = torch.tensor([time_decay ** k for k in powers], device=pred.device).reshape(1, T, 1, 1)
    return _reduce((pred - labels) ** 2 * w, mode)


def _perpendicular(x, n):
    return x - (x * n).sum(-1, keepdim=True) * n


def multiple_rollout_collision_avoidance_loss(pred, labels, time_decay, mode='none'):
    """simulators.py:230-249: the MSE of the components perpendicular to the label's first-to-last displacement."""
    n = labels[:, -1:] - labels[:, :1]
    n = n / (n.norm(p=2, dim=-1, keepdim=True) + 1e-6)
    return _reduce(multiple_rollout_mse_loss(_perpendicular(pred, n), _perpendicular(labels, n), time_decay), mode)


def multiple_rollout_collision_loss(pred, labels, time_decay, coll_focus_weight, collisions, mode='none',
                                    abnormal_mask=None):
    """simulators.py:197-228: the avoidance loss of every pedestrian that collided at any step of its channel
    (`collisions` (C,T,N) summed over T and binarised), optionally masked per pedestrian."""
    hit = (collisions.sum(dim=1) > 0).to(pred.dtype)                       # (C,N)
    loss = hit[:, None, :, None] * multiple_rollout_collision_avoidance_loss(pred, labels, time_decay)
    if abnormal_mask is not None:
        loss = loss * abnormal_mask.reshape(1, 1, -1, 1)
    return _reduce(loss, mode)
