"""Shared helpers for the parity tests."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def reference_available():
    """True where the upstream PIML source tree is reachable (PIML_REFERENCE, or the copy __graft_entry__.build()
    stages in baseline/_ref/).  The tests that import it live skip elsewhere.  The golden vectors hold its outputs
    on a fixed subset of their inputs only (test_oracle_golden, test_gpu_parity, test_gpu_training compare against
    those); the live tests' further inputs and the drop-in runs of its own code are checked only where it is present."""
    import sys
    if GOLDEN not in sys.path:
        sys.path.insert(0, GOLDEN)
    import _refharness
    return _refharness.available()


def group(z, prefix):
    """All arrays of an npz whose key starts with `prefix/`, keyed by the remainder."""
    pre = prefix + "/"
    return {k[len(pre):]: z[k] for k in z.files if k.startswith(pre)}


def rel_vec_err(x, ref, floor=1e-6):
    """SURVEY.md 8d gate: per-vector ||dx||_2 / max(||ref||_2, floor), max over vectors (NaN pattern must match)."""
    x, ref = np.asarray(x, np.float64), np.asarray(ref, np.float64)
    assert x.shape == ref.shape, (x.shape, ref.shape)
    nx, nr = np.isnan(x), np.isnan(ref)
    assert np.array_equal(nx, nr), "NaN pattern differs"
    x, ref = np.where(nx, 0.0, x), np.where(nr, 0.0, ref)
    num = np.sqrt(((x - ref) ** 2).sum(-1))
    den = np.maximum(np.sqrt((ref ** 2).sum(-1)), floor)
    return float((num / den).max()) if num.size else 0.0


def valid_sets(idx, dist, thr):
    """Per row: the set of (index, distance bits) with distance <= thr -- the bit-exact parity object (SURVEY 8d)."""
    idx, dist = np.asarray(idx), np.asarray(dist, np.float32)
    flat_i = idx.reshape(-1, idx.shape[-1])
    flat_d = dist.reshape(-1, dist.shape[-1])
    out = []
    for r in range(flat_i.shape[0]):
        ok = flat_d[r] <= thr
        out.append(sorted(zip(flat_i[r][ok].tolist(), flat_d[r][ok].view(np.uint32).tolist())))
    return out


def untied_finite(dist):
    """Mask of slots whose distance is finite and differs from both neighbours in its row: torch.sort is not
    stable, so the index order of exactly equal distances (and of inf slots) is unspecified in the reference."""
    d = np.asarray(dist, np.float32)
    ok = np.isfinite(d)
    ok[..., 1:] &= d[..., 1:] != d[..., :-1]
    ok[..., :-1] &= d[..., :-1] != d[..., 1:]
    return ok


def accel_err(got, ref, self_f, tau):
    """Error of a predicted acceleration relative to the magnitude of what is being summed: the network output is
    sum(messages) + (v0*e - v)/tau (model.py:1205-1212); when those cancel, fp32 rounding (in the reference's own
    MKL GEMMs as much as anywhere) is relative to the operands, not to the small result.  Per agent:
    ||got - ref|| / max(||ref||, ||dest term||, 1e-3); returns the max."""
    got, ref, self_f = np.asarray(got, np.float64), np.asarray(ref, np.float64), np.asarray(self_f, np.float64)
    n = np.linalg.norm(self_f[:, :2], axis=-1, keepdims=True)
    n = np.where(n == 0, 0.1, n)
    dterm = (self_f[:, 6:7] * self_f[:, :2] / n - self_f[:, 2:4]) / tau
    scale = np.maximum(np.maximum(np.linalg.norm(ref, axis=-1), np.linalg.norm(dterm, axis=-1)), 1e-3)
    return float((np.linalg.norm(got - ref, axis=-1) / scale).max())


def dense_tile_count(n, kp, ko):
    """128-row tiles of the tensor-core forward's dense mode for n agents with kp / ko slots (128 // k agents a tile
    and branch; ko = 0: no obstacle branch).  The library runs the compact mode only when this exceeds the SM count."""
    return -(-n // (128 // kp)) + (-(-n // (128 // ko)) if ko else 0)


def tc_forward_in_dense_chunks(spec, packed, packed_tc, ped, obs, slf, sms):
    """The tensor-core forward's acceleration without messages, evaluated in chunks of agents whose dense tiles fit
    one wave of `sms` CTAs, so that every chunk runs in the dense mode.  Channelled (C,N,.) inputs are split by whole
    channels, which keeps each channel's destination norm.  Returns the acceleration and each chunk's launch count."""
    import torch
    from piml_b200 import _lib as L, models as M
    kp, ko = ped.shape[-2], (obs.shape[-2] if spec.has_obs else 0)
    if slf.dim() == 3:
        step = max(c for c in range(1, slf.shape[0] + 1) if dense_tile_count(c * slf.shape[1], kp, ko) <= sms)
    else:
        per_tile = [128 // kp] + ([128 // ko] if ko else [])
        step = sms // len(per_tile) * min(per_tile)
    accs, launches = [], []
    for i in range(0, slf.shape[0], step):
        l0 = L.launch_count()
        accs.append(M.pinnsf_forward(spec, packed, ped[i:i + step], obs[i:i + step], slf[i:i + step], need_msgs=False,
                                     packed_tc=packed_tc)[0])
        launches.append(L.launch_count() - l0)
    return torch.cat(accs), launches
