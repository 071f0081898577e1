"""The agent-sharded symmetric MLAPM step (piml_mlapm_sym_pairs_push_f32, then piml_mlapm_sym_finalize_push_f32) with
every rank of a world on ONE device and stream: the pair stage of each rank (row blocks from I0 > 0 on all ranks but
the first, column stages split over several CTAs) stores its column-direction shares into the owners' inboxes, and each
owner's finalize kernel then pushes its rows' new state.  The assembled step against the dense whole-crowd symmetric
step (algorithm 3).  The two differ only in fp32 summation grouping (row splits, per-rank shares)."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 1e-5
KW = dict(tau=0.5, A=7.55, B=-3.00, C=0.2, D=-0.3, theta=56)
DT, RADIUS = 0.08, 0.3


def _crowd(N, seed):
    rng = np.random.default_rng(seed)
    L = np.sqrt(N / 0.5)
    p = (rng.random((N, 2)) * L).astype(np.float32)
    d = (rng.random((N, 2)) * L).astype(np.float32)
    v = rng.normal(0, 1, (N, 2)).astype(np.float32)
    v[rng.random(N) < 0.05] = 0.0                                       # stationary: view gate false
    near = rng.random(N) < 0.1                                          # these arrive within the step
    d[near] = p[near] + DT * v[near] + rng.normal(0, 0.05, (near.sum(), 2)).astype(np.float32)
    ds = (1.34 + 0.3 * rng.normal(0, 1, (N, 1))).astype(np.float32)
    return [torch.from_numpy(x).cuda() for x in (p, v, ds, d)]


def _sharded_step(model, p, v, ds, d, world):
    """Every rank's pair stage, then every rank's finalize; returns the assembled (action, new position, arrived)."""
    from piml_b200 import _lib as L
    lib, N, prm, st = L.load(), p.shape[0], model._params(), L.stream_ptr(p.device)
    inbox_floats = int(lib.piml_mlapm_sym_inbox_bytes(N, world)) // 4
    ws_bytes = int(lib.piml_mlapm_sym_shard_workspace_bytes(N, world))
    assert inbox_floats > 0 and ws_bytes > 0
    inbox = [torch.full((inbox_floats,), float("nan"), device=p.device) for _ in range(world)]
    ws = [torch.empty(ws_bytes, dtype=torch.uint8, device=p.device) for _ in range(world)]
    inbox_tab = (C.c_uint64 * world)(*[x.data_ptr() for x in inbox])
    pos_next = torch.full((N, 2), float("nan"), device=p.device)
    vel_next = torch.full((N, 2), float("nan"), device=p.device)
    pos_tab = (C.c_uint64 * world)(*[pos_next.data_ptr()] * world)
    vel_tab = (C.c_uint64 * world)(*[vel_next.data_ptr()] * world)
    rows = []
    for rank in range(world):
        r0, r1 = C.c_int64(), C.c_int64()
        L.check(lib.piml_mlapm_sym_shard_rows(N, world, rank, C.byref(r0), C.byref(r1)), "piml_mlapm_sym_shard_rows")
        rows.append((int(r0.value), int(r1.value)))
    assert rows[0][0] == 0 and rows[-1][1] == N and all(rows[g][1] == rows[g + 1][0] for g in range(world - 1))
    for rank in range(world):
        L.check(lib.piml_mlapm_sym_pairs_push_f32(L.ptr(p), L.ptr(v), L.ptr(d), N, world, rank, C.byref(prm),
                                                  inbox_tab, L.ptr(ws[rank]), ws_bytes, st),
                "piml_mlapm_sym_pairs_push_f32")
    arrived = [torch.full((r1 - r0,), 7, dtype=torch.uint8, device=p.device) for r0, r1 in rows]
    for rank in range(world):
        L.check(lib.piml_mlapm_sym_finalize_push_f32(L.ptr(p), L.ptr(v), L.ptr(ds), ds.shape[1], L.ptr(d), N, world,
                                                     rank, C.byref(prm), DT, RADIUS, L.ptr(inbox[rank]), pos_tab,
                                                     vel_tab, L.ptr(arrived[rank]), L.ptr(ws[rank]), ws_bytes, st),
                "piml_mlapm_sym_finalize_push_f32")
    torch.cuda.synchronize()
    return vel_next.cpu().numpy(), pos_next.cpu().numpy(), torch.cat(arrived).cpu().numpy()


def _dense_step(model, p, v, ds, d):
    from piml_b200 import _lib as L
    L.check(L.load().piml_set_mlapm_algorithm(3), "piml_set_mlapm_algorithm")
    try:
        a, q, arr = model.advance(p, v, ds, d, DT, RADIUS)
    finally:
        L.check(L.load().piml_set_mlapm_algorithm(0), "piml_set_mlapm_algorithm")
    return a.cpu().numpy(), q.cpu().numpy(), arr.cpu().numpy()


def _err(got, ref, operand):
    """Operand-scaled gate of test_mlapm_symmetric_evaluation: |got - ref| / max(|ref|, |operand|)."""
    num = np.linalg.norm(np.asarray(got, np.float64) - ref, axis=-1)
    den = np.maximum(np.maximum(np.linalg.norm(ref, axis=-1), np.linalg.norm(operand, axis=-1)), 1e-6)
    return float((num / den).max())


@pytest.mark.parametrize("ver", ["GC", "raw"])
@pytest.mark.parametrize("N", [5200, 8192, 20000])          # 11, 16 and 40 blocks of 512: odd / even, padded tails
def test_sharded_symmetric_step_matches_dense(N, ver):
    import piml_b200 as P
    model = P.MLAPM(version=ver, **KW)
    p, v, ds, d = _crowd(N, seed=3 * N + len(ver))
    act_ref, pos_ref, arr_ref = _dense_step(model, p, v, ds, d)
    assert np.isfinite(act_ref).all() and arr_ref.any() and not arr_ref.all()
    vn, pn = v.cpu().numpy(), p.cpu().numpy()
    for world in (2, 3, 8):
        act, pos, arr = _sharded_step(model, p, v, ds, d, world)
        assert np.isfinite(act).all() and np.isfinite(pos).all(), world
        assert _err(act, act_ref, vn) < TOL, world
        assert _err(pos, pos_ref, pn) < TOL, world
        assert np.isin(arr, (0, 1)).all() and np.array_equal(arr.astype(bool), arr_ref), world
