"""Drop-in for the reference's `MLAPM` (src/models/mlapm.py:5-58) on the CUDA all-pairs kernel."""
import torch

from . import _lib as L

_VERSIONS = {"raw": 0, "GC": 1}


class MLAPM:
    """Same constructor kwargs and `step` signature as reference models/mlapm.py.

    Extra (optional) kwarg `exact_math=True` selects the IEEE div/sqrt/expf validation variant of the pair kernel.
    """

    def __init__(self, **args):
        self.args = args
        self._ws = None

    def _params(self):
        a = self.args
        ver = a['version']
        if ver not in _VERSIONS:
            # 'UCY' raises a RuntimeError in the reference itself for any N != 2 (SURVEY.md Appendix B-15)
            raise NotImplementedError(f"MLAPM version {ver!r}")
        return L.MlapmParams(_VERSIONS[ver], float(a['tau']), float(a['A']), float(a['B']), float(a.get('C', 0.0)),
                             float(a.get('D', 0.0)), float(a.get('theta', 0.0)), 1 if a.get('exact_math') else 0)

    def _workspace(self, N, device, whole_crowd=False):
        """Caller-owned scratch of the kernels, the largest any path needs: ordered pairs 16 B per agent and split;
        symmetric dense 32 B records + 16 B row partials per split + 32 B fixed-point accumulators per agent; symmetric
        culled the same without the row partials, plus the spatial sort and the work list (0.1 GB at N = 10^6)."""
        lib = L.load()
        need = int(lib.piml_mlapm_workspace_bytes(N))
        if whole_crowd and not self.args.get('exact_math'):
            need = max(need, int(lib.piml_mlapm_workspace_bytes_sym(N)))
        if self._ws is None or self._ws.numel() < need or self._ws.device != device:
            self._ws = torch.empty(need, dtype=torch.uint8, device=device)
        return self._ws

    @staticmethod
    def _prep(position, velocity, desired_speed, destination):
        dev, origin, (position, velocity, desired_speed, destination) = L.stage(position, velocity, desired_speed,
                                                                                 destination)
        pos, vel, dest = L.f32c(position), L.f32c(velocity), L.f32c(destination)
        ds = L.f32c(desired_speed)
        if ds.dim() == 1:
            ds = ds.unsqueeze(-1)
        if pos.dim() != 2 or pos.shape[-1] != 2 or vel.shape != pos.shape or dest.shape != pos.shape:
            raise ValueError("MLAPM.step expects position, velocity, destination of shape [N, 2]")
        if ds.shape[0] != pos.shape[0] or ds.shape[1] not in (1, 2):
            raise ValueError("MLAPM.step expects desired_speed of shape [N, 1] or [N, 2]")
        return dev, origin, pos, vel, ds, dest

    def step(self, position, velocity, desired_speed, destination, dt, radius=0.3, rows=None):
        """position, velocity, destination [N,2]; desired_speed [N,1] or [N,2].  Returns velocity + force*dt.
        rows=(r0, r1): only those rows (agent-sharded ranks), output shape [r1-r0, 2]."""
        dev, origin, pos, vel, ds, dest = self._prep(position, velocity, desired_speed, destination)
        N = pos.shape[0]
        r0, r1 = rows if rows is not None else (0, N)
        action = torch.empty(r1 - r0, 2, dtype=torch.float32, device=dev)
        prm = self._params()
        ws = self._workspace(N, dev, whole_crowd=(r0 == 0 and r1 == N))
        L.check(L.load().piml_mlapm_advance_ws_f32(L.ptr(pos), L.ptr(vel), L.ptr(ds), ds.shape[1], L.ptr(dest), N, r0,
                                                   r1, L.C.byref(prm), float(dt), 0.0, L.ptr(action), None, None,
                                                   L.ptr(ws), ws.numel(), L.stream_ptr(dev)),
                "piml_mlapm_advance_ws_f32")
        return action if origin == dev else action.to(origin)

    def advance(self, position, velocity, desired_speed, destination, dt, radius=0.3, rows=None):
        """Fused main_mlapm.py:19-34 body: returns (action, new_position, arrived[bool])."""
        dev, origin, pos, vel, ds, dest = self._prep(position, velocity, desired_speed, destination)
        N = pos.shape[0]
        r0, r1 = rows if rows is not None else (0, N)
        action = torch.empty(r1 - r0, 2, dtype=torch.float32, device=dev)
        pnew = torch.empty(r1 - r0, 2, dtype=torch.float32, device=dev)
        arrived = torch.empty(r1 - r0, dtype=torch.uint8, device=dev)
        prm = self._params()
        ws = self._workspace(N, dev, whole_crowd=(r0 == 0 and r1 == N))
        L.check(L.load().piml_mlapm_advance_ws_f32(L.ptr(pos), L.ptr(vel), L.ptr(ds), ds.shape[1], L.ptr(dest), N, r0,
                                                   r1, L.C.byref(prm), float(dt), float(radius), L.ptr(action),
                                                   L.ptr(pnew), L.ptr(arrived), L.ptr(ws), ws.numel(),
                                                   L.stream_ptr(dev)), "piml_mlapm_advance_ws_f32")
        if origin != dev:
            return action.to(origin), pnew.to(origin), arrived.bool().to(origin)
        return action, pnew, arrived.bool()

    def advance_scenes(self, position, velocity, desired_speed, destination, active, dt, radius=0.3, params=None):
        """`advance` for S independent scenes in one launch.  position, velocity, destination [S,N,2]; desired_speed
        [S,N], [S,N,1] or [S,N,2]; active [S,N] bool (the agents of each scene); params None (the constructor's
        constants) or [S,6] = tau, A, B, C, D, theta (degrees) per scene.  Each scene's result is `advance` on its
        active agents alone; inactive slots give action = pos_new = NaN and arrived = False.
        Returns (action [S,N,2], new_position [S,N,2], arrived [S,N] bool)."""
        shape = tuple(position.shape)
        if len(shape) != 3 or shape[-1] != 2 or tuple(velocity.shape) != shape or tuple(destination.shape) != shape:
            raise ValueError("MLAPM.advance_scenes expects position, velocity, destination of shape [S, N, 2]")
        S, N = shape[0], shape[1]
        ds_shape = tuple(desired_speed.shape)
        if ds_shape != (S, N) and ds_shape not in ((S, N, 1), (S, N, 2)):
            raise ValueError("MLAPM.advance_scenes expects desired_speed of shape [S, N], [S, N, 1] or [S, N, 2]")
        if not isinstance(active, torch.Tensor) or active.dtype != torch.bool or tuple(active.shape) != (S, N):
            raise ValueError("MLAPM.advance_scenes expects active as a bool tensor of shape [S, N]")
        if params is not None and (not isinstance(params, torch.Tensor) or tuple(params.shape) != (S, 6)):
            raise ValueError("MLAPM.advance_scenes expects params None or of shape [S, 6] (tau, A, B, C, D, theta)")
        prm = self._params()
        dev, origin, (position, velocity, desired_speed, destination, active, params) = L.stage(
            position, velocity, desired_speed, destination, active, params)
        pos, vel, dest = L.f32c(position), L.f32c(velocity), L.f32c(destination)
        ds = L.f32c(desired_speed)
        if ds.dim() == 2:
            ds = ds.unsqueeze(-1)
        act = active.contiguous().view(torch.uint8)
        sp = None if params is None else L.f32c(params)
        action = torch.empty(S, N, 2, dtype=torch.float32, device=dev)
        pnew = torch.empty(S, N, 2, dtype=torch.float32, device=dev)
        arrived = torch.empty(S, N, dtype=torch.uint8, device=dev)
        L.check(L.load().piml_mlapm_scenes_advance_f32(L.ptr(pos), L.ptr(vel), L.ptr(ds), ds.shape[2], L.ptr(dest),
                                                       L.ptr(act), S, N, L.C.byref(prm), L.ptr(sp), float(dt),
                                                       float(radius), L.ptr(action), L.ptr(pnew), L.ptr(arrived),
                                                       L.stream_ptr(dev)), "piml_mlapm_scenes_advance_f32")
        arrived = arrived.view(torch.bool)
        if origin != dev:
            return action.to(origin), pnew.to(origin), arrived.to(origin)
        return action, pnew, arrived


def rollout(model, position, velocity, desired_speed, destination, steps=200, dt=0.08, radius=0.3):
    """The loop of reference src/main_mlapm.py:18-36 (without the plot).  position/velocity [N,2] initial state.
    Returns (position [N,steps+1,2], velocity [N,steps+1,2], mask [N,steps+1]) with NaN after arrival.  Like the
    reference (whose `mask.any()` looks at ALL time steps and therefore never breaks early) the arrays always span
    the full `steps`; once nobody is active the remaining columns stay NaN / False."""
    dev, origin, (position, velocity, desired_speed, destination) = L.stage(position, velocity, desired_speed,
                                                                             destination)
    N = position.shape[0]
    pos = torch.full((N, steps + 1, 2), float('nan'), device=dev)
    vel = torch.full((N, steps + 1, 2), float('nan'), device=dev)
    mask = torch.zeros(N, steps + 1, dtype=torch.bool, device=dev)
    pos[:, 0], vel[:, 0], mask[:, 0] = position, velocity, True
    for i in range(steps):
        idx = mask[:, i].nonzero(as_tuple=True)[0]             # boolean-mask compaction, main_mlapm.py:20-23
        v, p, arrived = model.advance(pos[idx, i], vel[idx, i], desired_speed[idx], destination[idx], dt, radius)
        pos[idx, i + 1] = p
        vel[idx, i + 1] = v
        mask[idx, i + 1] = ~arrived                            # main_mlapm.py:34
        if not bool(mask[:, i + 1].any()):                     # nothing left to simulate
            break
    return pos.to(origin), vel.to(origin), mask.to(origin)


def rollout_scenes(model, position, velocity, desired_speed, destination, steps=200, dt=0.08, radius=0.3, active=None,
                   params=None):
    """`rollout` for S independent scenes at once (MLAPM.advance_scenes per step).  position, velocity, destination
    [S,N,2]; desired_speed [S,N], [S,N,1] or [S,N,2]; active [S,N] bool, the agents of each scene (default: every
    slot); params as in advance_scenes.  Returns (position [S,N,steps+1,2], velocity [S,N,steps+1,2],
    mask [S,N,steps+1]) with NaN where a slot is not active.  Always runs `steps` steps and never waits for the host:
    the arrivals are removed on the device (active &= ~arrived), so a step can be captured in a CUDA graph."""
    dev, origin, (position, velocity, desired_speed, destination, active, params) = L.stage(
        position, velocity, desired_speed, destination, active, params)
    S, N = position.shape[0], position.shape[1]
    act = torch.ones(S, N, dtype=torch.bool, device=dev) if active is None else active.clone()
    pos = torch.full((S, N, steps + 1, 2), float('nan'), device=dev)
    vel = torch.full((S, N, steps + 1, 2), float('nan'), device=dev)
    mask = torch.zeros(S, N, steps + 1, dtype=torch.bool, device=dev)
    keep = act.unsqueeze(-1)
    p = torch.where(keep, position.float(), float('nan'))
    v = torch.where(keep, velocity.float(), float('nan'))
    pos[:, :, 0], vel[:, :, 0], mask[:, :, 0] = p, v, act
    for i in range(steps):
        v, p, arrived = model.advance_scenes(p, v, desired_speed, destination, act, dt, radius, params)
        pos[:, :, i + 1] = p
        vel[:, :, i + 1] = v
        act = act & ~arrived                                   # main_mlapm.py:34, per scene
        mask[:, :, i + 1] = act
    return pos.to(origin), vel.to(origin), mask.to(origin)
