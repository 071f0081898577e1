"""Inference rollout on the CUDA path: drop-in for `BaseSimulator.get_multiple_rollouts`
(reference src/models/simulators.py:556-657) and a scene-batched variant (SURVEY.md config 5b).

Per step the reference runs ~150 eager ops, 2N Python iterations and several host syncs; here a step is three
kernels with no host sync: fused network forward, fused integrate (record / Euler / arrival / entry), fused feature
rebuild (which also assembles self_features).
"""
import torch

from . import _lib as L
from .features import cos_threshold
from . import models as M
from .sfm import SfmSpec, SocialForce


def integrate_step(p, v, a, a_next, dest, dest_idx, dest_num, waypoints, dt, remove_on_arrival=True, entry=None,
                   p_gt=None, v_gt=None, a_gt=None, dest_gt=None, dest_idx_gt=None, hist_v=None, rec_p=None,
                   rec_v=None, rec_a=None, rec_mask=None):
    """simulators.py:596-639 in place on p, v, a, dest, dest_idx.  Tensors are (N,..) for one scene or (S,N,..);
    waypoints (D,N,2) or (S,D,N,2); dest_num (N) or (S,N)."""
    dev = L.require_cuda(p, v, a, a_next, dest, dest_idx, dest_num, waypoints)
    for t in (p, v, a, dest, dest_idx):
        if not t.is_contiguous():
            raise ValueError("integrate_step updates its state tensors in place; they must be contiguous")
    S = p.shape[0] if p.dim() == 3 else 1
    N = p.shape[-2]
    D = waypoints.shape[-3]
    if dest_num.numel() != S * N:
        dest_num = dest_num.expand(S, N)
    args = [L.f32c(a_next), L.f32c(waypoints)]
    dn = dest_num.contiguous()
    gts = [None] * 5
    if entry is not None:
        gts = [L.f32c(p_gt), L.f32c(v_gt), L.f32c(a_gt), L.f32c(dest_gt), dest_idx_gt.contiguous()]
        entry = entry.contiguous()
    L.check(L.load().piml_integrate_step_f32(
        L.ptr(p), L.ptr(v), L.ptr(a), L.ptr(args[0]), L.ptr(dest), L.ptr(dest_idx), L.ptr(dn), L.ptr(args[1]), S, D,
        N, float(dt), 1 if remove_on_arrival else 0, L.ptr(entry), *[L.ptr(g) for g in gts], L.ptr(hist_v),
        L.ptr(rec_p), L.ptr(rec_v), L.ptr(rec_a), L.ptr(rec_mask), L.stream_ptr(dev)), "piml_integrate_step_f32")


def state_features(p, v, a, dest, obstacles, hist_v, desired_speed, topk_ped, sight_angle_ped, dist_threshold_ped,
                   topk_obs, sight_angle_obs, dist_threshold_obs, out=None):
    """Feature rebuild of one rollout step for S scenes: returns (ped_f (S,N,kp,6), obs_f (S,N,ko,6),
    self_f (S,N,7)).  p, v, a, dest, hist_v (S,N,2); desired_speed (S,N); obstacles (M,2) or (S,M,2)."""
    dev = L.require_cuda(p, v, a, dest, obstacles, hist_v, desired_speed)
    S, N = p.shape[0], p.shape[1]
    M = obstacles.shape[-2] if obstacles.numel() else 0
    kp, ko = min(topk_ped, N), (min(topk_obs, M) if M else 0)
    if out is None:
        out = (torch.empty(S, N, kp, 6, device=dev), torch.empty(S, N, ko, 6, device=dev),
               torch.empty(S, N, 7, device=dev), torch.empty(S, N, 2, device=dev))
    ped_f, obs_f, self_f, dest_f = out
    L.check(L.load().piml_state_features_f32(
        L.ptr(p), L.ptr(v), L.ptr(a), L.ptr(dest), L.ptr(obstacles) if M else None,
        1 if (obstacles.dim() == 3 and M) else 0, S, N, M, topk_ped, cos_threshold(sight_angle_ped),
        float(dist_threshold_ped), topk_obs, cos_threshold(sight_angle_obs), float(dist_threshold_obs),
        L.ptr(hist_v), L.ptr(desired_speed), L.ptr(ped_f), L.ptr(obs_f) if M else None, L.ptr(self_f),
        L.ptr(dest_f), L.stream_ptr(dev)), "piml_state_features_f32")
    return ped_f, obs_f, self_f


class NNStep(object):
    """One NN-augmented rollout step as ONE library call (piml_nn_step_f32, csrc/nn_step.cu): features of the current
    state -> a_next = model(features) -> Euler / arrival / waypoints / entry, i.e. simulators.py:642-652, :602, :596-639
    in the order a loop over the STATE runs them.  Bit-identical to `state_features` -> `models.pinnsf_forward` ->
    `integrate_step`, in 7 launches instead of 12 and without the dense feature tensors.

    The state tensors p, v, a, dest, hist_v (S,N,2) and dest_idx (S,N) are bound once and updated in place by every
    `step()`; the other arguments are fixed for the object's lifetime.  Raises if the network is not one
    `piml_nn_step_supported` accepts (use the three calls then)."""

    def __init__(self, spec, packed_tc, p, v, a, dest, dest_idx, hist_v, dest_num, waypoints, desired_speed, obstacles,
                 dt, topk_ped, sight_angle_ped, dist_threshold_ped, topk_obs, sight_angle_obs, dist_threshold_obs,
                 remove_on_arrival=True, a_next=None, dense=None):
        dev = L.require_cuda(p, v, a, dest, dest_idx, hist_v, dest_num, waypoints, desired_speed, obstacles, packed_tc)
        for t in (p, v, a, dest, dest_idx, hist_v):
            if not t.is_contiguous() or t.dim() != (2 if t is dest_idx else 3):
                raise ValueError("NNStep updates its state tensors in place; they must be contiguous (S,N,..) tensors")
        S, N = p.shape[0], p.shape[1]
        Mo = obstacles.shape[-2] if obstacles.numel() else 0
        self._desc = spec.desc()
        if not L.load().piml_nn_step_supported(L.C.byref(self._desc)):
            raise NotImplementedError("piml_nn_step_f32 runs per-slot-decoder networks with hidden widths 32/64/128")
        if spec.has_obs and not Mo:
            raise ValueError("the network has an obstacle branch but the scene has no obstacles")
        dn = dest_num if dest_num.numel() == S * N else dest_num.expand(S, N)
        # everything the argument block points at stays referenced by the object
        self._keep = [packed_tc, p, v, a, dest, dest_idx, hist_v, dn.contiguous(), L.f32c(waypoints),
                      L.f32c(desired_speed), L.f32c(obstacles), a_next, dense]
        self.device = dev
        r = L.NnStepArgs()
        r.desc, r.packed_tc = L.C.pointer(self._desc), L.ptr(packed_tc)
        r.has_obs, r.tau = (1 if (spec.has_obs and Mo) else 0), spec.tau
        r.S, r.N, r.M, r.D, r.dt = S, N, Mo, self._keep[8].shape[-3], float(dt)
        r.remove_on_arrival = 1 if remove_on_arrival else 0
        r.kp, r.cos_p, r.thr_p = topk_ped, cos_threshold(sight_angle_ped), float(dist_threshold_ped)
        r.ko, r.cos_o, r.thr_o = topk_obs, cos_threshold(sight_angle_obs), float(dist_threshold_obs)
        r.obstacles = L.ptr(self._keep[10]) if Mo else None
        r.obs_per_scene = 1 if (obstacles.dim() == 3 and Mo) else 0
        r.dest_num, r.waypoints, r.desired_speed = L.ptr(self._keep[7]), L.ptr(self._keep[8]), L.ptr(self._keep[9])
        r.p, r.v, r.a, r.dest, r.dest_idx, r.hist_v = [L.ptr(x) for x in (p, v, a, dest, dest_idx, hist_v)]
        r.a_next = L.ptr(a_next)
        if dense is not None:                  # (ped_f, obs_f, self_f, dest_f) of the state the step starts from
            r.ped_f, r.obs_f, r.self_f, r.dest_f = [L.ptr(x) for x in dense]
        self._args = r
        self._fn = L.load().piml_nn_step_f32

    def step(self, entry=None, gt=None, rec=None):
        """gt = (p, v, a, dest, dest_idx) of the data at t+1 when `entry` (S,N) int64 is given; rec = (p, v, a, mask)
        buffers that receive the state at t."""
        r = self._args
        r.entry = L.ptr(entry)
        if entry is not None:
            r.p_gt, r.v_gt, r.a_gt, r.dest_gt, r.dest_idx_gt = [L.ptr(x) for x in gt]
        r.rec_p, r.rec_v, r.rec_a, r.rec_mask = [L.ptr(x) for x in rec] if rec is not None else [None] * 4
        L.check(self._fn(L.C.byref(r), L.stream_ptr(self.device)), "piml_nn_step_f32")


class RolloutResult(object):
    """What the reference returns as `RawData(p_res, v_res, a_res, destination, destination, obstacles, mask_p_new)`
    (simulators.py:655-656)."""

    def __init__(self, position, velocity, acceleration, destination, obstacles, mask_p, meta_data=None):
        self.position, self.velocity, self.acceleration = position, velocity, acceleration
        self.destination, self.waypoints, self.obstacles = destination, destination, obstacles
        self.mask_p, self.meta_data = mask_p, meta_data
        if meta_data is not None and 'time_unit' in meta_data:
            self.time_unit = meta_data['time_unit']
        self.num_steps, self.num_pedestrians = position.shape[-3], position.shape[-2]


def rollout_scenes(spec, packed, args, scene, t_start=0, num_frames=None, packed_tc=None, final_state=None):
    """Roll S independent scenes forward together (one launch per stage per step, no host sync).

    scene: dict of CUDA tensors
        position, velocity, acceleration, destination (S,T,N,2); dest_idx (S,T,N) int64; waypoints (S,D,N,2);
        dest_num (S,N) int64; obstacles (M,2) or (S,M,2); mask_p, mask_p_pred (S,T,N); desired_speed (S,N);
        ped_features0 (S,N,kp,6), obs_features0 (S,N,ko,6), self_features0 (S,N,7): features at t_start.
    Returns p_res, v_res, a_res (S,T,N,2) and mask_p_new (S,T,N) exactly as simulators.py:581-600 builds them.
    final_state: optional dict that receives the loop's final `dest_idx` (S,N) and `hist_v` (S,N,2).
    """
    pos, vel, acc, dst = scene["position"], scene["velocity"], scene["acceleration"], scene["destination"]
    dev = L.require_cuda(pos, vel, acc, dst, packed)
    S, T, N = pos.shape[0], pos.shape[1], pos.shape[2]
    T = T if num_frames is None else min(T, num_frames)
    dt = float(args.time_unit)
    # time-major copies so that frame t of all scenes is one contiguous (S,N,..) block for the kernels
    tm = {k: scene[k].transpose(0, 1).contiguous() for k in ("position", "velocity", "acceleration", "destination")}
    didx_tm = scene["dest_idx"].transpose(0, 1).contiguous()
    flag_tm = (scene["mask_p"] - scene["mask_p_pred"]).long().transpose(0, 1).contiguous()     # simulators.py:593
    p_res = torch.zeros(T, S, N, 2, device=dev)
    v_res = torch.zeros(T, S, N, 2, device=dev)
    a_res = torch.zeros(T, S, N, 2, device=dev)
    mask_new = torch.zeros(T, S, N, device=dev)
    p_res[:t_start + 1] = tm["position"][:t_start + 1]                                        # :585-587
    v_res[:t_start + 1] = tm["velocity"][:t_start + 1]
    a_res[:t_start + 1] = tm["acceleration"][:t_start + 1]
    mask_new[:t_start + 1] = scene["mask_p"].transpose(0, 1)[:t_start + 1].long().float()     # :591
    p, v, a = tm["position"][t_start].clone(), tm["velocity"][t_start].clone(), tm["acceleration"][t_start].clone()
    dest, didx = tm["destination"][t_start].clone(), didx_tm[t_start].clone()
    dnum, wp = scene["dest_num"].contiguous(), L.f32c(scene["waypoints"])
    obstacles = L.f32c(scene["obstacles"])
    ds = L.f32c(scene["desired_speed"])
    ped_f, obs_f, self_f = (L.f32c(scene["ped_features0"]), L.f32c(scene["obs_features0"]),
                            L.f32c(scene["self_features0"]))
    hist = torch.empty(S, N, 2, device=dev)
    kp, ko = ped_f.shape[-2], obs_f.shape[-2]
    Mo = obstacles.shape[-2] if obstacles.numel() else 0
    # feature buffers: hold the features of the state at t_start, then are rewritten in place every step
    ped_f, self_f = ped_f.reshape(S, N, kp, 6).clone(), self_f.reshape(S, N, 7).clone()
    obs_f = obs_f.reshape(S, N, ko, 6).clone() if Mo else None
    dest_f = torch.empty(S, N, 2, device=dev)
    a_next = torch.empty(S, N, 2, device=dev)
    if dnum.numel() != S * N:
        dnum = dnum.expand(S, N).contiguous()
    r = L.RolloutArgs()
    if isinstance(spec, SfmSpec):              # pure social-force mode (BASELINE config 2): no network
        sfm_prm = spec.params()
        r.sfm = L.C.cast(L.C.pointer(sfm_prm), L.C.c_void_p)
    else:
        desc = spec.desc()
        r.desc = L.C.pointer(desc)
        r.packed = L.ptr(packed)
        r.packed_tc = L.ptr(packed_tc) if packed_tc is not None else None
    r.has_obs, r.tau = (1 if (spec.has_obs and Mo) else 0), spec.tau
    r.S, r.N, r.M, r.D, r.T, r.t_start, r.dt = S, N, Mo, wp.shape[-3], T, t_start, dt
    r.kp, r.cos_p, r.thr_p = args.topk_ped, cos_threshold(args.sight_angle_ped), float(args.dist_threshold_ped)
    r.ko, r.cos_o, r.thr_o = args.topk_obs, cos_threshold(args.sight_angle_obs), float(args.dist_threshold_obs)
    r.obstacles, r.obs_per_scene = (L.ptr(obstacles) if Mo else None), (1 if (obstacles.dim() == 3 and Mo) else 0)
    r.pos_tm, r.vel_tm, r.acc_tm, r.dest_tm = [L.ptr(tm[k]) for k in ("position", "velocity", "acceleration",
                                                                        "destination")]
    r.dest_idx_tm, r.entry_tm, r.dest_num = L.ptr(didx_tm), L.ptr(flag_tm), L.ptr(dnum)
    r.waypoints, r.desired_speed = L.ptr(wp), L.ptr(ds)
    r.p, r.v, r.a, r.dest, r.dest_idx, r.hist_v = [L.ptr(x) for x in (p, v, a, dest, didx, hist)]
    r.ped_f, r.obs_f, r.self_f, r.dest_f, r.a_next = L.ptr(ped_f), L.ptr(obs_f), L.ptr(self_f), L.ptr(dest_f), \
        L.ptr(a_next)
    r.rec_p, r.rec_v, r.rec_a, r.rec_mask = L.ptr(p_res), L.ptr(v_res), L.ptr(a_res), L.ptr(mask_new)
    if spec.has_obs and not Mo:
        raise ValueError("the network has an obstacle branch but the scene has no obstacles")
    # the whole `for t in range(t_start, T)` loop of simulators.py:595-652: one C call, 3-4 launches per step
    L.check(L.load().piml_rollout_f32(L.C.byref(r), L.stream_ptr(dev)), "piml_rollout_f32")
    if final_state is not None:
        final_state["dest_idx"], final_state["hist_v"] = didx, hist
    return (p_res.transpose(0, 1), v_res.transpose(0, 1), a_res.transpose(0, 1), mask_new.transpose(0, 1))


def scene_from_data(data, t_start, device):
    """Pack a reference `TimeIndexedPedData` (src/data/data.py:604-863) into the dict rollout_scenes expects (S=1)."""
    def dv(x, dtype=None):
        x = x.to(device)
        return x.to(dtype) if dtype is not None else x
    return {
        "position": dv(data.position)[None], "velocity": dv(data.velocity)[None],
        "acceleration": dv(data.acceleration)[None], "destination": dv(data.destination)[None],
        "dest_idx": dv(data.dest_idx, torch.int64)[None], "waypoints": dv(data.waypoints)[None],
        "dest_num": dv(data.dest_num, torch.int64)[None], "obstacles": dv(data.obstacles),
        "mask_p": dv(data.mask_p)[None], "mask_p_pred": dv(data.mask_p_pred)[None],
        "desired_speed": dv(data.self_features)[t_start, :, -1][None].contiguous(),
        "ped_features0": dv(data.ped_features)[t_start][None], "obs_features0": dv(data.obs_features)[t_start][None],
        "self_features0": dv(data.self_features)[t_start][None],
    }


def get_multiple_rollouts(simulator, data, t_start=0, load_model=True, result_cls=None):
    """Drop-in body for `BaseSimulator.get_multiple_rollouts(self, data, t_start=0, load_model=True)`.

    `simulator` provides .args, .model (a reference PINNSF module or a piml_b200.models mirror), .load_model and
    .finetune_flag exactly like the reference class.  Returns `result_cls(p_res, v_res, a_res, destination,
    destination, obstacles, mask_p_new, meta_data=...)` -- pass the reference's DATA.RawData to get its type back.
    """
    args = simulator.args
    if load_model:
        simulator.load_model(args, set_model=False, finetune_flag=simulator.finetune_flag)      # :563-564
    if not torch.cuda.is_available():
        raise RuntimeError("piml_b200.get_multiple_rollouts needs a CUDA device; there is no CPU fallback")
    if data.position.dim() != 3:
        raise NotImplementedError("channelled rollouts: use rollout_scenes")
    dev = torch.device("cuda", torch.cuda.current_device())
    module = simulator.model.module if isinstance(simulator.model, torch.nn.DataParallel) else simulator.model
    if isinstance(module, SocialForce):
        spec, packed, packed_tc = module.spec, None, None
    else:
        spec = M.spec_from_module(module)
        packed = M.pack_device(module.state_dict(), spec, dev)
        packed_tc = M.pack_device_tc(module.state_dict(), spec, dev)    # None if the net cannot use the tensor cores
    if not hasattr(args, "time_unit"):
        args.time_unit = data.time_unit
    scene = scene_from_data(data, t_start, dev)
    final = {}
    p_res, v_res, a_res, mask_new = rollout_scenes(spec, packed, _with_dt(args, data.time_unit), scene, t_start,
                                                   data.num_frames, packed_tc=packed_tc, final_state=final)
    _write_back_side_effects(data, t_start, v_res[0], final)
    out_dev = data.position.device
    res = (p_res[0].to(out_dev), v_res[0].to(out_dev), a_res[0].to(out_dev))
    if result_cls is None:
        return RolloutResult(*res, data.destination, data.obstacles, mask_new[0].to(out_dev), data.meta_data)
    return result_cls(*res, data.destination, data.destination, data.obstacles, mask_new[0].to(out_dev),
                      meta_data=data.meta_data)


def _write_back_side_effects(data, t_start, v_res, final):
    """What a caller of the reference's loop can observe on `data` afterwards (simulators.py:571-578 hold VIEWS):
    `dest_idx_cur` is data.dest_idx[t_start] and is advanced in place at every step (:609, :613, :638), so it ends as the
    loop's final waypoint index; `hist_v` of the FIRST iteration is a view of data.self_features[t_start, :, 2:-3]
    and receives that step's new velocities, entrants taking their recorded history (:624-639).  Later iterations
    work on fresh tensors."""
    T = min(int(data.num_frames), data.position.shape[-3])
    if t_start >= T:
        return
    data.dest_idx[t_start].copy_(final["dest_idx"][0].to(data.dest_idx.device, data.dest_idx.dtype))
    sf = data.self_features
    if sf.shape[-1] != 7:                       # num_history_velocity == 1 is what the kernels implement
        return
    if t_start + 1 < T:
        hist = v_res[t_start + 1].to(sf.device)
        new = (data.mask_p[t_start + 1] - data.mask_p_pred[t_start + 1]).long().to(sf.device) == 1
        hist = torch.where(new.unsqueeze(-1), sf[t_start + 1, :, 2:4], hist)
    else:                                        # a single step at the last frame: v + a dt, never recorded
        hist = data.velocity[t_start] + data.acceleration[t_start] * data.time_unit
    sf[t_start, :, 2:4] = hist


def _sweep_spec(models):
    """The one NetSpec every model of a sweep shares (None for an empty list).  Touches neither library nor device."""
    if isinstance(models, torch.nn.Module) or not isinstance(models, (list, tuple)):
        raise ValueError("sweep_networks: models must be a list or tuple of PINNSF modules")
    mods = [m.module if isinstance(m, torch.nn.DataParallel) else m for m in models]
    specs = [M.spec_from_module(m) for m in mods]
    if not specs:
        return None, mods
    s0, c0 = specs[0], M._REF_CLASS_TO_MODEL[type(mods[0]).__name__]
    for i, (m, s) in enumerate(zip(mods, specs)):
        if M._REF_CLASS_TO_MODEL[type(m).__name__] != c0 or (s.enc_dims, s.proc_mode, s.dec_dims, s.coll_dims,
                                                              s.kind, s.has_obs) != \
                (s0.enc_dims, s0.proc_mode, s0.dec_dims, s0.coll_dims, s0.kind, s0.has_obs):
            raise ValueError(f"sweep_networks: model {i} differs from model 0 in class or widths; one sweep takes "
                             "one architecture")
        if s.tau != s0.tau:
            raise ValueError(f"sweep_networks: model {i} has tau {s.tau}, model 0 has {s0.tau}; one sweep takes one tau")
    return s0, mods


def sweep_networks(data_or_scene, models, args, t_start=0, num_frames=None, record=False):
    """Roll ONE clip out from t_start under S trained interaction networks in one library call (piml_nn_sweep_f32),
    and score each network: checkpoint selection, seed ensembles, grid-search evaluation.

    data_or_scene: a reference `TimeIndexedPedData` or the single-scene dict, exactly as `sfm.sweep` takes it.
    models: a list of S reference PINNSF modules (or piml_b200.models mirrors) of one class, the same widths and the
        same tau; networks the 16-bit tensor-core forward does not take (pinnsf_m / pinnsf, widths other than 32 / 64 /
        128) raise NotImplementedError before any device work.
    Network s rolls out exactly as `rollout_scenes(spec, None, args, scene, t_start, T, packed_tc=its vector)` on the
    clip alone.  Returns (err_sum (S,) float64, err_count (S,) int64) with sfm.sweep's definition, so networks and
    social-force constant sets rank on one scale; with record=True also (p_res, v_res, a_res (S,T,N,2),
    mask_p_new (S,T,N)).  Device memory: O(S N) plus the S packed networks (and 28 bytes per set, frame and slot with
    record=True)."""
    from .sfm import _clip_scene, _clip_shapes, _run_sweep, _stage_clip
    spec, mods = _sweep_spec(models)
    if spec is not None and not L.load().piml_nn_step_supported(L.C.byref(spec.desc())):
        raise NotImplementedError("sweep_networks runs the 16-bit tensor-core forward: per-slot-decoder networks "
                                  "(pinnsf_bm, pinnsf_bottleneck) with hidden widths 32 / 64 / 128")
    scene, dt, num_frames = _clip_scene(data_or_scene, args, t_start, num_frames, "sweep_networks")
    T, N, Mo = _clip_shapes(scene, args, dt, t_start, num_frames, "sweep_networks")
    if spec is not None and spec.has_obs and not Mo:
        raise ValueError("the network has an obstacle branch but the scene has no obstacles")
    S = len(mods)
    dev, sc = _stage_clip(scene)
    r = L.NnSweepArgs()
    if S:
        desc = spec.desc()
        n = int(L.load().piml_pinnsf_packed_tc_floats(L.C.byref(desc)))
        stride = -(-n // 32) * 32                  # 128-byte rows: each vector as aligned as a lone allocation
        packed = torch.empty(S, stride, dtype=torch.float32, device=dev)
        for s, m in enumerate(mods):
            M.pack_device_tc(m.state_dict(), spec, dev, out=packed[s])
        r.desc, r.packed_tc, r.set_stride = L.C.pointer(desc), L.ptr(packed), stride
        r.has_obs, r.tau = (1 if (spec.has_obs and Mo) else 0), spec.tau
    return _run_sweep(r, dev, sc, S, T, N, Mo, t_start, dt, args, record, "piml_nn_sweep")


class _with_dt(object):
    """args view whose time_unit is the clip's (simulators.py uses data.time_unit, not args.time_unit)."""

    def __init__(self, args, dt):
        self._a, self.time_unit = args, dt

    def __getattr__(self, k):
        return getattr(self._a, k)
