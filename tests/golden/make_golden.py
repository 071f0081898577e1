"""Generate the committed golden vectors by running the UNMODIFIED reference (located by tests/golden/_refharness.py).

    PIML_REFERENCE=<upstream PIML checkout> python tests/golden/make_golden.py [group ...]
Groups: features models mlapm sfm rollout sfm_rollout training metrics losses.   Output: tests/golden/*.npz (small, compressed).

The reference ships no tests and no golden vectors (SURVEY.md section 4 / 8c), so these files ARE the pin: they
hold the reference's own outputs on its own data files (GC / UCY / toy clips) and on seeded synthetic crowds.
Nothing here is imported at test time; tests only np.load the .npz files.
"""
import copy
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _refharness as H  # noqa: E402

DATA, MODEL, MLAPM, SIM, UTILS = H.import_reference()
torch.set_num_threads(1)        # reproducible fp32 reductions


def save(name, **arrs):
    path = os.path.join(HERE, name + ".npz")
    out = {}
    for k, v in arrs.items():
        if isinstance(v, torch.Tensor):
            v = v.detach().cpu().numpy()
        out[k] = np.asarray(v)
    np.savez_compressed(path, **out)
    print(f"wrote {path}  {os.path.getsize(path) / 1024:.1f} KiB")


def synthetic_crowd(N, M, seed=666, rho=0.5):
    """SURVEY.md 8d config 4 recipe (scenarios.py:363-366 flavoured). Returns fp32 tensors."""
    g = torch.Generator().manual_seed(seed)
    L = float(np.sqrt(N / rho))
    p = torch.rand(N, 2, generator=g) * L
    dest = torch.rand(N, 2, generator=g) * L
    e = dest - p
    e = e / e.norm(dim=-1, keepdim=True).clamp_min(1e-6)
    v = 1.34 * e * (0.5 + 0.5 * torch.rand(N, 1, generator=g)) + 0.1 * torch.randn(N, 2, generator=g)
    a = torch.zeros(N, 2)
    ds = (1.34 + np.sqrt(0.26) * torch.randn(N, 1, generator=g)).clamp_min(0.7)
    rings = max(M // 200, 1)
    per = M // rings
    ang = torch.arange(per) * (2 * np.pi / per)
    obs = []
    for r in range(rings):
        cx, cy = (r % 5 + 0.5) * L / 5, (r // 5 + 0.5) * L / 2
        obs.append(torch.stack([cx + 2.75 * ang.cos(), cy + 2.75 * ang.sin()], -1))
    obs = torch.cat(obs, 0).float()[:M]
    return p, v, a, dest, ds, obs


def feature_case(name, p, v, a, d, obs, kp=6, ap=90, tp=4, ko=10, ao=90, to=4):
    """Runs get_relative_features + the two get_nearby_obj_in_sight calls it makes (data.py:466-512)."""
    ped = DATA.Pedestrians()
    v_in, a_in = v.clone(), a.clone()
    v_w, a_w = v.clone(), a.clone()
    pf, of, df = ped.get_relative_features(p.clone(), v_w, a_w, d.clone(), obs.clone(), kp, ap, tp, ko, ao, to)
    head = ped.get_heading_direction(v_w)
    pd_, pi_ = ped.get_nearby_obj_in_sight(p.clone(), p.clone(), head, kp, ap)
    dim = obs.dim()
    T = p.shape[-3]
    obs_t = obs.unsqueeze(-3).repeat(*([1] * (dim - 2) + [T] + [1, 1]))
    od_, oi_ = ped.get_nearby_obj_in_sight(p.clone(), obs_t, head, ko, ao)
    pre = name + "/"
    return {pre + "position": p, pre + "velocity": v_in, pre + "acceleration": a_in, pre + "destination": d,
            pre + "obstacles": obs, pre + "params": np.array([kp, ap, tp, ko, ao, to], np.int64),
            pre + "velocity_after": v_w, pre + "acceleration_after": a_w, pre + "heading": head,
            pre + "ped_features": pf, pre + "obs_features": of, pre + "dest_features": df,
            pre + "ped_dist": pd_, pre + "ped_idx": pi_.to(torch.int32), pre + "obs_dist": od_,
            pre + "obs_idx": oi_.to(torch.int32)}


def gen_features():
    out = {}
    raw = H.load_raw(H.GC_CLIP)
    ts = [25, 100, 180, 260, 333, 410, 555, 700]
    out.update(feature_case("gc", raw.position[ts], raw.velocity[ts], raw.acceleration[ts], raw.destination[ts],
                            raw.obstacles))
    # a contiguous window: exercises the heading forward/backward fill over time (last frame of a ped has v=0)
    sl = slice(300, 340)
    out.update(feature_case("gc_window", raw.position[sl], raw.velocity[sl], raw.acceleration[sl],
                            raw.destination[sl], raw.obstacles))
    ucy = H.load_raw(H.UCY_CLIP)
    ts = [0, 50, 200, 400, 600, 675]
    out.update(feature_case("ucy", ucy.position[ts], ucy.velocity[ts], ucy.acceleration[ts], ucy.destination[ts],
                            ucy.obstacles))
    toy = H.load_raw(H.TOY_CLIP)
    sl = slice(20, 60)
    out.update(feature_case("toy", toy.position[sl], toy.velocity[sl], toy.acceleration[sl], toy.destination[sl],
                            toy.obstacles))
    p, v, a, d, ds, obs = synthetic_crowd(512, 2000)
    out.update(feature_case("syn512", p[None], v[None], a[None], d[None], obs))
    # wide field of view (self is selected at distance 0, SURVEY B-6), odd k / thresholds, NaN agents, NaN v/a
    p, v, a, d, ds, obs = synthetic_crowd(300, 400, seed=7)
    p[::17] = float('nan'); d[::17] = float('nan'); v[::17] = 0; v[5] = float('nan'); a[9] = float('nan')
    v[40:60] = 0
    out.update(feature_case("syn300_wide", p[None], v[None], a[None], d[None], obs, 4, 100, 3, 7, 120, 5))
    # channelled (C,T,N,2) with per-channel obstacles and stationary stretches
    g = torch.Generator().manual_seed(11)
    Cc, T, N, M = 3, 5, 40, 12
    p = torch.rand(Cc, T, N, 2, generator=g) * 9
    v = torch.randn(Cc, T, N, 2, generator=g)
    v[:, 1:3, ::3] = 0
    v[1, :, 7] = 0
    v[2, 4, :] = 0
    a = torch.randn(Cc, T, N, 2, generator=g)
    d = torch.rand(Cc, T, N, 2, generator=g) * 9
    p[0, :, 3] = float('nan'); d[0, :, 3] = float('nan')
    obs = torch.rand(Cc, M, 2, generator=g) * 9
    out.update(feature_case("channelled", p, v, a, d, obs))
    save("features", **out)


def model_args(kind, small=False, obs=True, dataset_name='ucy'):
    a = H.default_args(model=kind, dataset_name=dataset_name, obs_feature_dim=6 if obs else 0)
    if small:
        a.encoder_hidden_size = 32; a.processor_hidden_size = 32; a.decoder_hidden_size = 16
        a.encoder_hidden_layers = 2; a.processor_hidden_layers = 1; a.decoder_hidden_layers = 1
    return a


MODEL_CLASSES = {'pinnsf': 'PINNSF', 'pinnsf_bottleneck': 'PINNSF_bottleneck',
                 'pinnsf_bm': 'PINNSF_bottleneck_multitask', 'pinnsf_m': 'PINNSF_multitask'}


def build_model(kind, args, seed=666):
    torch.manual_seed(seed)
    m = getattr(MODEL, MODEL_CLASSES[kind])(args)
    m.eval()
    return m


def gen_models():
    raw = H.load_raw(H.GC_CLIP)
    args0 = H.default_args()
    d = H.make_time_indexed(args0, raw)
    t = 333
    ped, obs, slf = d.ped_features[t].clone(), d.obs_features[t].clone(), d.self_features[t].clone()
    chan = slice(330, 334)
    pedc, obsc, slfc = d.ped_features[chan].clone(), d.obs_features[chan].clone(), d.self_features[chan].clone()
    out = {"ped": ped, "obs": obs, "self": slf, "ped_c": pedc, "obs_c": obsc, "self_c": slfc}
    cases = [("pinnsf_bm", False, True, 'gc1560'), ("pinnsf_m", False, True, 'ucy'),
             ("pinnsf_bottleneck", True, True, 'ucy'), ("pinnsf", True, False, 'ucy')]
    for kind, small, has_obs, dsn in cases:
        args = model_args(kind, small, has_obs, dsn)
        m = build_model(kind, args)
        pre = kind + "/"
        for k, v in m.state_dict().items():
            out[pre + "sd/" + k] = v
        out[pre + "cfg"] = np.array([args.encoder_hidden_size, args.processor_hidden_size, args.decoder_hidden_size,
                                     args.encoder_hidden_layers, args.processor_hidden_layers,
                                     args.decoder_hidden_layers, 1 if has_obs else 0], np.int64)
        out[pre + "dataset_name"] = np.array(dsn)
        out[pre + "tau"] = np.float64(m.tau)
        with torch.no_grad():
            res = m(ped, obs, slf)
            resc = m(pedc, obsc, slfc)
        for i, r in enumerate(res):
            out[pre + f"out{i}"] = r
        for i, r in enumerate(resc):
            out[pre + f"outc{i}"] = r
    save("models", **out)


def gen_mlapm():
    out = {}
    # main_mlapm.py:6-36 scene, seeded
    torch.manual_seed(0)
    N, dt, radius = 7, 0.08, 0.3
    theta = torch.linspace(0, 2 * torch.pi * (1 - 1. / N), N)
    position = torch.stack([10 * theta.cos(), 10 * theta.sin()], dim=-1).view(-1, 1, 2)
    velocity = torch.rand(N, 1, 2)
    mask = torch.full([N, 1, 1], True)
    desired_speed = torch.full([N, 2], 1.5)
    destination = -position.view(-1, 2)
    model = MLAPM.MLAPM(version='GC', tau=0.5, A=7.55, B=-3.00, C=0.2, D=-0.3, theta=56)
    for i in range(200):
        v = model.step(position[mask[:, -1, 0], -1, :], velocity[mask[:, -1, 0], -1, :],
                       desired_speed[mask[:, -1, 0], :], destination[mask[:, -1, 0], :], dt=dt, radius=radius)
        p = position[mask[:, -1, 0], -1, :] + v * dt
        position = torch.concat([position, torch.full([N, 1, 2], float('nan'))], dim=1)
        velocity = torch.concat([velocity, torch.full([N, 1, 2], float('nan'))], dim=1)
        mask = torch.concat([mask, mask[:, (-1,), :]], dim=1)
        position[mask[:, -1, 0], -1, :] = p
        velocity[mask[:, -1, 0], -1, :] = v
        mask[:, -1, :] &= ~((position[:, -1, :] - destination).norm(dim=-1, keepdim=True) < radius)
        if not mask.any():
            break
    out.update({"circle/position": position, "circle/velocity": velocity, "circle/mask": mask[:, :, 0],
                "circle/desired_speed": desired_speed, "circle/destination": destination})
    kw = dict(tau=0.5, A=7.55, B=-3.00, C=0.2, D=-0.3, theta=56)
    for N in (257, 1000):
        p, v, a, d, ds, obs = synthetic_crowd(N, 200, seed=N)
        for ver in ("raw", "GC"):
            m = MLAPM.MLAPM(version=ver, **kw)
            act = m.step(p, v, ds, d, dt=0.08)
            out[f"syn{N}/{ver}/action"] = act
        vr = p.view(1, -1, 2) - p.view(-1, 1, 2)
        view = torch.einsum('nk,nmk->nm', v, vr) > 0.          # mlapm.py:27
        out[f"syn{N}/view_bits"] = np.packbits(view.numpy())
        out.update({f"syn{N}/position": p, f"syn{N}/velocity": v, f"syn{N}/desired_speed": ds,
                    f"syn{N}/destination": d})
    # (N,2) desired speed as main_mlapm passes it, non-default parameters
    p, v, a, d, ds, obs = synthetic_crowd(300, 200, seed=3)
    ds2 = torch.cat([ds, ds * 1.1], -1)
    m = MLAPM.MLAPM(version='GC', tau=0.7, A=5.0, B=-2.0, C=0.1, D=-0.2, theta=30)
    out.update({"syn300b/position": p, "syn300b/velocity": v, "syn300b/desired_speed": ds2,
                "syn300b/destination": d, "syn300b/GC/action": m.step(p, v, ds2, d, dt=0.05),
                "syn300b/params": np.array([0.7, 5.0, -2.0, 0.1, -0.2, 30, 0.05])})
    save("mlapm", **out)


def gen_sfm():
    raw = H.load_raw(H.GC_CLIP)
    d = H.make_time_indexed(H.default_args(), raw)
    ped = d.ped_features[333].clone()                    # (N,6,6)
    out = {"ped": ped}
    for ver, dsn in (("v0", "gc1560"), ("v0", "ucy"), ("v1", "gc2344"), ("v1", "ucy"), ("v2", "gc2344")):
        out[f"{ver}/{dsn}"] = UTILS.calc_acceleration(ped.clone(), ver, dsn)
    pc = d.ped_features[330:334].clone()                 # (4,N,6,6) -> the 'bnmj' einsum branch
    out["ped_c"] = pc
    out["v2c/gc2344"] = UTILS.calc_acceleration(pc.clone(), "v2", "gc2344")
    out["v0c/gc1560"] = UTILS.calc_acceleration(pc.clone(), "v0", "gc1560")
    save("sfm", **out)


def rollout_case(clip, kind, dataset_name, t_start=25, seed=666, max_frames=None, module=None):
    """BaseSimulator.get_multiple_rollouts (simulators.py:556-657) on a deepcopy of the clip, recording the state
    handed to get_relative_features each step (= the reference's own p/v/a/dest after update + entry)."""
    raw = H.load_raw(clip)
    args = H.default_args(model=kind, dataset_name=dataset_name)
    data = H.make_time_indexed(args, raw)
    if max_frames is not None and max_frames < data.num_frames:
        data.num_frames = max_frames
    args.ped_feature_dim, args.obs_feature_dim, args.self_feature_dim = 6, 6, 7
    torch.manual_seed(seed)
    with H.quiet():
        sim = SIM.BaseSimulator(args)
    if module is not None:
        sim.model = module
    sim.model.eval()
    inp = {}
    for k in ("position", "velocity", "acceleration", "destination", "waypoints", "obstacles", "mask_p",
              "mask_p_pred", "dest_num"):
        inp[k] = getattr(data, k).clone()
    inp["dest_idx"] = data.dest_idx.clone().to(torch.int32)
    inp["desired_speed"] = data.self_features[t_start, :, -1].clone()
    inp["ped_features0"] = data.ped_features[t_start].clone()
    inp["obs_features0"] = data.obs_features[t_start].clone()
    inp["self_features0"] = data.self_features[t_start].clone()
    rec_dest, rec_idx = [], []
    orig = sim.get_relative_features

    def spy(p, v, a, dst, *rest):
        rec_dest.append(dst.squeeze(-3).clone())
        return orig(p, v, a, dst, *rest)
    sim.get_relative_features = spy
    work = copy.deepcopy(data)
    with H.quiet(), torch.no_grad():
        res = sim.get_multiple_rollouts(work, t_start=t_start, load_model=False)
    T = data.num_frames
    out = {"in/" + k: v for k, v in inp.items()}
    out["in/t_start"] = np.int64(t_start)
    out["in/num_frames"] = np.int64(T)
    out["in/time_unit"] = np.float64(data.time_unit)
    out["in/model"] = np.array(kind)
    out["in/dataset_name"] = np.array(dataset_name)
    out["in/tau"] = np.float64(sim.model.tau)
    for k, v in sim.model.state_dict().items():
        out["sd/" + k] = v
    out["out/position"] = res.position[:T]
    out["out/velocity"] = res.velocity[:T]
    out["out/acceleration"] = res.acceleration[:T]
    out["out/mask_p"] = res.mask_p[:T]
    out["out/dest_after_step"] = torch.stack(rec_dest, 0)     # (T - t_start, N, 2): dest_cur after step t
    return out


class SocialForceComposed(torch.nn.Module):
    """BASELINE config 2 (SURVEY.md 8c): the generator of data/synthetic_data/*_simulation.npy (models.socialforce) is
    not shipped, so the pure social-force mode is pinned against a module COMPOSED OF SHIPPED REFERENCE CODE with the
    model(ped, obs, self) -> list interface (model.py:1185):
        ped messages   UTILS.calc_acceleration(ped_features, 'v0', dataset)        utils.py:46-58
        obs messages   the same v0 form with the obstacle constants of socialforce.yaml:52-56
                       (intensity 10, radius 0.2  ->  A = 10/0.2, B = -1/0.2, exactly as the shipped ped-ped constants
                       8.75 = 3.5/0.4, -2.5 = -1/0.4 relate to that file's intensity / radius)
        dest term      the lines model.py:1205-1210, verbatim, tau = 1/desired_speed_intensity = 0.5 (socialforce.yaml:29)
    rolled out by the UNMODIFIED BaseSimulator.get_multiple_rollouts."""

    def __init__(self, dataset, tau=0.5, A_obs=10 / 0.2, B_obs=-1 / 0.2):
        super().__init__()
        self.dataset, self.tau, self.A_obs, self.B_obs = dataset, tau, A_obs, B_obs

    def forward(self, ped_features, obs_features, self_features):
        ped_msgs = UTILS.calc_acceleration(ped_features, 'v0', self.dataset)
        pred_acc_ped = torch.sum(ped_msgs, dim=-2)
        dr = obs_features[..., 0:2]                                    # utils.py:53-58 with the obstacle constants
        r = torch.linalg.norm(dr, ord=2, dim=-1, keepdim=True)
        r += 1e-6
        obs_msgs = -(self.A_obs * torch.exp(self.B_obs * r)) * (dr / r)
        pred_acc_ped = pred_acc_ped + torch.sum(obs_msgs, dim=-2)
        desired_speed = self_features[..., -1].unsqueeze(-1)           # model.py:1205-1210
        temp = torch.norm(self_features[..., :2], p=2, dim=1, keepdim=True)
        temp_ = temp.clone()
        temp_[temp_ == 0] = temp_[temp_ == 0] + 0.1
        dest_direction = self_features[..., :2] / temp_
        pred_acc_dest = (desired_speed * dest_direction - self_features[..., 2:4]) / self.tau
        return [pred_acc_ped + pred_acc_dest, ped_msgs, obs_msgs]


def sfm_rollout_case(clip, dataset_name, t_start):
    """get_multiple_rollouts of the composed social-force module from the clip's own state at t_start."""
    out = rollout_case(clip, "pinnsf_bm", dataset_name, t_start=t_start, module=SocialForceComposed(dataset_name))
    out = {k: v for k, v in out.items() if not k.startswith("sd/")}
    out["in/model"] = np.array("sfm")
    out["in/tau"] = np.float64(0.5)
    out["in/sfm_consts"] = np.array([8.75, -2.5, 10 / 0.2, -1 / 0.2, 1e-6], np.float64)   # A_p, B_p, A_o, B_o, eps
    # one forward of the module on the features of frame 300, all three outputs
    raw = H.load_raw(clip)
    data = H.make_time_indexed(H.default_args(dataset_name=dataset_name), raw)
    with torch.no_grad():
        res = SocialForceComposed(dataset_name)(data.ped_features[300].clone(), data.obs_features[300].clone(),
                                                data.self_features[300].clone())
    out["fwd/ped"], out["fwd/obs"], out["fwd/self"] = data.ped_features[300], data.obs_features[300], \
        data.self_features[300]
    out["fwd/acc"], out["fwd/ped_msgs"], out["fwd/obs_msgs"] = res
    return out


def gen_sfm_rollout():
    save("rollout_syn_sfm", **sfm_rollout_case(H.SYN_CLIP, "gc1560", 25))


def gen_rollout():
    save("rollout_gc_bm", **rollout_case(H.GC_CLIP, "pinnsf_bm", "gc1560"))
    save("rollout_toy5_m", **rollout_case(H.TOY_CLIP, "pinnsf_m", "ucy", t_start=25))
    save("rollout_ucy_bm", **rollout_case(H.UCY_CLIP, "pinnsf_bm", "ucy", t_start=25, max_frames=200))


def _linear_keys(sd):
    """Linear layers the forward actually uses, in the order piml_b200.models.linear_keys produces them."""
    keys = []
    for br in ("ped", "obs"):
        l = 0
        while f"{br}_encoder.mlp.{2 * l}.weight" in sd:
            keys.append(f"{br}_encoder.mlp.{2 * l}"); l += 1
        l = 0
        while f"{br}_decoder.mlp.{2 * l}.weight" in sd:
            keys.append(f"{br}_decoder.mlp.{2 * l}"); l += 1
        keys.append(f"{br}_predictor.mlp.0")
    l = 0
    while f"ped_collision_predictor.mlp.{2 * l}.weight" in sd:
        keys.append(f"ped_collision_predictor.mlp.{2 * l}"); l += 1
    return keys


def single_step_case(kind, dsn, train_mode, ped, obs, slf, seed=666):
    """One forward + backward of the reference module (simulators.py:330-359 shape of work): a fixed random linear
    functional of every output, gradients w.r.t. every parameter and the three inputs.  In train() mode the
    Dropout multipliers the reference drew are recorded so the CUDA path can be fed the same ones."""
    args = model_args(kind, False, True, dsn)
    torch.manual_seed(seed)
    m = getattr(MODEL, MODEL_CLASSES[kind])(args)
    m.train(train_mode)
    masks = {}

    def hook(name):
        def f(mod, inp, out):
            x = inp[0]
            masks[name] = torch.where(x != 0, out / x, torch.ones_like(x) * float('nan')).detach()
        return f
    hs = [m.ped_processor.dropout.register_forward_hook(hook("ped")),
          m.obs_processor.dropout.register_forward_hook(hook("obs"))]
    ped, obs, slf = [x.clone().requires_grad_(True) for x in (ped, obs, slf)]
    torch.manual_seed(seed + 1)
    outs = m(ped, obs, slf)
    g = torch.Generator().manual_seed(seed + 2)
    ws = [torch.randn(o.shape, generator=g) for o in outs]
    loss = sum((o * w).sum() for o, w in zip(outs, ws))
    loss.backward()
    for h in hs:
        h.remove()
    pre = f"{kind}_{'train' if train_mode else 'eval'}/"
    out = {pre + "loss": loss.detach(), pre + "g_ped": ped.grad, pre + "g_obs": obs.grad, pre + "g_self": slf.grad,
           pre + "dataset_name": np.array(dsn)}
    for i, (o, w) in enumerate(zip(outs, ws)):
        out[pre + f"out{i}"] = o.detach()
        out[pre + f"w{i}"] = w
    named = dict(m.named_parameters())
    for k in _linear_keys(m.state_dict()):
        out[pre + "grad/" + k + ".weight"] = named[k + ".weight"].grad
        out[pre + "grad/" + k + ".bias"] = named[k + ".bias"].grad
    dead = [k for k, p_ in named.items() if p_.grad is None]
    out[pre + "dead"] = np.array(dead)
    if train_mode:
        # multiplier = 0 or 1/(1-p); where the input was exactly 0 the ratio is unknown -> any value gives 0
        for name in ("ped", "obs"):
            mk = masks[name]
            out[pre + "dropbits_" + name] = np.packbits((torch.nan_to_num(mk, nan=0.0) > 0).numpy())
            out[pre + "dropshape_" + name] = np.array(mk.shape)
    return out


def training_rollout_case(name, clip, kind, dsn, chans, valid_steps, **over):
    """BaseSimulator.test_multiple_rollouts_for_training (simulators.py:659-832) + loss.backward() (:359) on a
    channelled batch, eval() mode (no dropout)."""
    raw = H.load_raw(clip)
    args = H.default_args(model=kind, dataset_name=dsn, valid_steps=valid_steps, **over)
    data = H.make_time_indexed(args, raw)
    ch = DATA.ChanneledTimeIndexedPedData()
    with H.quiet():
        ch.load_from_time_indexed_peddata(data, stride=valid_steps, mode='slice')
    batch = DATA.ChanneledTimeIndexedPedData.slice(ch, chans)
    fields = ("ped_features", "obs_features", "self_features", "labels", "mask_p", "mask_p_pred", "position",
              "velocity", "acceleration", "destination", "dest_idx", "waypoints")
    for f in fields:
        setattr(batch, f, getattr(batch, f).clone())
    pre = name + "/"
    out = {pre + "in/" + f: getattr(batch, f).clone() for f in fields}
    out[pre + "in/obstacles"] = batch.obstacles.clone()
    out[pre + "in/dest_num"] = batch.dest_num.clone()
    out[pre + "in/abnormal_mask"] = batch.abnormal_mask.clone()
    out[pre + "in/time_unit"] = np.float64(batch.time_unit)
    out[pre + "in/num_frames"] = np.int64(batch.num_frames)
    out[pre + "in/model"] = np.array(kind)
    out[pre + "in/dataset_name"] = np.array(dsn)
    out[pre + "in/args"] = np.array([args.reg_weight, args.collision_threshold, args.collision_loss_weight,
                                     args.hard_collision_penalty, args.teacher_weight, args.collision_pred_weight,
                                     args.collision_focus_weight, args.new_collision_loss_flag, args.time_decay],
                                    np.float64)
    out[pre + "in/collision_loss_version"] = np.array(args.collision_loss_version)
    torch.manual_seed(666)
    with H.quiet():
        sim = SIM.BaseSimulator(args)
    sim.model.eval()
    sim.collision_count, sim.hard_collision_count, sim.epoch, sim.batch_idx = 0, 0, 0, 0
    with H.quiet():
        res = sim.test_multiple_rollouts_for_training(batch)
    res[0].backward()
    for i, r in enumerate(res):
        out[pre + f"out{i}"] = r.detach()
    out[pre + "collision_count"] = np.float64(sim.collision_count)
    out[pre + "hard_collision_count"] = np.float64(sim.hard_collision_count)
    out[pre + "dest_idx_after"] = batch.dest_idx.clone()
    named = dict(sim.model.named_parameters())
    for k in _linear_keys(sim.model.state_dict()):
        out[pre + "grad/" + k + ".weight"] = named[k + ".weight"].grad
        out[pre + "grad/" + k + ".bias"] = named[k + ".bias"].grad
    return out


def gen_training():
    raw = H.load_raw(H.GC_CLIP)
    d = H.make_time_indexed(H.default_args(), raw)
    t = 333
    ped, obs, slf = d.ped_features[t].clone(), d.obs_features[t].clone(), d.self_features[t].clone()
    out = {"ped": ped, "obs": obs, "self": slf}
    for kind, dsn in (("pinnsf_bm", "gc1560"), ("pinnsf_m", "ucy")):
        for train_mode in (False, True):
            out.update(single_step_case(kind, dsn, train_mode, ped, obs, slf))
    # channelled (C,N,.) inputs: the dim=1 destination-norm quirk in the backward
    chan = slice(330, 333)
    pedc, obsc, slfc = d.ped_features[chan].clone(), d.obs_features[chan].clone(), d.self_features[chan].clone()
    outc = single_step_case("pinnsf_bm", "ucy", False, pedc, obsc, slfc)
    out.update({k.replace("pinnsf_bm_eval/", "pinnsf_bm_chan/"): v for k, v in outc.items()})
    out.update({"ped_c": pedc, "obs_c": obsc, "self_c": slfc})
    save("training_step", **out)
    out = {}
    out.update(training_rollout_case("ucy_bm", H.UCY_CLIP, "pinnsf_bm", "ucy", slice(200, 206), 5))
    out.update(training_rollout_case("gc_bm_full", H.GC_CLIP, "pinnsf_bm", "gc1560", slice(300, 304), 6,
                                     reg_weight=1e-3, teacher_weight=0.5, new_collision_loss_flag=1, time_decay=0.9))
    save("training_rollout", **out)


def gen_losses():
    """f-3: the reference's own rollout-loss methods (simulators.py:172-249) called directly on seeded tensors shaped
    like a UCY / GC rollout-training batch: values with reduction 'sum' and d/d pred from the reference's autograd."""
    import types
    stub = types.SimpleNamespace(reduction=SIM.BaseSimulator.reduction)
    for name in ("multiple_rollout_mse_loss", "multiple_rollout_collision_avoidance_loss",
                 "multiple_rollout_collision_loss"):
        setattr(stub, name, types.MethodType(getattr(SIM.BaseSimulator, name), stub))
    out = {}
    for case, (C, T, N, decay, mask) in {"ucy": (8, 10, 144, 0.9, False), "gc": (6, 5, 122, 1.0, True),
                                         "tiny": (2, 1, 5, 0.5, False)}.items():
        g = torch.Generator().manual_seed(C * 1000 + T)
        wide = torch.randn(C, T, N, 12, generator=g) * 3
        pred = (wide[..., :2] + 0.3 * torch.randn(C, T, N, 2, generator=g)).clone().requires_grad_(True)
        a_pred = (wide[..., 4:6] + 0.1 * torch.randn(C, T, N, 2, generator=g)).clone().requires_grad_(True)
        coll = (torch.rand(C, T, N, generator=g) < 0.1).float() * 2
        hard = (torch.rand(C, T, N, generator=g) < 0.03).float()
        am = (torch.rand(N, generator=g) < 0.7).float() if mask else None
        labels = wide[..., :2]
        mse = stub.multiple_rollout_mse_loss(pred, labels, decay, reduction='sum')
        cl = stub.multiple_rollout_collision_loss(pred, labels, decay, 10, coll.clone(), reduction='sum',
                                                  abnormal_mask=am)
        hl = stub.multiple_rollout_collision_loss(pred, labels, decay, 10, hard.clone(), reduction='sum',
                                                  abnormal_mask=am)
        (mse + 10.0 * cl + 100.0 * hl).backward()
        amse = stub.multiple_rollout_mse_loss(a_pred, wide[..., 4:6], decay, reduction='sum', reverse=True)
        amse.backward()
        k = case + "/"
        out[k + "wide"], out[k + "pred"], out[k + "a_pred"] = wide, pred.detach(), a_pred.detach()
        out[k + "coll"], out[k + "hard"] = coll, hard
        if am is not None:
            out[k + "abnormal_mask"] = am
        out[k + "decay"] = np.float64(decay)
        out[k + "mse"], out[k + "collision"], out[k + "hard_collision"], out[k + "a_mse"] = mse, cl, hl, amse
        out[k + "g_pred"], out[k + "g_a_pred"] = pred.grad, a_pred.grad          # weights 1 / 10 / 100 and 1
    save("losses", **out)


def gen_metrics():
    """f-4: the evaluation metrics of test_multiple_rollouts (simulators.py:505-531) on the reference's own rollouts
    (golden trajectories): post_process (:443-463), then METRIC.mae / ot / mmd _with_time_mask (metrics.py:29-91) and
    METRIC.collision_count (:16-26), per frame where the reference loops over frames."""
    import functions.metrics as METRIC
    import types
    out = {}
    for name in ("rollout_gc_bm", "rollout_ucy_bm", "rollout_syn_sfm"):
        z = np.load(os.path.join(HERE, name + ".npz"))
        T = int(z["in/num_frames"])
        p_pred = torch.from_numpy(z["out/position"][:T].copy())
        pred_mask = torch.from_numpy(z["out/mask_p"][:T].copy())
        mask = torch.from_numpy(z["in/mask_p_pred"][:T].copy()).long()
        labels = torch.from_numpy(z["in/position"][:T].copy())
        stub = types.SimpleNamespace(waypoints=torch.from_numpy(z["in/waypoints"].copy()),
                                     dest_num=torch.from_numpy(z["in/dest_num"].copy()).long())
        t0 = int(z["in/t_start"])
        coll = METRIC.collision_count(p_pred[t0:].clone(), 0.5, reduction='sum')
        hard = METRIC.collision_count(p_pred[t0:].clone(), 0.25, reduction='sum')
        p_pp = SIM.BaseSimulator.post_process(stub, p_pred.clone(), pred_mask, mask)
        g = name + "/"
        out[g + "p_pred"], out[g + "labels"], out[g + "mask"] = p_pp, labels, mask
        out[g + "p_raw"], out[g + "t_start"] = p_pred, np.int64(t0)
        out[g + "collision_count"], out[g + "hard_collision_count"] = np.float64(coll), np.float64(hard)
        out[g + "mae_sum"] = np.float64(METRIC.mae_with_time_mask(p_pp, labels, mask, reduction='sum'))
        ot = METRIC.ot_with_time_mask(p_pp, labels, mask, reduction=None, dvs='cpu')
        mmd = METRIC.mmd_with_time_mask(p_pp, labels, mask, reduction=None)
        frames = [t for t in range(mask.shape[0]) if int(mask[t].sum()) > 1]
        assert len(ot) == len(frames) == len(mmd)
        out[g + "frames"] = np.asarray(frames, np.int64)
        out[g + "ot"], out[g + "mmd"] = np.asarray(ot, np.float64), np.asarray(mmd, np.float64)
        out[g + "ot_sum"] = np.float64(METRIC.ot_with_time_mask(p_pp, labels, mask, reduction='sum', dvs='cpu'))
        out[g + "mmd_sum"] = np.float64(METRIC.mmd_with_time_mask(p_pp, labels, mask, reduction='sum'))
        print(name, "frames", len(frames), "mae", out[g + "mae_sum"], "ot", out[g + "ot_sum"], "mmd", out[g + "mmd_sum"],
              "coll", coll, hard)
    save("metrics", **out)


GROUPS = {"metrics": gen_metrics, "losses": gen_losses, "features": gen_features, "models": gen_models, "mlapm": gen_mlapm, "sfm": gen_sfm,
          "rollout": gen_rollout, "sfm_rollout": gen_sfm_rollout, "training": gen_training}

if __name__ == "__main__":
    which = sys.argv[1:] or list(GROUPS)
    for gname in which:
        GROUPS[gname]()
