"""The PINNSF training backward (csrc/mlp_bwd.cu) against a float64 torch-autograd reference over the net shapes the
fused forward accepts: depths up to 8 encoder and 8 decoder layers, widths on the boundaries of the register tiles
(nj_for: 16/32/64) and of the 32-row weight chunks, 1 to 128 slots per agent, empty and single-row batches, batches
that fill all 64 dW row splits, more than 2^20 slot rows, and the destination norm over channels of 1 to 1000 agents.

Gate: per tensor, max |got - ref| <= 2e-5 * max |ref|, with `ref` the float64 autograd of tests/torch_ref.py on the
same fp32 weights, inputs and dropout multipliers, and on the ReLU on/off pattern of the CUDA forward (pinned_relu).
The CPU tests at the end show that the gate rejects what a split-range or tail bug of the dW kernel, or a misapplied
dropout multiplier, would produce; and that the dW job table holds every net the forward accepts."""
import math
import os
import re
import types

import pytest
import torch

from . import torch_ref as TR
from .golden_args import base_args

TOL = 2e-5
DEV = "cuda"


def compare(got, ref):
    """name -> max |got - ref| / max |ref| (inf for a missing tensor, a shape mismatch or a non-finite error; an
    all-zero reference must be matched exactly)."""
    out = {}
    for k, r in ref.items():
        g = got.get(k)
        if g is None or tuple(g.shape) != tuple(r.shape):
            out[k] = math.inf
            continue
        if r.numel() == 0:
            out[k] = 0.0
            continue
        r = r.detach().double()
        d = float((g.detach().to(r.device, torch.float64) - r).abs().max())
        s = float(r.abs().max())
        q = d / s if s > 0 else (0.0 if d == 0 else math.inf)
        out[k] = q if math.isfinite(q) else math.inf
    return out


def failures(ratios):
    return {k: v for k, v in ratios.items() if not v <= TOL}


def make_net(kind, ew=128, dw=64, n_enc=3, n_dec=2, n_proc=16, has_obs=True, seed=666):
    from piml_b200 import models as M
    args = base_args(model=kind, dataset_name="gc1560", encoder_hidden_size=ew, processor_hidden_size=ew,
                     decoder_hidden_size=dw, encoder_hidden_layers=n_enc, processor_hidden_layers=n_proc,
                     decoder_hidden_layers=n_dec, obs_feature_dim=6 if has_obs else 0)
    torch.manual_seed(seed)
    net = M.CLASSES[kind](args)
    net.train()
    return net


def make_inputs(spec, R, kp, ko, group=0, zero_dest=(), zero_channel=None, seed=0, device="cpu"):
    """Seeded features, {0, 2} dropout multipliers and loss weights.  group > 0: (C, group, .) channelled inputs."""
    g = torch.Generator(device=device).manual_seed(seed)
    lead = (R // group, group) if group else (R,)

    def rnd(*shape):
        return torch.randn(*shape, generator=g, device=device)

    ped = rnd(*lead, kp, 6)
    if kp > 1:
        ped[..., -1, :] = 0                                       # a zero-padded slot (f(0) path)
    obs = rnd(*lead, ko, 6)
    slf = rnd(*lead, 7)
    if group:
        if zero_channel is not None:
            slf[zero_channel, :, :2] = 0                          # channel norm 0 -> 0.1, no gradient through it
    else:
        for i in zero_dest:
            if i < R:
                slf[i, :2] = 0
    dp = (torch.rand(*lead, kp, spec.pw, generator=g, device=device) > 0.5).float() * 2
    do = (torch.rand(*lead, ko, spec.pw, generator=g, device=device) > 0.5).float() * 2
    return ped, obs, slf, dp, do, g


def reference(net, kind, ped, obs, slf, dp, do, ws, device, relu=TR._relu):
    """float64 autograd of tests/torch_ref.pinnsf_forward_ref: outputs, input gradients and the gradient of every
    Linear the forward uses (a parameter the reference does not use gets a zero gradient, the CUDA path's value)."""
    from piml_b200 import models as M
    spec = net.spec
    sd = {k: v.detach().to(device, torch.float64).requires_grad_(True) for k, v in net.state_dict().items()}
    ins = [x.detach().to(device, torch.float64).requires_grad_(True) for x in (ped, obs, slf)]
    outs = TR.pinnsf_forward_ref(sd, kind, spec.tau, *ins, spec.has_obs, dp.to(device, torch.float64),
                                 do.to(device, torch.float64) if spec.has_obs else None,
                                 single_block=spec.proc_mode == 1, relu=relu)
    sum((o * w.to(device, torch.float64)).sum() for o, w in zip(outs, ws)).backward()
    res = {f"out{i}": o.detach() for i, o in enumerate(outs)}
    res["g_ped"], res["g_self"] = ins[0].grad, ins[2].grad
    if spec.has_obs:
        res["g_obs"] = ins[1].grad
    for k in M.linear_keys(spec):
        for s in (".weight", ".bias"):
            t = sd[k + s]
            res[k + s] = t.grad if t.grad is not None else torch.zeros_like(t)
    return res


def stash_relu_masks(spec, R, kp, ko, stash, lead):
    """Linear name -> (ReLU output > 0) of the CUDA forward, read from its activation stash (layout: make_splan in
    csrc/mlp_tile.cuh)."""
    off, masks = 0, {}
    n_enc, n_dec = len(spec.enc_dims) - 1, len(spec.dec_dims) - 1

    def take(rows, width, name=None, k=None):
        nonlocal off
        if name is not None and (rows or R == 0):       # R == 0: empty masks, the reference still asks
            shape = (*lead, k, width) if k else (*lead, width)
            masks[name] = stash[off:off + rows * width].view(shape) > 0
        off += (rows * width + 3) // 4 * 4

    has_obs = spec.has_obs and ko > 0
    for br, k in (("ped", kp), ("obs", ko)):
        rows = R * k if (br == "ped" or has_obs) else 0
        for l in range(n_enc):
            take(rows, spec.enc_dims[l + 1], f"{br}_encoder.mlp.{2 * l}" if l < n_enc - 1 else None, k)
        if spec.proc_mode == 1:
            take(rows, spec.pw, f"{br}_processor.resnet.0.lin.mlp.0", k)
            take(rows, spec.pw)
        drows, dk = (rows, k) if spec.kind == 0 else ((R if rows else 0), None)
        for l in range(n_dec):
            take(drows, spec.dec_dims[l + 1], f"{br}_decoder.mlp.{2 * l}" if l < n_dec - 1 else None, dk)
        if spec.kind == 1:
            take(R if rows else 0, spec.pw)
        take(drows, 2)
    if len(spec.coll_dims) > 2:
        take(R * kp, spec.coll_dims[1], "ped_collision_predictor.mlp.0", kp)
    if spec.coll_dims:
        take(R * kp, 1)
    assert off == stash.numel()
    return masks


def pinned_relu(masks):
    """ReLU whose on/off pattern is the CUDA forward's.  Where a pre-activation lies within rounding of 0, fp32 and
    float64 can take different sides, and the backward then differs by that unit's whole gradient; at 10^5 - 10^6 rows
    this happens somewhere in every run.  With the pattern pinned, the reference is the exact gradient of the function
    the kernels evaluated.  The pattern may differ from float64's only at such near-ties."""
    def relu(x, name):
        m = masks[name].to(x.device)
        if x.numel():
            xd = x.detach()
            tie = xd.abs() <= 1e-5 * float(xd.abs().max())
            assert bool(((xd > 0) == m).logical_or(tie).all()), f"{name}: ReLU pattern differs beyond near-ties"
        return x * m
    return relu


def cuda_path(net, ped, obs, slf, dp, do):
    """Train-mode forward and backward through models.pinnsf_forward_autograd (the library's kernels both ways)."""
    from piml_b200 import models as M
    spec = net.spec
    ins = [x.to(DEV).requires_grad_(True) for x in (ped, obs, slf)]
    outs = M.pinnsf_forward_autograd(net, spec, net._train_cache, ins[0], ins[1] if spec.has_obs else None, ins[2],
                                     dp.to(DEV), do.to(DEV) if spec.has_obs else None)
    return outs, ins


def run_case(kind, R, kp=6, ko=10, has_obs=True, ew=128, dw=64, n_enc=3, n_dec=2, n_proc=16, group=0,
             zero_dest=(), zero_channel=None, seed=0):
    from piml_b200 import models as M
    net = make_net(kind, ew, dw, n_enc, n_dec, n_proc, has_obs).to(DEV)
    spec = net.spec
    ped, obs, slf, dp, do, g = make_inputs(spec, R, kp, ko, group, zero_dest, zero_channel, seed, DEV)
    outs, ins = cuda_path(net, ped, obs, slf, dp, do)
    stash = outs[0].grad_fn.saved_tensors[-1]
    masks = stash_relu_masks(spec, R, kp, ko, stash, slf.shape[:-1])
    ws = [torch.randn(o.shape, generator=g, device=DEV) for o in outs]
    sum((o * w).sum() for o, w in zip(outs, ws)).backward()
    got = {f"out{i}": o.detach() for i, o in enumerate(outs)}
    got["g_ped"], got["g_obs"], got["g_self"] = ins[0].grad, ins[1].grad, ins[2].grad
    named = dict(net.named_parameters())
    used = set()
    for k in M.linear_keys(spec):
        for s in (".weight", ".bias"):
            got[k + s] = named[k + s].grad
            used.add(k + s)
    for k, p in named.items():                    # dead weights (ResDNN block 0 under 2x): no gradient at all
        if k not in used:
            assert p.grad is None, k
    ref = reference(net, kind, ped, obs, slf, dp, do, ws, DEV, pinned_relu(masks))
    return compare(got, ref), got


@pytest.fixture
def worst(request):
    """Records the ratios of a case and prints the worst one (shown with -rA)."""
    seen = {}
    yield seen.update
    if seen:
        k = max(seen, key=seen.get)
        print(f"{request.node.name}: worst error ratio {seen[k]:.3e} ({k}); gate {TOL:.0e}")


def check(worst, ratios):
    worst(ratios)
    bad = failures(ratios)
    assert not bad, bad


KINDS = ["pinnsf", "pinnsf_res", "pinnsf_bottleneck", "pinnsf_bm", "pinnsf_m"]


# ---- depth: (6,4) and (6,5) need 26 dW jobs, (8,8) up to 38 ---------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("has_obs", [True, False], ids=["obs", "no_obs"])
@pytest.mark.parametrize("n_proc", [1, 16])
@pytest.mark.parametrize("n_enc,n_dec", [(1, 1), (6, 4), (6, 5), (8, 8)])
@pytest.mark.parametrize("kind", KINDS)
def test_depth(worst, kind, n_enc, n_dec, n_proc, has_obs):
    check(worst, run_case(kind, 37, 6, 10, has_obs, n_enc=n_enc, n_dec=n_dec, n_proc=n_proc,
                          seed=n_enc * 10 + n_dec)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("n_proc", [1, 16])
@pytest.mark.parametrize("kind", KINDS)
def test_depth_beyond_the_chunk_budget_is_rejected(kind, n_proc):
    """8 + 8 layers of width 128 need more than FT_MAXCH weight chunks per branch: the forward and the backward both
    refuse the net with an error before launching anything."""
    from piml_b200 import _lib as L
    from piml_b200 import models as M
    net = make_net(kind, 128, 128, 8, 8, n_proc).to(DEV)
    spec = net.spec
    R, kp, ko = 5, 6, 10
    ped, obs, slf, dp, do, _ = make_inputs(spec, R, kp, ko, device=DEV)
    with pytest.raises(RuntimeError, match="weight chunks"):
        cuda_path(net, ped, obs, slf, dp, do)
    desc = spec.desc()
    has = 1 if spec.has_obs else 0
    stash = torch.zeros(int(L.load().piml_pinnsf_stash_floats(L.C.byref(desc), has, R, kp, ko)), device=DEV)
    wsp = torch.zeros(int(L.load().piml_pinnsf_backward_workspace_floats(L.C.byref(desc), has, R, kp, ko)), device=DEV)
    pb = M.pack_device_bwd(net.state_dict(), spec)
    g_params = torch.full((M.pack_state_dict(net.state_dict(), spec).numel(),), float("nan"), device=DEV)
    g_acc = torch.zeros(R, 2, device=DEV)
    g_ped, g_obs, g_self = torch.empty_like(ped), torch.empty_like(obs), torch.empty_like(slf)
    rc = L.load().piml_pinnsf_backward_f32(
        L.C.byref(desc), L.ptr(pb), has, spec.tau, L.ptr(ped), L.ptr(obs), L.ptr(slf), R, kp, ko, 0, L.ptr(dp),
        L.ptr(do), L.ptr(stash), L.ptr(g_acc), None, None, None, L.ptr(g_params), L.ptr(g_ped), L.ptr(g_obs),
        L.ptr(g_self), L.ptr(wsp), L.stream_ptr())
    assert rc != 0 and "weight chunks" in L.last_error()
    torch.cuda.synchronize()
    assert bool(g_params.isnan().all())                            # nothing was written


# ---- widths on the nj_for (16/32/64) and FT_KC (32-row chunk) boundaries, 128 = FT_MAXW ---------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind,ew,dw,n_proc", [
    ("pinnsf_bm", 1, 127, 16), ("pinnsf_m", 16, 1, 1), ("pinnsf", 17, 7, 16), ("pinnsf_bottleneck", 33, 32, 1),
    ("pinnsf_bm", 65, 64, 1), ("pinnsf_m", 100, 127, 16), ("pinnsf_res", 128, 7, 1), ("pinnsf_m", 128, 127, 16),
    ("pinnsf_bm", 128, 127, 1), ("pinnsf_bottleneck", 17, 1, 16)])
def test_widths(worst, kind, ew, dw, n_proc):
    check(worst, run_case(kind, 45, 6, 10, ew=ew, dw=dw, n_proc=n_proc, seed=ew * 1000 + dw)[0])


# ---- slots per agent: 128 / kp agents per tile, ragged last tiles ------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind,R,kp,ko,has_obs", [
    ("pinnsf_bm", 300, 1, 1, True), ("pinnsf_m", 300, 1, 1, True), ("pinnsf_m", 101, 5, 128, True),
    ("pinnsf", 100, 7, 1, True), ("pinnsf_bottleneck", 9, 100, 128, True), ("pinnsf_bm", 7, 128, 0, False),
    ("pinnsf_m", 50, 7, 0, False), ("pinnsf_bm", 23, 100, 7, True), ("pinnsf_m", 3, 128, 128, True)])
def test_slots(worst, kind, R, kp, ko, has_obs):
    check(worst, run_case(kind, R, kp, ko, has_obs, seed=R + kp)[0])


# ---- rows ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["pinnsf_bm", "pinnsf_m", "pinnsf"])
def test_empty_batch_gives_zero_gradients(worst, kind):
    """R = 0: no rows, every parameter gradient is exactly zero (the backward's memset path)."""
    ratios, got = run_case(kind, 0)
    for k, v in got.items():
        if v is not None and v.numel():
            assert int(torch.count_nonzero(v)) == 0, k
    check(worst, ratios)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,kp,ko", [("pinnsf_bm", 6, 10), ("pinnsf_m", 6, 10), ("pinnsf_bm", 1, 1),
                                        ("pinnsf", 128, 128)])
def test_single_row(worst, kind, kp, ko):
    check(worst, run_case(kind, 1, kp, ko, seed=kp)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["pinnsf_bm", "pinnsf_m"])
def test_all_dw_splits(worst, kind):
    """20000 agents x (6 + 10) slots: 200000 obstacle rows, so the dW kernel runs its cap of 64 row splits and every
    split of both branches holds many 32-row chunks."""
    check(worst, run_case(kind, 20000, 6, 10, seed=7)[0])


@pytest.mark.gpu
def test_more_than_2_pow_20_rows(worst):
    """8200 agents x 128 pedestrian slots = 1049600 slot rows (> 2^20): the split chunk ranges c0/c1 still cover every
    row exactly once, and 64-bit row offsets hold."""
    R, kp = 8200, 128
    assert R * kp > 1 << 20
    check(worst, run_case("pinnsf_bm", R, kp, 1, seed=11)[0])


# ---- destination term --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind,group,C", [("pinnsf_bm", 1, 40), ("pinnsf_m", 129, 3), ("pinnsf_bm", 1000, 3),
                                          ("pinnsf", 1000, 2)])
def test_channel_norm(worst, kind, group, C):
    """(C, group, 7) self features: the norm reduces over the agents of a channel (> 128 = the kernel's threads for
    129 and 1000); channel 1 has all-zero destination vectors."""
    check(worst, run_case(kind, C * group, 6, 10, group=group, zero_channel=1, seed=group)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["pinnsf_bm", "pinnsf_m"])
def test_row_norm_with_zero_destinations(worst, kind):
    check(worst, run_case(kind, 257, 6, 10, zero_dest=(0, 1, 2, 127, 128, 200, 256), seed=3)[0])


# ---- CPU: the gate rejects the mistakes a split-range, tail or dropout bug would make --------------------------------
def dw_splits(max_rows):
    """Row splits of the dW kernel (dw_splits in csrc/mlp_bwd.cu)."""
    return int(min(64, max(1, (max_rows + 127) // 128)))


def reference_dropping_rows(net, kind, inputs, ws, key, lo, hi):
    """The float64 reference with rows [lo, hi) of Linear `key` left out of that Linear's dW and db only (its output
    and every other gradient unchanged): what the dW kernel returns when it skips those rows."""
    target = None
    lin = torch.nn.functional.linear

    def linear(x, w, b=None):
        if w is not target:
            return lin(x, w, b)
        keep = torch.ones(x.numel() // x.shape[-1], 1, dtype=x.dtype)
        keep[lo:hi] = 0
        keep = keep.reshape(*x.shape[:-1], 1)
        return lin(x * keep, w) + keep * b + lin(x * (1 - keep), w.detach()) + (1 - keep) * b.detach()

    orig_ref = TR.pinnsf_forward_ref

    def forward_ref(sd, *a, **kw):
        nonlocal target
        target = sd[key + ".weight"]
        return orig_ref(sd, *a, **kw)

    saved = TR.F, TR.pinnsf_forward_ref
    TR.F, TR.pinnsf_forward_ref = types.SimpleNamespace(linear=linear), forward_ref
    try:
        return reference(net, kind, *inputs, ws, "cpu")
    finally:
        TR.F, TR.pinnsf_forward_ref = saved


@pytest.fixture(scope="module")
def mid_case():
    kind, R, kp, ko = "pinnsf_bm", 150, 6, 10
    net = make_net(kind)
    ped, obs, slf, dp, do, g = make_inputs(net.spec, R, kp, ko, seed=5)
    inputs = (ped, obs, slf, dp, do)
    with torch.no_grad():
        shapes = [o.shape for o in TR.pinnsf_forward_ref(net.state_dict(), kind, net.spec.tau, ped, obs, slf, True,
                                                         dp, do)]
    ws = [torch.randn(s, generator=g) for s in shapes]
    return net, kind, inputs, ws, reference(net, kind, *inputs, ws, "cpu"), (R, kp, ko)


def test_gate_accepts_fp32_rounding_of_the_reference(mid_case):
    _, _, _, _, ref, _ = mid_case
    assert not failures(compare({k: v.float() for k, v in ref.items()}, ref))


@pytest.mark.parametrize("key,which", [("ped_encoder.mlp.2", "chunk"), ("ped_decoder.mlp.0", "tail"),
                                       ("obs_encoder.mlp.0", "chunk"), ("ped_collision_predictor.mlp.2", "tail")])
def test_gate_rejects_a_dropped_chunk(mid_case, key, which):
    net, kind, inputs, ws, ref, (R, kp, ko) = mid_case
    rows = R * (ko if key.startswith("obs") else kp)
    nchunks = (rows + 31) // 32
    c = nchunks // 2 if which == "chunk" else nchunks - 1                  # the tail chunk is ragged: 900 = 28 * 32 + 4
    bad = failures(compare(reference_dropping_rows(net, kind, inputs, ws, key, 32 * c, min(32 * c + 32, rows)), ref))
    assert key + ".weight" in bad and key + ".bias" in bad, bad


@pytest.mark.parametrize("key", ["ped_encoder.mlp.0", "obs_decoder.mlp.2", "ped_predictor.mlp.0"])
def test_gate_rejects_a_dropped_split(mid_case, key):
    net, kind, inputs, ws, ref, (R, kp, ko) = mid_case
    nsplit = dw_splits(R * max(kp, ko))
    rows = R * (ko if key.startswith("obs") else kp)
    nchunks = (rows + 31) // 32
    s = nsplit - 1
    c0, c1 = nchunks * s // nsplit, nchunks * (s + 1) // nsplit
    assert nsplit > 1 and c1 > c0
    bad = failures(compare(reference_dropping_rows(net, kind, inputs, ws, key, 32 * c0, min(32 * c1, rows)), ref))
    assert key + ".weight" in bad, bad


@pytest.mark.parametrize("branch", ["ped", "obs"])
def test_gate_rejects_a_flipped_dropout_multiplier(mid_case, branch):
    net, kind, inputs, ws, ref, _ = mid_case
    ped, obs, slf, dp, do = inputs
    dp, do = dp.clone(), do.clone()
    m = dp if branch == "ped" else do
    m[17, 2, 5] = 2.0 - m[17, 2, 5]
    bad = failures(compare(reference(net, kind, ped, obs, slf, dp, do, ws, "cpu"), ref))
    assert bad and f"{branch}_encoder.mlp.4.weight" in bad, bad


# ---- CPU: the dW job table holds every net the forward accepts ---------------------------------------------------------
def dw_jobs(spec):
    """Jobs piml_pinnsf_backward_f32 puts into its dW table: per branch one per encoder Linear, the single processor
    block, one per decoder Linear and the predictor; then the collision head's Linears."""
    n = 0
    for _ in range(2 if spec.has_obs else 1):
        n += (len(spec.enc_dims) - 1) + spec.proc_mode + (len(spec.dec_dims) - 1) + 1
    return n + max(len(spec.coll_dims) - 1, 0)


def test_dw_job_table_holds_every_accepted_net():
    from piml_b200 import _lib as L
    from piml_b200 import models as M
    worst = 0
    for kind in M.MODEL_KINDS:
        for n_enc in range(1, 9):
            for n_dec in range(1, 9):
                for n_proc in (1, 16):
                    for has_obs in (True, False):
                        args = base_args(model=kind, encoder_hidden_layers=n_enc, decoder_hidden_layers=n_dec,
                                         processor_hidden_layers=n_proc, obs_feature_dim=6 if has_obs else 0)
                        n = dw_jobs(M.spec_from_args(kind, args))
                        assert n <= L.PINNSF_DW_JOBS, (kind, n_enc, n_dec, n_proc, has_obs, n)
                        worst = max(worst, n)
    assert worst == L.PINNSF_DW_JOBS == 2 * (8 + 1 + 8 + 1) + 2
    # nets that overflowed the earlier 24-entry table
    deep = M.spec_from_args("pinnsf_m", base_args(model="pinnsf_m", encoder_hidden_layers=6, decoder_hidden_layers=4,
                                                  processor_hidden_layers=1))
    assert dw_jobs(deep) == 26
    deep = M.spec_from_args("pinnsf_bm", base_args(model="pinnsf_bm", encoder_hidden_layers=6, decoder_hidden_layers=5))
    assert dw_jobs(deep) == 26


def test_dw_job_capacity_matches_the_kernel_source():
    from piml_b200 import _lib as L
    src = os.path.join(os.path.dirname(L.__file__), "csrc", "mlp_bwd.cu")
    with open(src) as f:
        m = re.search(r"constexpr int DW_MAX_JOBS = (\d+);", f.read())
    assert m and int(m.group(1)) == L.PINNSF_DW_JOBS
