"""Physics-infused interaction networks on the CUDA path.

Mirrors of the reference's `MLP` / `ResBlock` / `ResDNN` containers and of the four PINNSF models named in
SURVEY.md 8a (reference src/models/model.py:40-119, :720-792, :1062-1135, :1138-1221, :1224-1305).  The classes
here hold their parameters under the SAME state_dict keys as the reference (so its checkpoints load unchanged, and
the same `torch.manual_seed` gives the same initial weights), but `forward` runs one fused CUDA kernel
(`piml_pinnsf_forward_f32`) instead of 9-11 addmm calls.

`forward_from_module(module, ped, obs, self)` runs the same kernel on the weights of an UNMODIFIED reference
module; piml_b200.patch uses it to drop the CUDA path in behind `model(*state_features)`.
"""

import torch
import torch.nn as nn

from . import _lib as L

MODEL_KINDS = {
    # name -> (kind, collision head input: None | 'dec' | 'proc', default tau by dataset)
    'pinnsf': (1, None),
    'pinnsf_res': (1, None),
    'pinnsf_bottleneck': (0, None),
    'pinnsf_bm': (0, 'dec'),
    'pinnsf_m': (1, 'proc'),
}


def model_tau(model, dataset_name):
    """model.py:733, :1074, :1151-1154, :1237-1240"""
    if model == 'pinnsf_bm':
        return 5 / 6 if dataset_name in {'ucy'} else 2
    if model == 'pinnsf_m':
        return 5 / 6 if dataset_name in {'ucy'} else 0.5
    return 2


class NetSpec(object):
    """Static description of one PINNSF-family network (what piml_net_desc carries)."""

    def __init__(self, enc_dims, proc_mode, dec_dims, coll_dims, kind, has_obs, tau, dropout=0.0, n_blocks=None):
        self.enc_dims, self.proc_mode, self.dec_dims = list(enc_dims), int(proc_mode), list(dec_dims)
        self.coll_dims, self.kind, self.has_obs = list(coll_dims), int(kind), bool(has_obs)
        self.tau, self.dropout = float(tau), float(dropout)
        # ResBlocks in the processor (= processor_hidden_layers): only matters for how many dropout masks the
        # reference draws per forward in train() mode (model.py:115-119, one per block, the last one applied)
        self.n_blocks = int(n_blocks) if n_blocks is not None else (1 if self.proc_mode == 1 else 16)

    @property
    def pw(self):
        return self.enc_dims[-1]

    @property
    def msg_width(self):
        return 2 if self.kind == 0 else self.pw

    def desc(self):
        d = L.NetDesc()
        d.n_enc = len(self.enc_dims) - 1
        for i, v in enumerate(self.enc_dims):
            d.enc_dims[i] = v
        d.proc_mode = self.proc_mode
        d.n_dec = len(self.dec_dims) - 1
        for i, v in enumerate(self.dec_dims):
            d.dec_dims[i] = v
        d.n_coll = max(len(self.coll_dims) - 1, 0)
        for i, v in enumerate(self.coll_dims):
            d.coll_dims[i] = v
        d.kind = self.kind
        return d


def spec_from_args(model, args):
    """Layer plan of `args.model` exactly as the reference constructors derive it from `args`."""
    if model not in MODEL_KINDS:
        raise NotImplementedError(model)
    kind, coll = MODEL_KINDS[model]
    if args.encoder_hidden_size != args.processor_hidden_size:
        raise ValueError('In ResBlock, the feature size must be equal to the hidden size!')   # model.py:104-106
    enc = [args.ped_feature_dim] + [args.encoder_hidden_size] * args.encoder_hidden_layers
    dec = [args.processor_hidden_size] + [args.decoder_hidden_size] * args.decoder_hidden_layers
    proc_mode = 0 if args.processor_hidden_layers > 1 else 1
    if proc_mode == 1 and str(getattr(args, 'activation', 'relu')).lower() != 'relu':
        # the single-block processor relu(Wx+b)+x is the only place args.activation reaches the forward
        # (model.py:1164, :76); the kernels implement ReLU
        raise NotImplementedError(f"processor activation {args.activation!r}: the CUDA path implements 'relu'")
    coll_dims = []
    if coll == 'dec':
        coll_dims = [dec[-1], dec[-1], 1]
    elif coll == 'proc':
        coll_dims = [args.processor_hidden_size, dec[-1], 1]
    return NetSpec(enc, proc_mode, dec, coll_dims, kind, args.obs_feature_dim > 0,
                   model_tau(model, getattr(args, 'dataset_name', 'ucy')), getattr(args, 'dropout', 0.0),
                   n_blocks=args.processor_hidden_layers)


def _linear_keys(spec, branch):
    """state_dict key prefixes of the Linears of one branch in forward order."""
    keys = [f"{branch}_encoder.mlp.{2 * l}" for l in range(len(spec.enc_dims) - 1)]
    if spec.proc_mode == 1:
        keys.append(f"{branch}_processor.resnet.0.lin.mlp.0")
    keys += [f"{branch}_decoder.mlp.{2 * l}" for l in range(len(spec.dec_dims) - 1)]
    keys.append(f"{branch}_predictor.mlp.0")
    return keys


def linear_keys(spec):
    keys = _linear_keys(spec, "ped") + _linear_keys(spec, "obs")
    keys += [f"ped_collision_predictor.mlp.{2 * l}" for l in range(max(len(spec.coll_dims) - 1, 0))]
    return keys


def pack_state_dict(sd, spec):
    """Concatenate the parameters the forward pass uses into ONE fp32 vector in torch's own layout: ped branch, obs
    branch, collision head; per Linear `weight` (out,in) then `bias`.  This is what piml_pinnsf_pack_f32 (and the
    oracle) take; dead weights (ResDNN block 0 when processor_hidden_layers > 1) are not included."""
    parts = []
    for k in linear_keys(spec):
        parts.append(sd[k + ".weight"].detach().to(torch.float32).contiguous().reshape(-1))
        parts.append(sd[k + ".bias"].detach().to(torch.float32).reshape(-1))
    return torch.cat(parts)


def pack_device(sd, spec, device=None):
    """Device parameter layout of the fused forward kernel (piml_pinnsf_pack_f32); call once per weight update."""
    dev = device if device is not None else L.cuda_device()
    src = pack_state_dict(sd, spec).to(dev)
    desc = spec.desc()
    n = int(L.load().piml_pinnsf_packed_floats(L.C.byref(desc)))
    if n < 0:
        raise RuntimeError(f"piml_pinnsf_packed_floats failed: {L.last_error()}")
    out = torch.empty(n, dtype=torch.float32, device=dev)
    L.check(L.load().piml_pinnsf_pack_f32(L.C.byref(desc), L.ptr(src), L.ptr(out), L.stream_ptr(dev)),
            "piml_pinnsf_pack_f32")
    return out


def pack_device_tc(sd, spec, device=None, out=None):
    """Parameter layout of the tensor-core forward (piml_pinnsf_pack_tc_f32): per Linear the tf32 hi / lo images of the
    weight as UMMA K-major core matrices, fp32 biases and predictor.  Returns None when the network cannot run on the
    tensor-core path (widths not multiples of 32, single-block processor); callers then use the FP32-pipe kernel.
    out: a contiguous, 16-byte aligned float32 CUDA tensor of at least piml_pinnsf_packed_tc_floats floats to write
    the vector into (e.g. one row of a sweep's stacked networks); default: a new tensor."""
    dev = device if device is not None else L.cuda_device()
    desc = spec.desc()
    n = int(L.load().piml_pinnsf_packed_tc_floats(L.C.byref(desc)))
    if n < 0:
        return None
    src = pack_state_dict(sd, spec).to(dev)
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=dev)
    elif out.dtype != torch.float32 or not out.is_contiguous() or out.numel() < n or out.device != torch.device(dev):
        raise ValueError(f"pack_device_tc: out must be a contiguous float32 tensor of >= {n} floats on {dev}")
    L.check(L.load().piml_pinnsf_pack_tc_f32(L.C.byref(desc), L.ptr(src), L.ptr(out), L.stream_ptr(dev)),
            "piml_pinnsf_pack_tc_f32")
    return out


def pinnsf_forward(spec, packed, ped_features, obs_features, self_features, drop_ped=None, drop_obs=None,
                   need_msgs=True, packed_tc=None):
    """Run the fused forward.  Returns the reference's list [acc, ped_msgs, (obs_msgs), (pred_collision)].
    With `packed_tc` (pack_device_tc) and a request the tensor-core kernel covers -- eval mode, no collision head
    output, messages only for the per-slot-decoder models -- the tcgen05 path runs instead of the FP32-pipe kernel."""
    dev = L.require_cuda(packed if packed is not None else packed_tc, ped_features, self_features)
    if self_features.shape[-1] != 7:
        raise AssertionError('Error: PINN model do not accept inputs of historical velocity')   # model.py:763
    ped, slf = L.f32c(ped_features), L.f32c(self_features)
    lead = slf.shape[:-1]
    R = 1
    for s in lead:
        R *= s
    kp = ped.shape[-2]
    if slf.dim() == 2:
        group = 0
    elif slf.dim() == 3:
        group = slf.shape[1]          # torch.norm(..., dim=1) on (C,N,2) reduces over agents (model.py:1206)
    else:
        raise NotImplementedError("self_features must be (N,7) or (C,N,7)")
    obs, ko = None, 0
    if spec.has_obs:
        obs = L.f32c(obs_features)
        ko = obs.shape[-2]
    acc = torch.empty(*lead, 2, dtype=torch.float32, device=dev)
    mw = spec.msg_width
    use_tc = (packed_tc is not None and drop_ped is None and drop_obs is None
              and (not need_msgs or (spec.kind == 0 and not spec.coll_dims)))
    if use_tc:
        pm = torch.empty(*lead, kp, 2, dtype=torch.float32, device=dev) if need_msgs else None
        om = torch.empty(*lead, ko, 2, dtype=torch.float32, device=dev) if (need_msgs and spec.has_obs) else None
        desc = spec.desc()
        L.check(L.load().piml_pinnsf_forward_tc_f32(
            L.C.byref(desc), L.ptr(packed_tc), 1 if spec.has_obs else 0, spec.tau, L.ptr(ped), L.ptr(obs), L.ptr(slf),
            R, kp, ko, group, L.ptr(acc), L.ptr(pm), L.ptr(om), L.stream_ptr(dev)), "piml_pinnsf_forward_tc_f32")
        out = [acc, pm]
        if spec.has_obs:
            out.append(om)
        if spec.coll_dims:
            out.append(None)
        return out
    pm = torch.empty(*lead, kp, mw, dtype=torch.float32, device=dev) if need_msgs else None
    om = torch.empty(*lead, ko, mw, dtype=torch.float32, device=dev) if (need_msgs and spec.has_obs) else None
    coll = torch.empty(*lead, kp, 1, dtype=torch.float32, device=dev) if (spec.coll_dims and need_msgs) else None
    desc = spec.desc()
    L.check(L.load().piml_pinnsf_forward_f32(
        L.C.byref(desc), L.ptr(packed), 1 if spec.has_obs else 0, spec.tau, L.ptr(ped), L.ptr(obs), L.ptr(slf), R,
        kp, ko, group, L.ptr(drop_ped), L.ptr(drop_obs), L.ptr(acc), L.ptr(pm), L.ptr(om), L.ptr(coll),
        L.stream_ptr(dev)), "piml_pinnsf_forward_f32")
    out = [acc, pm]
    if spec.has_obs:
        out.append(om)
    if spec.coll_dims:
        out.append(coll.squeeze() if coll is not None else None)      # model.py:1215 `.squeeze()`
    return out


class _PackCache(object):
    """Packed parameter vector, rebuilt only when a parameter was modified (optimizer step / load_state_dict)."""

    def __init__(self):
        self.key, self.packed = None, None

    def get(self, module, spec):
        params = [p for _, p in sorted(module.state_dict(keep_vars=True).items())]
        key = tuple((p.data_ptr(), p._version) for p in params)
        if key != self.key:
            self.packed = pack_device(module.state_dict(), spec, params[0].device)
            self.key = key
        return self.packed


def pack_device_bwd(sd, spec, device=None):
    """Backward-pass parameter layout (piml_pinnsf_pack_bwd_f32): torch's (out,in) matrices, tile-permuted columns."""
    dev = device if device is not None else L.cuda_device()
    src = pack_state_dict(sd, spec).to(dev)
    desc = spec.desc()
    n = int(L.load().piml_pinnsf_packed_bwd_floats(L.C.byref(desc)))
    if n < 0:
        raise RuntimeError(f"piml_pinnsf_packed_bwd_floats failed: {L.last_error()}")
    out = torch.empty(n, dtype=torch.float32, device=dev)
    L.check(L.load().piml_pinnsf_pack_bwd_f32(L.C.byref(desc), L.ptr(src), L.ptr(out), L.stream_ptr(dev)),
            "piml_pinnsf_pack_bwd_f32")
    return out


class _TrainPackCache(object):
    """Forward and backward packed parameter vectors for the autograd path, rebuilt when a parameter changed."""

    def __init__(self):
        self.key, self.fwd, self.bwd = None, None, None

    def get(self, module, spec):
        named = dict(module.named_parameters())
        params = []
        for k in linear_keys(spec):
            params += [named[k + ".weight"], named[k + ".bias"]]
        key = tuple((p.data_ptr(), p._version) for p in params)
        if key != self.key:
            sd = module.state_dict()
            dev = params[0].device
            self.fwd, self.bwd, self.key = pack_device(sd, spec, dev), pack_device_bwd(sd, spec, dev), key
        return params, self.fwd, self.bwd


def pinnsf_forward_autograd(module, spec, cache, ped_features, obs_features, self_features, drop_ped, drop_obs):
    """Differentiable forward: the reference's list [acc, ped_msgs, (obs_msgs), (pred_collision)] with gradients to
    the module's parameters and to the three feature tensors, through autograd.PinnsfFunction (CUDA both ways)."""
    from .autograd import PinnsfFunction
    if self_features.shape[-1] != 7:
        raise AssertionError('Error: PINN model do not accept inputs of historical velocity')   # model.py:763
    params, pf, pb = cache.get(module, spec)
    outs = list(PinnsfFunction.apply(spec, pf, pb, ped_features, obs_features if spec.has_obs else None,
                                     self_features, drop_ped, drop_obs, *params))
    if spec.coll_dims:
        outs[-1] = outs[-1].squeeze()                                                          # model.py:1215
    return outs


def _wants_grad(module, *tensors):
    if not torch.is_grad_enabled():
        return False
    return any(p.requires_grad for p in module.parameters()) or any(
        t is not None and t.requires_grad for t in tensors)


def _dropout_multipliers(spec, training, ped, obs):
    """Dropout(p) on the processor output in train() (model.py:108,118): multipliers drawn with torch's RNG in the
    reference's order (ped first, then obs) and with the reference's shapes."""
    if not training or spec.dropout <= 0:
        return None, None

    def draw(x):
        # ResDNN.forward (model.py:115-119) calls self.dropout once per block and keeps only the LAST result, so the
        # reference consumes n_blocks masks per branch: draw and discard the first n_blocks - 1 to keep torch's RNG
        # stream (the mask that is applied, and everything drawn afterwards) aligned with the reference under a seed
        ones = torch.ones(*x.shape[:-1], spec.pw, device=x.device)
        for _ in range(max(spec.n_blocks, 1) - 1):
            torch.nn.functional.dropout(ones, spec.dropout, True)
        return torch.nn.functional.dropout(ones, spec.dropout, True)
    return draw(ped), (draw(obs) if spec.has_obs else None)


# ---- containers with the reference's parameter names -------------------------------------------------------------

class MLP(nn.Module):
    """Linear+activation stack; the last activation is `output_act` (reference model.py:40-65)."""

    def __init__(self, input_size, layer_sizes, activation=nn.ReLU(), dropout=0, output_act=nn.Identity()):
        super(MLP, self).__init__()
        sizes = [input_size] + list(layer_sizes)
        layers = []
        for i in range(len(sizes) - 1):
            layers += [nn.Linear(sizes[i], sizes[i + 1]), activation if i < len(sizes) - 2 else output_act]
        self.mlp = nn.Sequential(*layers)

    def forward(self, x):
        return self.mlp(x)


class ResBlock(nn.Module):
    def __init__(self, in_dim, hidden_units, activation):
        super(ResBlock, self).__init__()
        self.lin = MLP(in_dim, hidden_units, activation, 0, activation)

    def forward(self, x):
        return self.lin(x) + x


class ResDNN(nn.Module):
    """Parameter container matching reference model.py:82-119: block 0 owns a Linear(d,d), blocks >= 1 are empty."""

    def __init__(self, input_dim, hidden_units, activation=nn.ReLU(), dropout=0):
        super(ResDNN, self).__init__()
        self.dropout = nn.Dropout(dropout)
        units = [list(h) for h in hidden_units]
        units[0] = [input_dim] + units[0]
        self.resnet = nn.ModuleList([ResBlock(h[0], h[1:], activation) for h in units])


class _PINNSFBase(nn.Module):
    """Shared constructor: creates the sub-modules in the reference's order (same RNG stream => same init)."""
    MODEL = None

    def __init__(self, args):
        super(_PINNSFBase, self).__init__()
        self.spec = spec_from_args(self.MODEL, args)
        self.tau = model_tau(self.MODEL, getattr(args, 'dataset_name', 'ucy'))
        self.ped_feature_dim = args.ped_feature_dim
        self.obs_feature_dim = args.obs_feature_dim
        self.self_feature_dim = args.self_feature_dim
        enc = [args.encoder_hidden_size for _ in range(args.encoder_hidden_layers)]
        pro = [[args.processor_hidden_size] for _ in range(args.processor_hidden_layers)]
        dec = [args.decoder_hidden_size for _ in range(args.decoder_hidden_layers)]
        act = nn.ReLU()
        self.ped_encoder = MLP(self.ped_feature_dim, enc)
        self.obs_encoder = MLP(6, enc)
        self.ped_processor = ResDNN(enc[-1], [list(h) for h in pro], act, args.dropout)
        self.obs_processor = ResDNN(enc[-1], [list(h) for h in pro], act, args.dropout)
        self.ped_decoder = MLP(pro[-1][-1], dec)
        self.obs_decoder = MLP(pro[-1][-1], dec)
        self.ped_predictor = MLP(dec[-1], [2])
        self.obs_predictor = MLP(dec[-1], [2])
        coll = MODEL_KINDS[self.MODEL][1]
        if coll == 'dec':
            self.ped_collision_predictor = MLP(dec[-1], [dec[-1], 1])
        elif coll == 'proc':
            self.ped_collision_predictor = MLP(pro[-1][-1], [dec[-1], 1])
        self._cache = _PackCache()
        self._train_cache = _TrainPackCache()

    def forward(self, ped_features, obs_features, self_features):
        dp, do = _dropout_multipliers(self.spec, self.training, ped_features, obs_features)
        if _wants_grad(self, ped_features, obs_features, self_features):
            return pinnsf_forward_autograd(self, self.spec, self._train_cache, ped_features, obs_features,
                                           self_features, dp, do)
        packed = self._cache.get(self, self.spec)
        return pinnsf_forward(self.spec, packed, ped_features, obs_features, self_features, dp, do)


class PINNSF(_PINNSFBase):
    MODEL = 'pinnsf'


class PINNSF_bottleneck(_PINNSFBase):
    MODEL = 'pinnsf_bottleneck'


class PINNSF_bottleneck_multitask(_PINNSFBase):
    MODEL = 'pinnsf_bm'


class PINNSF_multitask(_PINNSFBase):
    MODEL = 'pinnsf_m'


CLASSES = {'pinnsf': PINNSF, 'pinnsf_res': PINNSF, 'pinnsf_bottleneck': PINNSF_bottleneck,
           'pinnsf_bm': PINNSF_bottleneck_multitask, 'pinnsf_m': PINNSF_multitask}

_REF_CLASS_TO_MODEL = {'PINNSF': 'pinnsf', 'PINNSF_bottleneck': 'pinnsf_bottleneck',
                       'PINNSF_bottleneck_multitask': 'pinnsf_bm', 'PINNSF_multitask': 'pinnsf_m'}


def spec_from_module(module):
    """Derive the NetSpec from an (unmodified reference or mirror) module instance by inspecting its Linears."""
    name = _REF_CLASS_TO_MODEL.get(type(module).__name__)
    if name is None:
        raise NotImplementedError(f"no CUDA path for model class {type(module).__name__}")
    kind, coll = MODEL_KINDS[name]
    sd = module.state_dict()

    def widths(prefix):
        dims, l = [], 0
        while f"{prefix}.mlp.{2 * l}.weight" in sd:
            w = sd[f"{prefix}.mlp.{2 * l}.weight"]
            if not dims:
                dims.append(w.shape[1])
            dims.append(w.shape[0])
            l += 1
        return dims
    enc, dec = widths("ped_encoder"), widths("ped_decoder")
    n_blocks = len(module.ped_processor.resnet)
    proc_mode = 0 if n_blocks > 1 else 1
    if proc_mode == 1:
        act = module.ped_processor.resnet[0].lin.mlp[1]
        if not isinstance(act, nn.ReLU):        # an activation has no parameters: load_state_dict cannot catch this
            raise NotImplementedError(f"processor activation {type(act).__name__}: the CUDA path implements ReLU")
    coll_dims = widths("ped_collision_predictor") if coll else []
    return NetSpec(enc, proc_mode, dec, coll_dims, kind, module.obs_feature_dim > 0, module.tau,
                   module.ped_processor.dropout.p, n_blocks=n_blocks)


_MODULE_CACHES = {}


def forward_from_module(module, ped_features, obs_features, self_features):
    """CUDA forward using the weights held by `module` (a reference model or one of the mirrors above)."""
    ent = _MODULE_CACHES.get(id(module))
    if ent is None or ent[0] is not module:
        ent = (module, spec_from_module(module), _PackCache(), _TrainPackCache())
        _MODULE_CACHES[id(module)] = ent
    _, spec, cache, train_cache = ent
    dp, do = _dropout_multipliers(spec, module.training, ped_features, obs_features)
    if _wants_grad(module, ped_features, obs_features, self_features):
        return pinnsf_forward_autograd(module, spec, train_cache, ped_features, obs_features, self_features, dp, do)
    packed = cache.get(module, spec)
    return pinnsf_forward(spec, packed, ped_features, obs_features, self_features, dp, do)
