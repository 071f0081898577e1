"""Agent-sharded MLAPM crowd across the GPUs of one node (SURVEY.md 8e, BASELINE config 5a).

Rank g owns rows [g N/G, (g+1) N/G) and needs every agent's (position, velocity) each step -- the path's only exchange.
Instead of a separate all-gather, the finalize kernel of `piml_mlapm_advance_push_f32` stores each new row straight
into EVERY rank's next-state arrays over NVLink / NVSwitch peer memory (torch symmetric memory provides the peer
mappings), so the transfer rides on the kernel's own epilogue; a step then needs one cross-rank barrier only.

`symmetric=True` (the default for crowds of >= 16 384 agents per the library's own rule): every UNORDERED pair is
evaluated once for both rows.  Rank g then owns whole 512-agent blocks and evaluates the block pairs of its own row
blocks; the column-direction sums that belong to other ranks' agents are reduced per rank and stored into the owners'
inboxes by the pair stage (`piml_mlapm_sym_pairs_push_f32`), a barrier, and the owners' finalize kernel
(`piml_mlapm_sym_finalize_push_f32`) adds the shares in rank order and pushes the new state as above.

One process per GPU (`torchrun`), `torch.distributed` initialised with the NCCL backend.
"""
import ctypes as C

import torch
import torch.distributed as dist

from . import _lib as L


def shard_rows(N, world, rank):
    """Block partition of the agents: rank g owns rows [g N/G, (g+1) N/G)."""
    if N % world:
        raise ValueError(f"{N} agents are not divisible by {world} ranks")
    shard = N // world
    return rank * shard, (rank + 1) * shard


def allgather_state(pos_next, vel_next, pos_rows, vel_rows, group=None):
    """The exchange as a separate collective (the baseline the fused push replaces; also what a backend without peer
    memory uses): every rank contributes its rows' new positions / velocities, all ranks end with the full (N,2)
    arrays.  Works on NCCL (GPU) and gloo (CPU tests of the partition logic)."""
    if dist.get_backend(group) == "gloo":
        world = dist.get_world_size(group)
        for full, part in ((pos_next, pos_rows), (vel_next, vel_rows)):
            chunks = list(full.chunk(world, dim=0))
            dist.all_gather(chunks, part.contiguous(), group=group)
    else:
        dist.all_gather_into_tensor(pos_next, pos_rows, group=group)
        dist.all_gather_into_tensor(vel_next, vel_rows, group=group)
    return pos_next, vel_next


def allgather_rows(full, part, group=None):
    """All-gather of equally sized row blocks: rank g contributes `part` = rows [g n/G, (g+1) n/G) of `full` (n, ...).
    NCCL: one all_gather_into_tensor; gloo (CPU tests of the host logic): all_gather into row-block views."""
    if dist.get_backend(group) == "gloo":
        chunks = list(full.chunk(dist.get_world_size(group), dim=0))
        dist.all_gather(chunks, part.contiguous(), group=group)
    else:
        dist.all_gather_into_tensor(full, part.contiguous(), group=group)
    return full


class ShardedCrowd(object):
    """Double-buffered crowd state in symmetric memory: buf[parity][0] = positions (N,2), buf[parity][1] = velocities."""

    SYM_MIN_AGENTS = 16384

    def __init__(self, N, group=None, device=None, symmetric=None):
        import torch.distributed._symmetric_memory as symm
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        self.device = device if device is not None else L.cuda_device()
        self.N = N
        self.symmetric = (N >= self.SYM_MIN_AGENTS) if symmetric is None else bool(symmetric)
        if self.symmetric:
            r0, r1 = C.c_int64(), C.c_int64()
            L.check(L.load().piml_mlapm_sym_shard_rows(N, self.world, self.rank, C.byref(r0), C.byref(r1)),
                    "piml_mlapm_sym_shard_rows")
            self.rows = (int(r0.value), int(r1.value))
            self.inbox = symm.empty((int(L.load().piml_mlapm_sym_inbox_bytes(N, self.world)) // 4,),
                                    dtype=torch.float32, device=self.device)
            self.inbox_hdl = symm.rendezvous(self.inbox, self.group)
            self._inbox_tab = (C.c_uint64 * self.world)(*[int(p) for p in self.inbox_hdl.buffer_ptrs])
            self._sym_ws = torch.empty(int(L.load().piml_mlapm_sym_shard_workspace_bytes(N, self.world)),
                                       dtype=torch.uint8, device=self.device)
        else:
            self.rows = shard_rows(N, self.world, self.rank)
        self.shard = self.rows[1] - self.rows[0]
        self.buf = symm.empty((2, 2, N, 2), dtype=torch.float32, device=self.device)
        self.hdl = symm.rendezvous(self.buf, self.group)
        self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        if len(self.ptrs) != self.world:
            raise RuntimeError("symmetric memory rendezvous returned an unexpected number of peer buffers")
        # destinations of ALL agents (the column side of the symmetric gates needs them): symmetric too, so that a rank
        # can upload only its own rows and hand them to its peers (scatter_rows)
        self.dest_buf = symm.empty((N, 2), dtype=torch.float32, device=self.device)
        self.dest_hdl = symm.rendezvous(self.dest_buf, self.group)
        self._dest_tab = (C.c_uint64 * self.world)(*[int(p) for p in self.dest_hdl.buffer_ptrs])
        self.parity = 0
        self.arrived = torch.empty(self.shard, dtype=torch.uint8, device=self.device)
        plane = N * 2 * 4                                        # bytes of one (N,2) fp32 array
        self._tables = []
        for par in (0, 1):
            pos = (C.c_uint64 * self.world)(*[p + (par * 2) * plane for p in self.ptrs])
            vel = (C.c_uint64 * self.world)(*[p + (par * 2 + 1) * plane for p in self.ptrs])
            self._tables.append((pos, vel))

    def load(self, position, velocity):
        """Every rank passes the full initial state (N,2)."""
        self.buf[self.parity, 0].copy_(position)
        self.buf[self.parity, 1].copy_(velocity)
        torch.cuda.current_stream(self.device).synchronize()
        dist.barrier(self.group)

    def scatter_rows(self, position_rows, velocity_rows, destination_rows=None):
        """The host-buffer entry of a sharded step: every rank passes ONLY ITS rows [rows[0], rows[1]) (pinned host or
        device tensors): one H2D of 1/G of the state, then the rows are stored into every rank's current-state arrays
        over NVLink peer memory and a barrier makes the crowd complete everywhere.  destination_rows likewise into
        .dest_buf."""
        r0, r1 = self.rows
        dev = self.device
        stage = [L.f32c(x.to(dev, non_blocking=True) if not x.is_cuda else x) for x in (position_rows, velocity_rows)]
        dst = destination_rows
        if dst is not None:
            dst = L.f32c(dst.to(dev, non_blocking=True) if not dst.is_cuda else dst)
        pos_tab, vel_tab = self._tables[self.parity]
        L.check(L.load().piml_scatter_rows_push_f32(
            L.ptr(stage[0]), L.ptr(stage[1]), L.ptr(dst), r0, r1 - r0, self.world, pos_tab, vel_tab,
            self._dest_tab if dst is not None else None, L.stream_ptr(dev)), "piml_scatter_rows_push_f32")
        self.hdl.barrier(channel=0)

    @property
    def position(self):
        return self.buf[self.parity, 0]

    @property
    def velocity(self):
        return self.buf[self.parity, 1]

    def step(self, model, desired_speed, destination, dt, radius=0.3, trace=None):
        """One iteration of src/main_mlapm.py:18-36 for this rank's rows, exchange included.  Returns arrived[bool]
        for the local rows; afterwards .position / .velocity hold the new state of ALL agents.
        trace: optional list that receives CUDA events at the stage boundaries of this step (pairs + share push |
        barrier | finalize + state push | barrier), for per-rank timelines."""
        nxt = 1 - self.parity
        pos_tab, vel_tab = self._tables[nxt]
        ds = desired_speed if desired_speed.dim() == 2 else desired_speed.unsqueeze(-1)
        r0, r1 = self.rows

        def mark():
            if trace is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                trace.append(e)
        mark()
        if self.symmetric:
            lib, prm, st = L.load(), model._params(), L.stream_ptr(self.device)
            L.check(lib.piml_mlapm_sym_pairs_push_f32(
                L.ptr(self.position), L.ptr(self.velocity), L.ptr(destination), self.N, self.world, self.rank,
                C.byref(prm), self._inbox_tab, L.ptr(self._sym_ws), self._sym_ws.numel(), st),
                "piml_mlapm_sym_pairs_push_f32")
            mark()
            self.hdl.barrier(channel=0)    # every rank's column-direction shares have landed in the owners' inboxes
            mark()
            L.check(lib.piml_mlapm_sym_finalize_push_f32(
                L.ptr(self.position), L.ptr(self.velocity), L.ptr(ds), ds.shape[1], L.ptr(destination), self.N,
                self.world, self.rank, C.byref(prm), float(dt), float(radius), L.ptr(self.inbox), pos_tab, vel_tab,
                L.ptr(self.arrived), L.ptr(self._sym_ws), self._sym_ws.numel(), st),
                "piml_mlapm_sym_finalize_push_f32")
            mark()
            self.hdl.barrier(channel=0)    # ... and every rank's new rows in every rank's next-state arrays
            mark()
            self.parity = nxt
            return self.arrived.bool()
        L.check(L.load().piml_mlapm_advance_push_f32(
            L.ptr(self.position), L.ptr(self.velocity), L.ptr(ds), ds.shape[1], L.ptr(destination), self.N, r0, r1,
            C.byref(model._params()), float(dt), float(radius), self.world, pos_tab, vel_tab, L.ptr(self.arrived),
            L.ptr(model._workspace(self.N, self.device)), L.stream_ptr(self.device)), "piml_mlapm_advance_push_f32")
        mark()
        self.hdl.barrier(channel=0)        # every rank's rows have landed in every rank's next-state arrays
        mark()
        self.parity = nxt
        return self.arrived.bool()


class ShardedNNCrowd(object):
    """Agent-sharded NN-augmented (or pure social-force) rollout of ONE large scene (SURVEY.md 8e): the loop body of
    `get_multiple_rollouts` (simulators.py:602-652) with rank g computing rows [g N/G, (g+1) N/G).

    *Fused path* (per-slot-decoder networks the tensor-core step runs, `piml_nn_step_shard_f32`): every rank holds every
    agent's p, v, a, double-buffered in symmetric memory.  Per step a rank builds the cell list over all agents, evaluates
    features -> network -> Euler / arrival for its OWN rows in sorted (spatial) order, and the last kernel stores the new
    p, v, a of those rows into every rank's next-state arrays over NVLink peer memory; one cross-rank barrier ends the
    step.  No collective, no replicated state update; dest / dest_idx / hist_v of a row live on its owner only
    (`gather_state()` assembles them everywhere on request).

    *Three-call path* (social-force model, other networks): own-row features (`piml_state_features_rows_f32`) -> forward
    -> NCCL all-gather of the new accelerations (8 B per agent) -> the elementwise state update replicated on every rank.

    Both are bit-identical to the unsharded step sequence (`scripts/check_nn_sharded.py`)."""

    def __init__(self, model, args, N, obstacles, group=None, device=None, fused=None):
        from . import models as M
        from .sfm import SocialForce
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        self.device = device if device is not None else L.cuda_device()
        self.N, self.rows = N, shard_rows(N, self.world, self.rank)
        self.args, self.model = args, model
        self.sfm = isinstance(model, SocialForce)
        if not self.sfm:
            self.spec = model.spec if hasattr(model, "spec") else M.spec_from_module(model)
            self.packed = M.pack_device(model.state_dict(), self.spec, self.device)
            self.packed_tc = M.pack_device_tc(model.state_dict(), self.spec, self.device)
        self.obstacles = L.f32c(obstacles.to(self.device))
        self.Mo = self.obstacles.shape[-2] if self.obstacles.numel() else 0
        can_fuse = False
        if not self.sfm and self.packed_tc is not None:
            self._desc = self.spec.desc()
            can_fuse = bool(L.load().piml_nn_step_supported(C.byref(self._desc))) and self.world <= 8
        self.fused = can_fuse if fused is None else (bool(fused) and can_fuse)
        dev = self.device
        if self.fused:
            import torch.distributed._symmetric_memory as symm
            self.buf = symm.empty((2, 3, N, 2), dtype=torch.float32, device=dev)     # [parity][p | v | a]
            self.hdl = symm.rendezvous(self.buf, self.group)
            ptrs = [int(x) for x in self.hdl.buffer_ptrs]
            plane = N * 2 * 4
            self._tabs = [[(C.c_uint64 * self.world)(*[q + (par * 3 + k) * plane for q in ptrs]) for k in range(3)]
                          for par in (0, 1)]
            self.parity = 0
        else:
            n = self.rows[1] - self.rows[0]
            kp, ko = min(args.topk_ped, N), (min(args.topk_obs, self.Mo) if self.Mo else 0)
            self.ped_f, self.obs_f = torch.empty(n, kp, 6, device=dev), torch.empty(n, ko, 6, device=dev)
            self.self_f, self.dest_f = torch.empty(n, 7, device=dev), torch.empty(n, 2, device=dev)
            self.a_next = torch.empty(1, N, 2, device=dev)

    def load(self, position, velocity, acceleration, destination, dest_idx, dest_num, waypoints, desired_speed,
             hist_v=None):
        """Every rank passes the whole initial state: (N,2) x4, dest_idx / dest_num (N) int64, waypoints (D,N,2),
        desired_speed (N)."""
        dv = lambda x, dt=torch.float32: x.to(self.device, dt).contiguous()
        if self.fused:
            for k, x in enumerate((position, velocity, acceleration)):
                self.buf[self.parity, k].copy_(dv(x))
            self.dest = dv(destination)[None].clone()
        else:
            self.p, self.v, self.a, self.dest = [dv(x)[None].clone() for x in (position, velocity, acceleration,
                                                                               destination)]
        self.didx, self.dnum = dv(dest_idx, torch.int64)[None].clone(), dv(dest_num, torch.int64)[None].clone()
        self.wp, self.ds = dv(waypoints)[None].clone(), dv(desired_speed).reshape(1, self.N).clone()
        self.hist = (dv(hist_v)[None] if hist_v is not None else dv(velocity)[None]).clone()
        if self.fused:
            self._bind()
            torch.cuda.current_stream(self.device).synchronize()
            dist.barrier(self.group)
        else:
            self._features()

    # ---- fused path
    def _bind(self):
        from .features import cos_threshold
        a, r = self.args, L.NnStepArgs()
        r.desc, r.packed_tc = C.pointer(self._desc), L.ptr(self.packed_tc)
        r.has_obs, r.tau = (1 if (self.spec.has_obs and self.Mo) else 0), self.spec.tau
        r.S, r.N, r.M, r.D = 1, self.N, self.Mo, self.wp.shape[-3]
        r.kp, r.cos_p, r.thr_p = a.topk_ped, cos_threshold(a.sight_angle_ped), float(a.dist_threshold_ped)
        r.ko, r.cos_o, r.thr_o = a.topk_obs, cos_threshold(a.sight_angle_obs), float(a.dist_threshold_obs)
        r.obstacles, r.obs_per_scene = (L.ptr(self.obstacles) if self.Mo else None), 0
        r.dest_num, r.waypoints, r.desired_speed = L.ptr(self.dnum), L.ptr(self.wp), L.ptr(self.ds)
        r.dest, r.dest_idx, r.hist_v = L.ptr(self.dest), L.ptr(self.didx), L.ptr(self.hist)
        self._args = r
        self._fn = L.load().piml_nn_step_shard_f32

    @property
    def p(self):
        return self.buf[self.parity, 0][None] if self.fused else self._p

    @p.setter
    def p(self, x):
        self._p = x

    @property
    def v(self):
        return self.buf[self.parity, 1][None] if self.fused else self._v

    @v.setter
    def v(self, x):
        self._v = x

    @property
    def a(self):
        return self.buf[self.parity, 2][None] if self.fused else self._a

    @a.setter
    def a(self, x):
        self._a = x

    def gather_state(self):
        """Fused path: dest, dest_idx and hist_v of a row are kept by its owner; this assembles them on every rank."""
        if self.fused and self.world > 1:
            r0, r1 = self.rows
            for full in (self.dest, self.hist, self.didx):
                allgather_rows(full[0], full[0, r0:r1].clone(), self.group)
        return self.dest, self.didx, self.hist

    def _features(self):
        from .features import cos_threshold
        a, (r0, r1) = self.args, self.rows
        L.check(L.load().piml_state_features_rows_f32(
            L.ptr(self.p), L.ptr(self.v), L.ptr(self.a), L.ptr(self.dest), L.ptr(self.obstacles) if self.Mo else None,
            self.N, self.Mo, r0, r1, a.topk_ped, cos_threshold(a.sight_angle_ped), float(a.dist_threshold_ped),
            a.topk_obs, cos_threshold(a.sight_angle_obs), float(a.dist_threshold_obs), L.ptr(self.hist),
            L.ptr(self.ds), L.ptr(self.ped_f), L.ptr(self.obs_f) if self.Mo else None, L.ptr(self.self_f),
            L.ptr(self.dest_f), L.stream_ptr(self.device)), "piml_state_features_rows_f32")

    def step(self, dt=None, remove_on_arrival=True):
        """One rollout step; afterwards .p / .v / .a hold the new state of ALL agents on every rank."""
        from . import models as M
        from .rollout import integrate_step
        dt = float(self.args.time_unit if dt is None else dt)
        if self.fused:
            r, cur, nxt = self._args, self.buf[self.parity], 1 - self.parity
            r.p, r.v, r.a = L.ptr(cur[0]), L.ptr(cur[1]), L.ptr(cur[2])
            r.dt, r.remove_on_arrival = dt, (1 if remove_on_arrival else 0)
            tp, tv, ta = self._tabs[nxt]
            L.check(self._fn(C.byref(r), self.rows[0], self.rows[1], self.world, tp, tv, ta,
                             L.stream_ptr(self.device)), "piml_nn_step_shard_f32")
            self.hdl.barrier(channel=0)        # every rank's new rows are in every rank's next-state arrays
            self.parity = nxt
            return
        if self.sfm:
            a_own = self.model(self.ped_f, self.obs_f, self.self_f)[0]
        else:
            a_own = M.pinnsf_forward(self.spec, self.packed, self.ped_f, self.obs_f, self.self_f, need_msgs=False,
                                     packed_tc=self.packed_tc)[0]
        if self.world > 1:                   # the path's one exchange: 8 B per agent
            allgather_rows(self.a_next.view(self.N, 2), a_own, self.group)
        else:
            self.a_next.view(self.N, 2).copy_(a_own)
        integrate_step(self.p, self.v, self.a, self.a_next, self.dest, self.didx, self.dnum, self.wp, dt,
                       remove_on_arrival, hist_v=self.hist)
        self._features()
