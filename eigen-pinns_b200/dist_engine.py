"""Vertex-sharded training step: one process per GPU, torch.distributed (NCCL over NVLink) for the
three exchanges the path really has (SURVEY 8e):

  1. halo rows of U_pred before K U / M U, and of KU, MU before the backward gather
     (point-to-point, only between ranks whose vertex ranges touch);
  2. all-reduce (sum) of the packed fp64 partials [G | num | sKK | sKM | sMM] per level  -> global
     Rayleigh quotients, residual and Gram terms; every rank then finalises identically;
  3. all-reduce (sum) of the flat weight-gradient buffer before clip + Adam.

Row space of a rank, per level:  [owned rows | halo rows].  The corrector MLP simply runs over the halo
rows too (zero input features, result overwritten by the exchange), so every kernel of the single-GPU
engine is reused unchanged on rank-local CSR blocks whose columns index that row space.
"""
import os

import numpy as np
import torch
import torch.distributed as dist

from . import ops
from .engine import TrainStepEngine, FlatParams, StepConfig
from .partition import LevelPlan
from .sparse import OperatorPair


def nccl_comm_ptr(group=None):
    """ncclComm_t of this rank in `group` as an integer (what the C ABI's multi-GPU entry points take), or None when
    the group is not an NCCL group of this torch build.  The communicator is created lazily by the first collective."""
    try:
        pg = group if group is not None else dist.distributed_c10d._get_default_group()
        backend = pg._get_backend(torch.device("cuda", torch.cuda.current_device()))
        ptr = backend._comm_ptr()
        return int(ptr) if ptr else None
    except Exception:
        return None


class _StreamWork:
    """wait() makes the current stream wait for what was enqueued on the side stream (mirrors dist.Work.wait)."""

    def __init__(self, event):
        self.event = event

    def wait(self):
        torch.cuda.current_stream().wait_event(self.event)


class CabiHaloExchanger:
    """The same exchange through the C ABI (`ep_halo_exchange_f32`: gather kernel + one NCCL group of sends / receives on
    a side stream) instead of torch.distributed's batch_isend_irecv - the path a non-Python host takes.  Selected with
    EP_HALO_CABI=1; results are identical (tests/multi_gpu_check.py, mode `cabi`)."""

    def __init__(self, plan: LevelPlan, device, group=None):
        import ctypes
        self.plan, self.group = plan, group
        peers = sorted(set(plan.send) | set(plan.recv))
        send_off, recv_off, idx = [0], [0], []
        for p in peers:
            ix = plan.send.get(p, np.zeros(0, np.int64))
            idx.append(np.asarray(ix, dtype=np.int32))
            send_off.append(send_off[-1] + len(ix))
        # the halo block is laid out peer by peer in ascending peer order (partition.LevelPlan.recv: peer -> (off, cnt))
        for p in peers:
            off, cnt = plan.recv.get(p, (recv_off[-1], 0))
            assert cnt == 0 or off == recv_off[-1], "halo blocks must be contiguous in peer order"
            recv_off.append(recv_off[-1] + cnt)
        arr = lambda v: (ctypes.c_int * len(v))(*[int(x) for x in v])
        self.n_peers = len(peers)
        self._peers, self._send_off, self._recv_off = arr(peers), arr(send_off), arr(recv_off)
        self.send_idx = torch.from_numpy(np.concatenate(idx) if idx else np.zeros(0, np.int32)).to(device)
        self.n_send = send_off[-1]
        self._bufs = {}
        self.stream = torch.cuda.Stream(device=device)
        self._comm = None

    def start(self, rows, n_own):
        import ctypes
        from . import _cabi
        if self.n_peers == 0:
            return []
        if self._comm is None:
            self._comm = nccl_comm_ptr(self.group)
            if self._comm is None:
                raise _cabi.EpError("EP_HALO_CABI=1 needs an initialised NCCL process group (run one collective first)")
        k = rows.shape[1]
        assert rows.is_contiguous() and rows.dtype == torch.float32
        if k not in self._bufs:
            self._bufs[k] = torch.empty((max(self.n_send, 1), k), dtype=torch.float32, device=rows.device)
        ready = torch.cuda.Event()
        ready.record()
        self.stream.wait_event(ready)
        P = lambda t: ctypes.c_void_p(t.data_ptr())
        with torch.cuda.stream(self.stream):
            _cabi.call("ep_halo_exchange_f32", ctypes.c_void_p(self._comm), self.n_peers, self._peers, self._send_off,
                       P(self.send_idx), self._recv_off, k, P(rows), k, P(self._bufs[k]),
                       ctypes.c_void_p(rows.data_ptr() + n_own * k * 4), ctypes.c_void_p(self.stream.cuda_stream))
        done = torch.cuda.Event()
        done.record(self.stream)
        return [_StreamWork(done)]

    def exchange(self, rows, n_own):
        for w in self.start(rows, n_own):
            w.wait()
        return rows


class HaloExchanger:
    """Moves the rows listed in plan.send to their peers and receives this rank's halo block.
    gather(src_rows_tensor, idx_tensor) -> packed rows; injected so the host logic can be exercised on
    CPU tensors (gloo) in the tests while the product passes the CUDA gather kernel."""

    def __init__(self, plan: LevelPlan, device, gather, group=None):
        self.plan, self.group, self.gather = plan, group, gather
        self.send_idx = {p: torch.from_numpy(ix).to(device) for p, ix in sorted(plan.send.items())}
        self.recv = dict(sorted(plan.recv.items()))
        self._bufs = {}                     # (peer, k) -> preallocated send buffer (stable under graph capture)

    def exchange(self, rows, n_own):
        """rows: (n_own + n_halo) x k tensor; fills rows[n_own:] from the owners."""
        for w in self.start(rows, n_own):
            w.wait()
        return rows

    def start(self, rows, n_own):
        """Enqueue the exchange and return the pending work objects: kernels launched on the current stream before
        `wait()` is called on them overlap the transfer (NCCL point-to-point runs on the communicator's own stream)."""
        reqs, keep = [], []
        for p, idx in self.send_idx.items():
            key = (p, rows.shape[1])
            if key not in self._bufs:
                self._bufs[key] = torch.empty((idx.numel(), rows.shape[1]), dtype=rows.dtype, device=rows.device)
            buf = self.gather(rows, idx, self._bufs[key])
            keep.append(buf)
            reqs.append(dist.P2POp(dist.isend, buf, p, self.group))
        for p, (off, cnt) in self.recv.items():
            reqs.append(dist.P2POp(dist.irecv, rows[n_own + off:n_own + off + cnt], p, self.group))
        self._keep = keep
        return dist.batch_isend_irecv(reqs) if reqs else []


def resolve_send_lists(plan: LevelPlan, group=None):
    """Every rank tells every other rank which of its rows it needs (one all_gather of small index lists)."""
    world = dist.get_world_size(group)
    mine = {p: ids.tolist() for p, ids in plan.requests().items()}
    everyone = [None] * world
    dist.all_gather_object(everyone, mine, group=group)
    wanted = {p: np.asarray(everyone[p].get(plan.rank, []), dtype=np.int64) for p in range(world) if p != plan.rank}
    plan.set_send_lists(wanted)
    return plan


def _refuse_mode_scales(has_scales, w_smooth_corr):
    if has_scales or float(w_smooth_corr) != 0.0:
        raise NotImplementedError("the vertex-sharded step does not train per-mode scales or the smoothness of the "
                                  "correction (w_smooth_corr): they would need the halo rows of the raw corrector output "
                                  "and an all-reduce of the scale gradient; use the single-GPU TrainStepEngine")


def _refuse_dropout(p):
    if float(p) > 0.0:
        raise NotImplementedError("the vertex-sharded step does not support dropout (got %g): use the single-GPU "
                                  "TrainStepEngine, or dropout = 0.0" % float(p))


class ShardedTrainStepEngine(TrainStepEngine):
    def __init__(self, h_local, U_base_local, plans, params: FlatParams, cfg: StepConfig, lam_target=None,
                 mlp_mode="fp32", group=None, symmetric=True, pairs=None):
        dev = h_local.device
        _refuse_mode_scales(params.mode_scales is not None, cfg.w_smooth_corr)
        _refuse_dropout(cfg.dropout)
        if not symmetric:
            raise NotImplementedError("the vertex-sharded step needs symmetric K, M (FEM / tufted Laplacians): the "
                                      "transposed products of a non-symmetric operator would need a halo scatter-add")
        self.plans, self.group = plans, group
        if pairs is None:
            pairs = [OperatorPair(pl.K_local, pl.M_local, dev, assume_symmetric=symmetric) for pl in plans]
        for pair, pl in zip(pairs, plans):
            pair.n = pl.n_own
        offsets, off = [], 0
        for pl in plans:
            offsets.append(off)
            off += pl.n_own + pl.n_halo
        assert off == h_local.shape[0] == U_base_local.shape[0]
        super().__init__(h_local, U_base_local, pairs, offsets, params, cfg, lam_target, mlp_mode)
        if os.environ.get("EP_HALO_CABI") == "1":
            self.halo = [CabiHaloExchanger(pl, dev, group) for pl in plans]
        else:
            self.halo = [HaloExchanger(pl, dev, lambda rows, idx, out: ops.gather_rows(rows, idx, out=out), group) for pl in plans]
        self.overlap = True                     # interior rows while the halo is in flight
        self._grad_work = []
        # Seven small all-reduces interleaved with the backward only pay when the kernels they hide behind are long:
        # measured on 8 B200, 2 M vertices per rank (torus 16 M, k = 64): 10.29 vs 10.48 ms per step with the per-layer
        # overlap; 125 k vertices per rank (icosphere 1 M): 0.856 vs 0.795 ms - there ONE all-reduce after the backward wins.
        self.overlap_grads = self.n_mlp >= 1_000_000
        self.dCorr.zero_()                      # halo rows never receive a gradient on this rank

    def add_projection_term(self, level, P, U_coarse, w_proj):
        raise NotImplementedError("the vertex-sharded step has no projection term: it would need the rank-local rows of "
                                  "the prolongation and its transpose; use the single-GPU TrainStepEngine")

    def _mlp_rows(self):
        # single level: rows are [owned | halo], and the corrector is only needed on the owned ones (the halo rows
        # of U_pred arrive through the exchange).  Stacked levels interleave owned and halo blocks: evaluate all.
        return self.plans[0].n_own if len(self.plans) == 1 else self.n_total

    def _ext(self, buf, li):
        pl = self.plans[li]
        off = self.offsets[li]
        return buf[off:off + pl.n_own + pl.n_halo]

    def _n_global(self, li):
        return self.plans[li].n_global

    def _reduce_partials(self, li):
        dist.all_reduce(self.partials[li], group=self.group)

    def _layer_grads_ready(self, l):
        """All-reduce the [W_l | b_l] block of the flat gradient as soon as the backward has produced it: the transfers
        of the last layers overlap the kernels of the earlier ones; only layer 0's (the smallest) is exposed.  Used for
        large per-rank meshes only (see overlap_grads)."""
        if not self.overlap_grads:
            return
        a, b = self.params.layer_range[l]
        self._grad_work.append(dist.all_reduce(self.params.grad[a:b], group=self.group, async_op=True))

    def _reduce_grads(self):
        if not self._grad_work:                                   # backward ran without the hook (unit tests)
            dist.all_reduce(self.params.grad, group=self.group)
        for w in self._grad_work:
            w.wait()
        self._grad_work = []

    def loss_forward(self):
        """Per level: start the halo exchange of U_pred, apply K and M to the interior rows meanwhile, wait, apply them
        to the boundary rows; then partials -> all-reduce -> finalize exactly as on one GPU."""
        c = self.cfg
        for li, (pl, pair) in enumerate(zip(self.plans, self.pairs)):
            s = self._level_slices(li)
            U_ext = self._ext(self.U_pred, li)
            pending = self.halo[li].start(U_ext, pl.n_own)
            a, b = pl.interior if self.overlap else (0, 0)
            ops.spmm2(pair, U_ext, out_K=self.KU[s], out_M=self.MU[s], rows=(a, b))
            for w in pending:
                w.wait()
            ops.spmm2(pair, U_ext, out_K=self.KU[s], out_M=self.MU[s], rows=(0, a))
            ops.spmm2(pair, U_ext, out_K=self.KU[s], out_M=self.MU[s], rows=(b, pl.n_own))
            ops.eigen_partials(self.U_pred[s], self.KU[s], self.MU[s], out=self.partials[li])
            self._reduce_partials(li)
            ops.eigen_finalize(self.k, self._n_global(li), self.partials[li], c.w_res, c.w_orth, self.loss_acc,
                               coef=self.coefs[li], lam_out=self.lams[li], level0=(li == 0),
                               lam_target=self.lam_target, w_trace=c.w_trace, w_order=c.w_order, w_eigen=c.w_eigen,
                               overwrite=(li == 0), w_mean=c.w_mean, w_smooth=c.w_smooth)

    def loss_backward(self, scale, scale_dev=None):
        """K U and M U live side by side in one row (engine.KUMU), so their halo rows travel as ONE message; the
        gradient of the interior rows is computed while it is in flight."""
        for li, (pl, pair) in enumerate(zip(self.plans, self.pairs)):
            s = self._level_slices(li)
            pending = self.halo[li].start(self._ext(self.KUMU, li), pl.n_own)
            a, b = pl.interior if self.overlap else (0, 0)
            args = (pair, self.U_pred[s], self.KU[s], self.MU[s], self.coefs[li], scale, self.dCorr[s], scale_dev)
            ops.eigen_loss_bwd(*args, rows=(a, b))
            for w in pending:
                w.wait()
            ops.eigen_loss_bwd(*args, rows=(0, a))
            ops.eigen_loss_bwd(*args, rows=(b, pl.n_own))


def shard_rows(global_rows, plans, global_offsets):
    """Stack [owned | zero halo] blocks of every level from a stacked global array."""
    blocks = []
    for pl, goff in zip(plans, global_offsets):
        blocks.append(global_rows[goff + pl.lo:goff + pl.hi])
        blocks.append(torch.zeros((pl.n_halo, global_rows.shape[1]), dtype=global_rows.dtype, device=global_rows.device))
    return torch.cat(blocks, dim=0).contiguous()


def make_sharded_engine(gnn, x_feats, edge_index, U_base, K, M, lam_target, optimizer, rank, world, group=None):
    """Single-level helper used by bench.py: every rank holds the global arrays once at set-up, keeps its
    vertex range, and builds the rank-local engine."""
    import torch.nn as nn
    _refuse_mode_scales(hasattr(gnn.model, "mode_scales"), getattr(gnn, "w_smooth_corr", 0.0))
    _refuse_dropout(getattr(gnn, "dropout", 0.0) or 0.0)
    dev = gnn.device
    h_global = gnn.model.corrector_input(x_feats.to(dev), edge_index.to(dev))
    plan = resolve_send_lists(LevelPlan(K, M, rank, world), group)
    h_local = shard_rows(h_global, [plan], [0])
    U_local = shard_rows(U_base.to(dev), [plan], [0])
    del h_global
    linears = [m for m in gnn.model.net if isinstance(m, nn.Linear)]
    params = FlatParams.adopt(linears)
    g = optimizer.param_groups[0]
    cfg = StepConfig(lr=g['lr'], weight_decay=g['weight_decay'], corr_scale=gnn.corr_scale, w_res=gnn.w_res,
                     w_orth=gnn.w_orth, w_trace=gnn.w_trace, w_order=gnn.w_order, w_eigen=gnn.w_eigen,
                     grad_clip=gnn.grad_clip, beta1=g['betas'][0], beta2=g['betas'][1], eps=g['eps'])
    return ShardedTrainStepEngine(h_local, U_local, [plan], params, cfg, lam_target=lam_target,
                                  mlp_mode=gnn.mlp_mode, group=group)
