"""SyncBatchNorm (+ residual add) (+ ReLU) on the sm_100a kernels of csrc/po2_bn.cu.

The reference models place an ``nn.SyncBatchNorm`` and usually a ReLU behind every QuantizedConv2d
(models/resnet.py:38-61).  ``FusedSyncBatchNorm`` is that module -- same parameters, buffers and
``state_dict`` -- whose ``forward`` also accepts the residual and the activation of the surrounding
block so that ``relu(bn(x) + shortcut)`` is one streaming pass forward and one backward:

    forward :  bn_stats  -> [all_gather of 2C+1 statistics when world_size > 1] -> bn_apply
    backward:  bn_bwd_reduce -> [all_reduce of 2C sums]                         -> bn_bwd_apply
               (one rank, small tensors: ONE launch, po2_bn_bwd_fused)

The collective sits exactly where torch's SyncBatchNorm has it (same algebra: per-rank mean / M2 /
count combined with the parallel-variance formula; gradient of the affine parameters from local
sums).  Within one NVLink domain (<= 8 ranks) the bracketed collectives are not separate launches at
all: the producing kernel stores this rank's vector into every rank's mailbox (symmetric memory,
``PeerExchange``) and the consuming kernel waits for the R vectors -- see csrc/po2_bn.cu.  NCCL
(``PO2_BN_EXCHANGE=nccl``, larger groups, or no symmetric memory) remains the other path.  With one
rank, tensors that fit the registers of their CTAs take the forward as a single launch
(``po2_bn_fwd_fused``).  Inputs the kernels do not cover (CPU tensors, non-fp32, eval mode under
autograd, ``momentum=None``) take ``nn.SyncBatchNorm.forward`` itself followed by the add and the
activation.
"""
import ctypes
import os
import sys
from typing import Optional

import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops

_bn_workspaces = {}


def _bn_workspace(device: torch.device, C: int) -> torch.Tensor:
    """Zero-initialised scratch (ticket counters + partial sums), one per (device, stream); the
    kernels leave the counters at zero."""
    stream = torch.cuda.current_stream(device)
    key = (device.index, stream.cuda_stream)
    ws = _bn_workspaces.get(key)
    need = int(_lib.load().po2_bn_workspace_bytes(C))
    if ws is None or ws.numel() < need:
        ws = torch.zeros(max(need, 1 << 16), dtype=torch.uint8, device=device)
        _bn_workspaces[key] = ws
    return ws


def _ptr(t: Optional[torch.Tensor]):
    return t.data_ptr() if t is not None else None


# ------------------------------------------------------------------------------------------------
# peer exchange: the two SyncBatchNorm collectives done inside the kernels over NVLink stores
# ------------------------------------------------------------------------------------------------
class PeerExchange:
    """This rank's mailbox (csrc/po2_bn.cu, BnMailbox) in symmetric memory plus the host array of
    every rank's mailbox pointer as mapped here.  One per process group; at most 8 ranks."""

    def __init__(self, peers, rank: int, world: int, keepalive=None):
        self.peers = (ctypes.c_void_p * world)(*peers)
        self.rank, self.world = rank, world
        self.mailbox = peers[rank]
        self._keepalive = keepalive

    @classmethod
    def create(cls, group) -> "PeerExchange":
        import torch.distributed._symmetric_memory as symm_mem
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        dev = torch.device("cuda", torch.cuda.current_device())
        buf = symm_mem.empty(int(_lib.load().po2_bn_mailbox_bytes()), dtype=torch.uint8, device=dev)
        buf.zero_()
        # BnMailbox.timeout_s (csrc/po2_bn.cu): how long a kernel polls for a peer's values before it gives
        # up, raises the error flag and poisons its output with NaN
        buf[8:12].view(torch.int32).fill_(max(1, int(os.environ.get("PO2_BN_EXCHANGE_TIMEOUT_S", "60"))))
        handle = symm_mem.rendezvous(buf, group)
        peers = [int(p) for p in handle.buffer_ptrs]
        if len(peers) != world or peers[rank] != buf.data_ptr():
            raise RuntimeError("symmetric-memory rendezvous returned an unexpected pointer table")
        torch.cuda.synchronize(dev)
        return cls(peers, rank, world, keepalive=(buf, handle))

    def error_flag(self) -> int:
        """non-zero once a wait timed out (a peer stopped publishing); synchronises the device"""
        buf = self._keepalive[0] if self._keepalive else None
        return int(buf[4:8].view(torch.int32).item()) if buf is not None else 0

    def check(self) -> None:
        """Raise if an earlier exchange timed out.  Costs no synchronisation: each call looks at the
        flag value that an EARLIER call copied to pinned host memory, then queues the next copy.  The
        kernels themselves already made the failure loud on the device (NaN output, running statistics
        left untouched); this is what turns it into a Python exception on the host, the way a stalled
        NCCL collective would raise."""
        buf = self._keepalive[0] if self._keepalive else None
        if buf is None or torch.cuda.is_current_stream_capturing():
            return
        host = self.__dict__.get("_host_flag")
        if host is None:
            host = self.__dict__["_host_flag"] = torch.zeros(1, dtype=torch.int32).pin_memory()
            self.__dict__["_flag_event"] = None
        ev = self.__dict__["_flag_event"]
        if ev is not None:
            if not ev.query():
                return
            if int(host[0]) != 0:
                raise RuntimeError(
                    f"FusedSyncBatchNorm: a peer of rank {self.rank} stopped publishing its statistics (mailbox error "
                    f"{int(host[0])}: 1 = poll timed out after PO2_BN_EXCHANGE_TIMEOUT_S, 2 = channel barrier); the "
                    "outputs of that step are NaN and the running statistics were not updated")
        host.copy_(buf[4:8].view(torch.int32), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.__dict__["_flag_event"] = ev


_exchanges = {}


def peer_exchange_for(group) -> Optional[PeerExchange]:
    """The PeerExchange of `group`, created (collectively) on first use; None when the group spans
    more than 8 ranks, PO2_BN_EXCHANGE=nccl, or symmetric memory cannot be set up on EVERY rank (the
    ranks agree through one all_reduce, so either all use it or none does)."""
    key = id(group)
    if key in _exchanges:
        return _exchanges[key]
    ex = None
    world = dist.get_world_size(group)
    want = os.environ.get("PO2_BN_EXCHANGE", "peer") == "peer" and 1 < world <= 8
    if want:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("the first multi-rank FusedSyncBatchNorm call sets up symmetric memory and must "
                               "not happen inside a CUDA graph capture: run one eager step first")
        try:
            ex = PeerExchange.create(group)
        except Exception as e:  # noqa: BLE001 -- any failure on any rank demotes every rank to NCCL
            print(f"[po2] peer exchange unavailable on rank {dist.get_rank(group)} ({type(e).__name__}: {e}); "
                  "SyncBatchNorm statistics go through NCCL", file=sys.stderr)
            ex = None
        ok = torch.tensor([1 if ex is not None else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if ok.item() == 0:
            ex = None
        dist.barrier(group)                      # every mailbox is zeroed and mapped before anyone publishes
    _exchanges[key] = ex
    return ex


def _peer_args(exch):
    return (exch.peers, exch.rank, exch.world) if exch is not None else (None, 0, 1)


# ------------------------------------------------------------------------------------------------
# raw launchers
# ------------------------------------------------------------------------------------------------
def bn_stats_out(x: torch.Tensor, stat: torch.Tensor, exch: Optional[PeerExchange] = None) -> None:
    """stat[0:C] = mean, stat[C:2C] = sum of squared deviations, stat[2C] = B*H*W (this rank); with
    `exch` the vector is also stored into every rank's mailbox."""
    B, C = x.shape[0], x.shape[1]
    HW = x.numel() // (B * C)
    ws = _bn_workspace(x.device, C)
    ops.LAUNCHES += 1
    _lib.check(_lib.load().po2_bn_stats(x.data_ptr(), B, C, HW, stat.data_ptr(), ws.data_ptr(), ws.numel(),
                                        *_peer_args(exch), ops._stream_ptr(x.device)), "po2_bn_stats")


def bn_apply_out(x, residual, y, stats, weight, bias, running_mean, running_var, num_batches_tracked,
                 momentum, eps, relu, use_running, save_mean, save_invstd, exch=None, stats_dense=None) -> None:
    B, C = x.shape[0], x.shape[1]
    HW = x.numel() // (B * C)
    if exch is not None:
        R = exch.world
    else:
        R = 1 if stats is None else stats.numel() // (2 * C + 1)
    ops.LAUNCHES += 1
    _lib.check(_lib.load().po2_bn_apply(
        x.data_ptr(), _ptr(residual), y.data_ptr(), _ptr(stats), R, exch.mailbox if exch is not None else None,
        _ptr(stats_dense), _ptr(weight), _ptr(bias), _ptr(running_mean), _ptr(running_var),
        _ptr(num_batches_tracked), float(momentum), float(eps), int(relu), int(use_running),
        _ptr(save_mean), _ptr(save_invstd), B, C, HW, ops._stream_ptr(x.device)), "po2_bn_apply")


def bn_fwd_fused_out(x, residual, y, weight, bias, running_mean, running_var, num_batches_tracked, momentum, eps,
                     relu, save_mean, save_invstd, stats_dense, exch=None) -> bool:
    """statistics + apply in one launch (tensors that fit the registers of their CTAs); False if the
    shape is not taken"""
    if os.environ.get("PO2_BN_FUSED", "1") != "1":
        return False
    B, C = x.shape[0], x.shape[1]
    HW = x.numel() // (B * C)
    ws = _bn_workspace(x.device, C)
    rc = _lib.load().po2_bn_fwd_fused(
        x.data_ptr(), _ptr(residual), y.data_ptr(), _ptr(weight), _ptr(bias), _ptr(running_mean), _ptr(running_var),
        _ptr(num_batches_tracked), float(momentum), float(eps), int(relu), _ptr(save_mean), _ptr(save_invstd),
        _ptr(stats_dense), B, C, HW, ws.data_ptr(), ws.numel(), *_peer_args(exch), ops._stream_ptr(x.device))
    if rc == -10:
        return False
    _lib.check(rc, "po2_bn_fwd_fused")
    ops.LAUNCHES += 1
    return True


def bn_bwd_fused_out(dy, x, y, save_mean, save_invstd, weight, dgamma, dbeta, dx, dres, relu, bias=None, dy2=None) -> bool:
    """sums + apply of the backward in one launch (one rank, tensors that fit the registers of their CTAs);
    False if the shape is not taken"""
    if os.environ.get("PO2_BN_FUSED", "1") != "1" or os.environ.get("PO2_BN_FUSED_BWD", "1") != "1":
        return False
    B, C = x.shape[0], x.shape[1]
    HW = x.numel() // (B * C)
    ws = _bn_workspace(x.device, C)
    rc = _lib.load().po2_bn_bwd_fused(
        dy.data_ptr(), _ptr(dy2), x.data_ptr(), _ptr(y), save_mean.data_ptr(), save_invstd.data_ptr(), _ptr(weight), _ptr(bias),
        _ptr(dgamma), _ptr(dbeta), dx.data_ptr(), _ptr(dres), int(relu), B, C, HW, ws.data_ptr(), ws.numel(),
        ops._stream_ptr(x.device))
    if rc == -10:
        return False
    _lib.check(rc, "po2_bn_bwd_fused")
    ops.LAUNCHES += 1
    return True


def bn_bwd_reduce_out(dy, x, y, save_mean, save_invstd, sums, dgamma, dbeta, relu, exch=None, weight=None,
                      bias=None, dy2=None) -> None:
    B, C = x.shape[0], x.shape[1]
    HW = x.numel() // (B * C)
    ws = _bn_workspace(x.device, C)
    ops.LAUNCHES += 1
    _lib.check(_lib.load().po2_bn_bwd_reduce(
        dy.data_ptr(), _ptr(dy2), x.data_ptr(), _ptr(y), save_mean.data_ptr(), save_invstd.data_ptr(), _ptr(weight), _ptr(bias),
        sums.data_ptr(), _ptr(dgamma), _ptr(dbeta), int(relu), B, C, HW, ws.data_ptr(), ws.numel(), *_peer_args(exch),
        ops._stream_ptr(x.device)), "po2_bn_bwd_reduce")


def bn_bwd_apply_out(dy, x, y, save_mean, save_invstd, weight, sums, stats, dx, dres, relu, exch=None, bias=None,
                     dy2=None) -> None:
    B, C = x.shape[0], x.shape[1]
    HW = x.numel() // (B * C)
    R = stats.numel() // (2 * C + 1)
    ops.LAUNCHES += 1
    _lib.check(_lib.load().po2_bn_bwd_apply(
        dy.data_ptr(), _ptr(dy2), x.data_ptr(), _ptr(y), save_mean.data_ptr(), save_invstd.data_ptr(), _ptr(weight), _ptr(bias),
        _ptr(sums), stats.data_ptr(), R, exch.mailbox if exch is not None else None, dx.data_ptr(), _ptr(dres),
        int(relu), B, C, HW, ops._stream_ptr(x.device)), "po2_bn_bwd_apply")


# ------------------------------------------------------------------------------------------------
# autograd
# ------------------------------------------------------------------------------------------------
class _BatchNormTrain(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, residual, weight, bias, running_mean, running_var, num_batches_tracked, momentum, eps,
                relu, group, world, exch):
        x = x.contiguous()
        if residual is not None:
            residual = residual.contiguous()
        C = x.shape[1]
        with torch.cuda.device(x.device):
            stat = torch.empty(2 * C + 1, dtype=torch.float32, device=x.device)
            y = torch.empty_like(x)
            save_mean = torch.empty(C, dtype=torch.float32, device=x.device)
            save_invstd = torch.empty(C, dtype=torch.float32, device=x.device)
            fused = False
            if world == 1 or (exch is not None and os.environ.get("PO2_BN_FUSED_MULTI", "0") == "1"):
                # small tensors: statistics + apply as ONE launch.  With several ranks the kernel can do the
                # exchange inside too (verified by tools/check_sync_bn.py with PO2_BN_FUSED_MULTI=1), but its
                # CTAs then sit on the SMs waiting for the peers with the NVLink latency fully exposed:
                # measured 4.18 vs 4.07 ms per step at N=2, so the two-kernel form stays the default there
                stats = torch.empty(world, 2 * C + 1, dtype=torch.float32, device=x.device)
                fused = bn_fwd_fused_out(x, residual, y, weight, bias, running_mean, running_var, num_batches_tracked,
                                         momentum, eps, relu, save_mean, save_invstd, stats, exch if world > 1 else None)
            if fused:
                pass
            elif world > 1 and exch is not None:
                # all_gather inside the kernels: stats publishes to every rank's mailbox, apply waits for R vectors
                bn_stats_out(x, stat, exch)
                stats = torch.empty(world, 2 * C + 1, dtype=torch.float32, device=x.device)
                bn_apply_out(x, residual, y, None, weight, bias, running_mean, running_var, num_batches_tracked,
                             momentum, eps, relu, False, save_mean, save_invstd, exch=exch, stats_dense=stats)
            else:
                bn_stats_out(x, stat)
                if world > 1:
                    stats = torch.empty(world, 2 * C + 1, dtype=torch.float32, device=x.device)
                    dist.all_gather_into_tensor(stats.view(-1), stat, group=group)
                else:
                    stats = stat.view(1, -1)
                bn_apply_out(x, residual, y, stats, weight, bias, running_mean, running_var, num_batches_tracked,
                             momentum, eps, relu, False, save_mean, save_invstd)
        ctx.relu, ctx.has_res, ctx.group, ctx.world, ctx.exch = int(relu), residual is not None, group, world, exch
        # ReLU / ReLU6 mask on y; SiLU (3) recomputes its argument from x, gamma and beta instead
        ctx.save_for_backward(x, y if relu in (1, 2, True) else None, weight, save_mean, save_invstd, stats,
                              bias if int(relu) == 3 else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y, weight, save_mean, save_invstd, stats, bias = ctx.saved_tensors
        need_x, need_res, need_w, need_b = ctx.needs_input_grad[:4]
        # the gradient that came back over a skip connection (_SkipGrad) is added inside the kernels
        skipped = ctx.__dict__.pop("_po2_skip_grads", None) if hasattr(ctx, "__dict__") else None
        dy2 = None
        if skipped:
            dy2 = skipped[0].contiguous()
            for extra in skipped[1:]:
                dy2 = dy2 + extra
            if dy is None or dy2.shape != dy.shape or dy2.dtype != dy.dtype:
                dy, dy2 = (dy2 if dy is None else dy + dy2), None
        dx, dres, dgamma, dbeta = bn_backward(dy, x, y, weight, bias, save_mean, save_invstd, stats, ctx.relu,
                                              ctx.has_res and need_res, ctx.world, ctx.exch, ctx.group, dy2=dy2)
        return (dx if need_x else None, dres, dgamma if need_w else None, dbeta if need_b else None,
                None, None, None, None, None, None, None, None, None)


def bn_backward(dy, x, y, weight, bias, save_mean, save_invstd, stats, act, want_res, world=1, exch=None, group=None,
                dy2=None):
    """(dx, dres, dgamma, dbeta) of act(bn(x) + residual) in train mode from the tensors the forward saved; dy2: a second
    gradient of the output (a skip connection's), added inside the kernels"""
    dy = dy.contiguous()
    if dy2 is not None and not act and want_res:
        dy, dy2 = dy + dy2, None                                     # the residual branch gets dy itself: form it
    C = x.shape[1]
    exch = exch if world > 1 else None
    with torch.cuda.device(x.device):
        dgamma = torch.empty(C, dtype=torch.float32, device=x.device) if weight is not None else None
        dbeta = torch.empty(C, dtype=torch.float32, device=x.device) if weight is not None else None
        dx = torch.empty_like(x)
        dres = None
        if want_res:
            dres = torch.empty_like(x) if act else dy                # without the ReLU the branch gets dy itself
        # one rank, small tensor: sums + apply as ONE launch (dy / x / y read once)
        if not (world == 1 and bn_bwd_fused_out(dy, x, y, save_mean, save_invstd, weight, dgamma, dbeta, dx,
                                                dres if act else None, act, bias, dy2)):
            sums = torch.empty(2 * C, dtype=torch.float32, device=x.device)
            bn_bwd_reduce_out(dy, x, y, save_mean, save_invstd, sums, dgamma, dbeta, act, exch, weight, bias, dy2)
            if world > 1 and exch is None:
                dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
            bn_bwd_apply_out(dy, x, y, save_mean, save_invstd, weight, sums, stats, dx,
                             dres if act else None, act, exch, bias, dy2)
    return dx, dres, dgamma, dbeta


class _SkipGrad(torch.autograd.Function):
    """Identity on a tensor that a FusedSyncBatchNorm produced and that is about to be used as another norm's residual
    branch (models/resnet.py:69 ``out += self.shortcut(x)`` with the identity shortcut).  Its backward does not hand
    the skip connection's gradient to autograd -- which would add it to the conv branch's gradient with a separate
    accumulation kernel -- but leaves it at the producing norm's autograd node; that node's backward runs after all
    its consumers (autograd's dependency count covers this edge although it carries no gradient) and adds the two
    gradients inside its own kernels (dy + dy2, the same fp32 addition)."""

    @staticmethod
    def forward(ctx, t, node):
        ctx.node = node
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        ctx.node.__dict__.setdefault("_po2_skip_grads", []).append(g)      # (kept on ctx: backward may run again)
        return None, None


def _route_skip_gradient(residual: torch.Tensor) -> torch.Tensor:
    node = residual.grad_fn
    if (node is None or type(node).__name__ != "_BatchNormTrainBackward" or not hasattr(node, "__dict__")
            or os.environ.get("PO2_SKIP_GRAD", "1") != "1"):
        return residual
    return _SkipGrad.apply(residual, node)


# the norm kernels index x in 32 bits: po2_bn_* refuse 2^31 or more elements (PO2_E_SIZE)
BN_MAX_NUMEL = 2**31 - 1


def _kernel_ok(x: torch.Tensor) -> bool:
    return (x.is_cuda and x.dtype == torch.float32 and x.dim() >= 2 and 0 < x.numel() <= BN_MAX_NUMEL
            and x.shape[1] <= 4096)


ACT = {None: 0, "none": 0, "relu": 1, "relu6": 2, "silu": 3}
_ACT_FN = {0: lambda t: t, 1: F.relu, 2: F.relu6, 3: F.silu}


class FusedSyncBatchNorm(nn.SyncBatchNorm):
    """``nn.SyncBatchNorm`` whose forward can absorb the residual add and the activation that follow it.

    ``act`` ("relu", "relu6", "silu" or None) is the activation the model applies right after this norm
    -- given at construction so that an ``nn.Sequential(conv, FusedSyncBatchNorm(c, act="relu6"),
    nn.Identity())`` keeps the reference's ``state_dict`` keys -- or per call with ``relu=True``.
    SiLU runs inside the kernels forward and backward (its backward recomputes the activation's argument from x,
    gamma and beta); only SiLU behind a residual add under autograd is applied by ``F.silu`` after the norm kernel."""

    fused_residual_relu = True

    def __init__(self, num_features, eps=1e-5, momentum=0.1, affine=True, track_running_stats=True,
                 process_group=None, device=None, dtype=None, act=None):
        super().__init__(num_features, eps, momentum, affine, track_running_stats, process_group, device, dtype)
        if act not in ACT:
            raise ValueError(f"act must be one of {sorted(k for k in ACT if k)} or None")
        self.act = act

    def forward(self, input: torch.Tensor, residual: Optional[torch.Tensor] = None, relu: bool = False) -> torch.Tensor:
        act = 1 if relu else ACT[getattr(self, "act", None)]
        use_batch_stats = self.training or (self.running_mean is None and self.running_var is None)
        fast = _kernel_ok(input) and (residual is None or (residual.shape == input.shape and _kernel_ok(residual)))
        if fast and use_batch_stats and (self.momentum is not None or self.running_mean is None):
            if input.numel() // input.shape[1] <= 1:
                raise ValueError(f"Expected more than 1 value per channel when training, got input size {input.size()}")
            world, group, exch = 1, None, None
            if self.training and dist.is_available() and dist.is_initialized():
                group = self.process_group if self.process_group is not None else dist.group.WORLD
                world = dist.get_world_size(group)
                if os.environ.get("PO2_BN_EXCHANGE") == "local":     # nn.BatchNorm2d semantics: per-rank statistics
                    world = 1
                if world > 1:
                    exch = peer_exchange_for(group)
                    if exch is not None:
                        n = exch.__dict__["_calls"] = exch.__dict__.get("_calls", 0) + 1
                        if n % 64 == 0:                              # about once per ResNet-56 step
                            exch.check()
            if residual is not None and torch.is_grad_enabled() and residual.requires_grad:
                residual = _route_skip_gradient(residual)
            track = self.training and self.track_running_stats
            # SiLU's backward is in the kernels for the plain conv-norm-SiLU case; behind a residual add it stays F.silu
            kact = act if (act != 3 or residual is None) else 0
            out = _BatchNormTrain.apply(
                input, residual, self.weight, self.bias, self.running_mean if track else None,
                self.running_var if track else None, self.num_batches_tracked if track else None,
                self.momentum if self.momentum is not None else 0.0, self.eps, kact, group, world, exch)
            if track:
                # the kernels wrote the running statistics through raw pointers: bump their version counters, as
                # torch's in-place update would (fold._affine caches the eval-mode scale / shift on them)
                torch.autograd.graph.increment_version([self.running_mean, self.running_var, self.num_batches_tracked])
            return F.silu(out) if kact != act else out
        if fast and not use_batch_stats and not (torch.is_grad_enabled() and (
                input.requires_grad or (residual is not None and residual.requires_grad) or
                (self.weight is not None and self.weight.requires_grad))):
            x = input.contiguous()
            y = torch.empty_like(x)
            with torch.cuda.device(x.device):
                bn_apply_out(x, residual.contiguous() if residual is not None else None, y, None, self.weight,
                             self.bias, self.running_mean, self.running_var, None, 0.0, self.eps, act, True,
                             None, None)
            return y
        # stock path (CPU tensors, other dtypes, eval mode under autograd, cumulative-average momentum):
        # a library path, reported once per reason (an error under PO2_STRICT=1)
        why = ("CPU tensor" if not input.is_cuda else f"dtype {input.dtype}" if input.dtype != torch.float32 else
               f"{input.numel()} elements (the kernels take up to 2^31 - 1)" if input.numel() > BN_MAX_NUMEL else
               "residual of another shape/dtype" if not fast else
               "eval mode under autograd" if not use_batch_stats else "momentum=None (cumulative average)")
        ops.note_library_path("bn:" + why, f"FusedSyncBatchNorm runs nn.SyncBatchNorm's own forward: {why}")
        out = super().forward(input)
        if residual is not None:
            out = out + residual
        return _ACT_FN[act](out)
