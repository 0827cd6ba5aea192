"""Batch-sharded execution across the GPUs of one box (SURVEY.md 8e; net new, the reference has no
distributed code).

Every (n, c) plane is independent in the forward pass and in grad_input; only
``grad_weight[c, :] = sum over n and space`` couples the batch.  So: one process per GPU
(torchrun), rank r owns ``x[shard_range(N, r, G)]``, weights are replicated, there is NO data-path
collective in forward or grad_input, and exactly ONE all-reduce (sum) of the tiny ``C x dim``
grad_weight per backward -- for all shift layers of a model coalesced into a single flat buffer.
Works with any torch.distributed backend (NCCL over NVLink on the B200 box, gloo in the CPU tests).
"""
import ctypes as ct
from typing import Iterable, Optional, Tuple

import torch
import torch.distributed as dist


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, balanced [lo, hi) slice of a batch of ``n`` for ``rank`` of ``world`` (first
    ``n % world`` ranks get one extra item; ranks beyond ``n`` get an empty slice)."""
    assert 0 <= rank < world
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_batch(x: torch.Tensor, rank: Optional[int] = None, world: Optional[int] = None) -> torch.Tensor:
    rank = dist.get_rank() if rank is None else rank
    world = dist.get_world_size() if world is None else world
    lo, hi = shard_range(x.shape[0], rank, world)
    return x[lo:hi]


def _shift_weights(module_or_params) -> Iterable[torch.nn.Parameter]:
    if isinstance(module_or_params, torch.nn.Module):
        from torchshifts.modules.shifts import _Shiftnd
        return [m.weight for m in module_or_params.modules() if isinstance(m, _Shiftnd)]
    return list(module_or_params)


def allreduce_grad_weights(module_or_params, group=None, average: bool = False) -> int:
    """Sum (or average) ``weight.grad`` of every shift layer over the ranks with ONE collective.

    Returns the number of elements reduced.  Parameters without a gradient contribute zeros so
    that all ranks issue the same collective.

    The coalesced buffer has ONE dtype: fp32, which holds fp16 / bf16 / fp32 gradients exactly (mixed-precision layers
    keep fp32 weights and gradients, all-16-bit layers bf16 or fp16 ones), or fp64 when some layer has fp64 weights.
    Every piece returns to its own parameter's dtype after the sum."""
    params = [p for p in _shift_weights(module_or_params)]
    if not params:
        return 0
    wide = torch.float64 if any(p.dtype == torch.float64 for p in params) else torch.float32
    flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1).to(wide) for p in params])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    if average:
        flat /= dist.get_world_size(group)
    off = 0
    for p in params:
        n = p.numel()
        piece = flat[off:off + n].reshape(p.shape).to(p.dtype)
        if p.grad is None:
            p.grad = piece.clone()
        else:
            p.grad.copy_(piece)
        off += n
    return int(flat.numel())


def broadcast_weights(module_or_params, src: int = 0, group=None) -> None:
    """Make the replicated shift weights identical on every rank (one broadcast)."""
    params = [p for p in _shift_weights(module_or_params)]
    if not params:
        return
    flat = torch.cat([p.data.reshape(-1).to(torch.float32) for p in params])
    dist.broadcast(flat, src=src, group=group)
    off = 0
    for p in params:
        n = p.numel()
        p.data.copy_(flat[off:off + n].reshape(p.shape).to(p.dtype))
        off += n


class FusedGradWeightAllReduce:
    """grad_weight leaves the backward already summed over the ranks: the deterministic pass-2
    reduction kernel exchanges the ``C x dim`` values over NVLink peer memory itself (one 8-byte
    {epoch : value} peer store per contribution, ``ts_shift_backward_allreduce``), so the step has no
    separate collective launch at all.

    Usage (every rank, after ``init_process_group``)::

        fused = torchshifts.sharded.FusedGradWeightAllReduce()      # allocates + rendezvous
        with fused:                                                  # or fused.enable() / fused.disable()
            loss.backward()          # shift layers' weight.grad are global sums; do NOT all-reduce them again

    Contract (checked where it can be, see ``_ops._check_fused``):

    * every rank runs the same sequence of shift backward calls with the same ``C x dim`` while the mode
      is enabled (true for replicated models); a rank whose batch shard is EMPTY still takes part and
      contributes zeros (``shard_batch`` hands empty slices to ranks beyond a ragged last batch);
    * mixed-precision layers (fp16 / bf16 activations, fp32 weights) take part like any other: every contribution
      travels as fp32 and their ``grad_weight`` is fp32;
    * fp64 weights, more than ``capacity`` weight elements or tensors on another device raise instead of
      silently skipping the exchange (a rank-local skip would leave the peers waiting);
    * the call counter lives in device memory, so a step that contains the exchange can be captured in a
      CUDA graph and replayed (``torchshifts.host.GraphedShiftStep``);
    * ``timeout_s``: how long a rank waits inside the kernel for its peers.  Default 1800 s (three times the
      NCCL watchdog default): a data-loader stall, a checkpoint on rank 0 or a first-step compile must not
      kill the job.  On expiry the kernel records the call in ``self.state[128]`` and traps (the CUDA context is
      lost, like an NCCL watchdog abort); 0 waits for ever.
    * with ``DistributedDataParallel`` call :meth:`exclude_from_ddp` BEFORE wrapping the model so DDP does
      not all-reduce (and average) the shift weights a second time.

    The exchange buffer is symmetric memory (``torch.distributed._symmetric_memory``); with a single rank a
    plain device buffer is used and the protocol degenerates to a local copy."""

    STATE_WORDS = 129             # per-CTA call counters (128 CTAs of 32 outputs) + the timed-out epoch

    def __init__(self, group=None, capacity: int = 4096, device=None, timeout_s: float = 1800.0):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        assert 1 <= self.world <= 8, 'one box: at most 8 ranks'
        self.capacity = int(capacity)
        assert 1 <= self.capacity <= 4096, 'at most 4096 grad_weight elements per layer'
        self.timeout_s = float(timeout_s)
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        words = 2 * self.world * self.capacity          # uint64 {epoch : value} words, double-buffered by epoch parity
        if self.world == 1:
            self.buf = torch.zeros(words, dtype=torch.int64, device=self.device)
            ptrs = [self.buf.data_ptr()]
        else:
            import torch.distributed._symmetric_memory as symm_mem
            pg = group if group is not None else dist.group.WORLD
            with torch.cuda.device(self.device):
                self.buf = symm_mem.empty(words, dtype=torch.int64, device=self.device)
            self.buf.zero_()
            self.handle = symm_mem.rendezvous(self.buf, pg.group_name)
            ptrs = [int(p) for p in self.handle.buffer_ptrs]
            torch.cuda.synchronize(self.device)
            dist.barrier(group=group)             # every buffer is zeroed before anybody's first exchange
        self.state = torch.zeros(self.STATE_WORDS, dtype=torch.int32, device=self.device)
        self._ptrs = ptrs
        self._prev = None
        from ._cabi import PeerGroup
        pg = PeerGroup()
        pg.world, pg.rank, pg.capacity, pg.reserved = self.world, self.rank, self.capacity, 0
        pg.timeout_ns = int(self.timeout_s * 1e9)
        for p in range(self.world):
            pg.bufs[p] = self._ptrs[p]
        pg.state = self.state.data_ptr()
        self._pg = pg

    def peer_group(self):
        """ctypes ``ts_peer_group`` (constant: the call counter lives on the device)."""
        return self._pg

    def calls(self) -> int:
        """Number of exchanges this rank has run so far (reads the device counter of CTA 0)."""
        return int(self.state[0].item())

    def enable(self):
        from . import _ops
        self._prev = _ops._FUSED_ALLREDUCE
        _ops._FUSED_ALLREDUCE = self
        return self

    def disable(self):
        from . import _ops
        _ops._FUSED_ALLREDUCE = self._prev
        self._prev = None

    __enter__ = enable

    def __exit__(self, *exc):
        self.disable()
        return False

    @staticmethod
    def exclude_from_ddp(module: torch.nn.Module) -> list:
        """Tell ``DistributedDataParallel`` (call BEFORE wrapping ``module``) to leave the shift weights out of
        its gradient buckets: with the fused exchange their ``.grad`` is already the global SUM when the
        backward returns, a second bucketed all-reduce would double-count (and average) it.  Returns the
        excluded parameter names.  DDP averages, this exchange sums: divide by the world size in the
        optimiser step (or scale the loss) if the mean is wanted -- see ``ddp_sum_to_mean_hook``."""
        from torchshifts.modules.shifts import _Shiftnd
        names = [f'{name}.weight' if name else 'weight' for name, m in module.named_modules() if isinstance(m, _Shiftnd)]
        prev = list(getattr(module, '_ddp_params_and_buffers_to_ignore', []))
        torch.nn.parallel.DistributedDataParallel._set_params_and_buffers_to_ignore_for_model(module, prev + names)
        return names


def ddp_sum_to_mean_hook(module_or_params, world: Optional[int] = None):
    """Register ``post_accumulate_grad`` hooks that turn the fused exchange's SUM into DDP's MEAN for the shift
    weights (``grad /= world``), so a model whose shift weights were excluded from DDP with
    :meth:`FusedGradWeightAllReduce.exclude_from_ddp` sees the same gradients as under stock DDP.  Returns the
    hook handles."""
    world = dist.get_world_size() if world is None else int(world)
    scale = 1.0 / world

    def hook(p):
        p.grad.mul_(scale)
    return [p.register_post_accumulate_grad_hook(hook) for p in _shift_weights(module_or_params)]
