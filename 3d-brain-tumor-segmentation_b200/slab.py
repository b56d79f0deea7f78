"""Whole-volume inference sharded into depth slabs (BASELINE config 4; SURVEY §8e).

The reference runs `model(x, training=False, inference=True)` (/root/reference/test.py:133) on one padded
[1, 160, 192, 160, C] volume.  Here the volume is cut along D into `world` slabs whose boundaries are multiples of
2**(depth-1) (so every down/upsampling stays local); each rank runs THE SAME layer code (layers/*.py, model.py) on
its slab while a `SlabContext` reroutes the three operations whose result depends on other slabs:

  * 3x3x3 convolutions: one-slice halo exchange with the +-1 neighbours before the conv
      stride 1: (before, after) = (1, 1);  stride 2 (TF 'same' pads 0/1): (0, 1);  Conv3DTranspose: (1, 0);
      zeros at the volume ends = TF 'SAME' padding.  The conv kernels read the halo slices in place
      (`b3d_conv3d_fwd_halo`), the output holds only this slab's slices.
  * GroupNormalization (group_norm.py:83-124): its "groups" are contiguous 1/G chunks of the WHOLE flat volume
      (SURVEY F1) and do not line up with slabs => every rank reduces partial (sum, sum^2) per global chunk
      (`b3d_gn_stats` on the slab's voxel window of the volume), one all-reduce of 2*G doubles, then `b3d_gn_apply`
      on the same window.
      A channels_first model's groups are true channel groups (a fixed set of channels over every voxel of the
      volume): the slab's own `b3d_gn_channel_stats` are the partial sums, all-reduced the same way, then
      `b3d_gn_channel_apply_slab`.  Such a model takes and returns NCDHW tensors, so the drivers below cut and
      gather along dim 2 instead of dim 1.
  * channel squeeze-excitation (resnet.py:45-58): the global-average-pool sums from the pointwise conv's epilogue
      are all-reduced (F floats) and divided by the global voxel count.

Communication goes through a tiny `Comm` interface with two implementations: `DistComm` (torch.distributed: NCCL
over NVLink on the GPUs of one box, gloo in the CPU tests) and `ThreadComm` (N virtual ranks = N threads of one
process sharing one GPU; used to validate the slab arithmetic on a single-GPU box).
"""
from __future__ import annotations

import threading
from typing import List, Optional, Sequence, Tuple

import torch

_f32 = torch.float32


# ------------------------------------------------------------------------------------------ partition
def slab_bounds(depth: int, world: int, align: int = 8) -> List[Tuple[int, int]]:
    """[d0, d1) per rank: `depth // align` units dealt as evenly as possible, larger slabs first
    (160 slices, 8 ranks, align 8 -> 24,24,24,24,16,16,16,16; SURVEY §8e)."""
    if depth % align != 0:
        raise ValueError(f"depth {depth} must be a multiple of {align} (pad_to_spatial_res does that)")
    units = depth // align
    if world > units:
        raise ValueError(f"cannot cut {units} units of {align} slices into {world} slabs")
    base, extra = divmod(units, world)
    out, d = [], 0
    for r in range(world):
        n = (base + (1 if r < extra else 0)) * align
        out.append((d, d + n))
        d += n
    return out


# ------------------------------------------------------------------------------------------ communication
class Comm:
    rank: int
    world: int

    def exchange(self, send_prev, send_next, recv_prev, recv_next) -> None:
        """Neighbour exchange along the slab axis.  send_prev goes to rank-1 (arrives in its recv_next),
        send_next to rank+1 (arrives in its recv_prev).  Arguments are None where there is no neighbour or
        nothing to move; all ranks call with the same pattern."""
        raise NotImplementedError

    def all_reduce_sum(self, t: torch.Tensor) -> None:
        raise NotImplementedError

    def all_reduce_sum2(self, a: torch.Tensor, b: torch.Tensor) -> None:
        """A fp64 and a fp32 vector summed over the ranks; backends that can do so use ONE exchange."""
        self.all_reduce_sum(a)
        self.all_reduce_sum(b)

    def all_gather_cat(self, t: torch.Tensor, sizes: Sequence[int], dim: int = 1) -> torch.Tensor:
        """Concatenate the ranks' tensors (extents `sizes` along `dim`) on every rank."""
        raise NotImplementedError


def _gather_parts(t: torch.Tensor, sizes: Sequence[int], dim: int) -> List[torch.Tensor]:
    return [torch.empty(tuple(t.shape[:dim]) + (n,) + tuple(t.shape[dim + 1:]), dtype=t.dtype, device=t.device)
            for n in sizes]


class DistComm(Comm):
    """torch.distributed backend (NCCL P2P + all-reduce over NVLink/NVSwitch; gloo for the CPU tests)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)

    def exchange(self, send_prev, send_next, recv_prev, recv_next):
        d, ops_ = self.dist, []
        # receives first; every op is posted in one batch (ncclGroupStart/End) so no ordering can deadlock
        if recv_prev is not None:
            ops_.append(d.P2POp(d.irecv, recv_prev, self.rank - 1, self.group))
        if recv_next is not None:
            ops_.append(d.P2POp(d.irecv, recv_next, self.rank + 1, self.group))
        if send_prev is not None:
            ops_.append(d.P2POp(d.isend, send_prev, self.rank - 1, self.group))
        if send_next is not None:
            ops_.append(d.P2POp(d.isend, send_next, self.rank + 1, self.group))
        if ops_:
            for w in d.batch_isend_irecv(ops_):
                w.wait()

    def all_reduce_sum(self, t):
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)

    def all_gather_cat(self, t, sizes, dim=1):
        if self.world == 1:
            return t
        parts = _gather_parts(t, sizes, dim)
        self.dist.all_gather(parts, t.contiguous(), group=self.group)
        return torch.cat(parts, dim=dim)


class PeerComm(Comm):
    """NVLink peer-memory backend: every rank allocates one symmetric buffer (torch symmetric memory: cuMem allocation
    mapped into all peers of the box), boundary slices are stored straight into the neighbour's mailbox by a copy
    kernel and published / awaited with system-scope release / acquire flags; small reductions are one-kernel
    all-to-all sums (csrc/slab_comm.cu).  No NCCL call on the data path, everything is CUDA-graph capturable."""

    def __init__(self, group=None, mailbox_bytes: int = 8 << 20):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        from ._lib import lib
        self.dist = dist
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        self.mailbox_bytes = int(mailbox_bytes)
        dev = torch.device("cuda", torch.cuda.current_device())
        nbytes = int(lib.b3d_slab_sym_bytes(self.mailbox_bytes))
        self.sym = symm.empty(nbytes // 4, dtype=_f32, device=dev)
        self.sym.zero_()
        torch.cuda.synchronize()
        self.hdl = symm.rendezvous(self.sym, self.group)
        ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        self.peers = torch.tensor(ptrs, dtype=torch.int64, device=dev)
        self.prev_base = ptrs[self.rank - 1] if self.rank > 0 else 0
        self.next_base = ptrs[self.rank + 1] if self.rank < self.world - 1 else 0
        self.epoch = torch.zeros(1, dtype=torch.int64, device=dev)
        self.hseq = self.aseq = 0
        torch.cuda.synchronize()
        dist.barrier(self.group)

    def begin_forward(self):
        """Called once per forward (SlabContext.__enter__): new epoch, sequence numbers restart."""
        from . import ops
        ops._call("b3d_epoch_tick", self.epoch)
        self.hseq = self.aseq = 0

    def exchange(self, send_prev, send_next, recv_prev, recv_next):
        from . import ops
        if self.world == 1:
            return
        c = lambda t: None if t is None else t.contiguous()
        ops._call("b3d_halo_exchange", c(send_prev), c(send_next), recv_prev, recv_next, self.prev_base, self.next_base,
                  self.sym, self.epoch, self.hseq, self.mailbox_bytes)
        self.hseq += 1

    def all_reduce_sum(self, t):
        from . import ops
        if self.world == 1:
            return
        ops._call("b3d_peer_allreduce", t, self.peers, self.rank, self.sym, self.epoch, self.aseq)
        self.aseq += 1

    def all_reduce_sum2(self, a, b):
        from . import ops
        if self.world == 1:
            return
        if a.numel() * 8 + b.numel() * 4 > 2048:
            return Comm.all_reduce_sum2(self, a, b)
        ops._call("b3d_peer_allreduce2", a, b, self.peers, self.rank, self.sym, self.epoch, self.aseq)
        self.aseq += 1

    def all_gather_cat(self, t, sizes, dim=1):
        if self.world == 1:
            return t
        parts = _gather_parts(t, sizes, dim)
        self.dist.all_gather(parts, t.contiguous(), group=self.group)
        return torch.cat(parts, dim=dim)


class _ThreadShared:
    def __init__(self, world):
        self.world = world
        self.barrier = threading.Barrier(world)
        self.slots = [None] * world


class ThreadComm(Comm):
    """N virtual ranks = N threads of one process on ONE device (same CUDA stream, so program order across the
    barrier is also stream order).  Reductions add in rank order, so every rank gets bit-identical sums."""

    def __init__(self, shared: _ThreadShared, rank: int):
        self.sh, self.rank, self.world = shared, rank, shared.world

    @staticmethod
    def make(world: int) -> List["ThreadComm"]:
        sh = _ThreadShared(world)
        return [ThreadComm(sh, r) for r in range(world)]

    def exchange(self, send_prev, send_next, recv_prev, recv_next):
        sh = self.sh
        sh.slots[self.rank] = (send_prev, send_next)
        sh.barrier.wait()
        if recv_prev is not None:
            recv_prev.copy_(sh.slots[self.rank - 1][1])
        if recv_next is not None:
            recv_next.copy_(sh.slots[self.rank + 1][0])
        sh.barrier.wait()

    def all_reduce_sum(self, t):
        sh = self.sh
        sh.slots[self.rank] = t.clone()
        sh.barrier.wait()
        total = sh.slots[0].clone()
        for r in range(1, self.world):
            total += sh.slots[r]
        sh.barrier.wait()
        t.copy_(total)

    def all_gather_cat(self, t, sizes, dim=1):
        sh = self.sh
        sh.slots[self.rank] = t
        sh.barrier.wait()
        out = torch.cat([sh.slots[r] for r in range(self.world)], dim=dim)
        sh.barrier.wait()
        return out


# ------------------------------------------------------------------------------------------ context
_TLS = threading.local()


def current() -> Optional["SlabContext"]:
    return getattr(_TLS, "ctx", None)


class SlabContext:
    """Active while a rank runs the model on its slab; consulted by ops.conv3d / group_norm / block_epilogue."""

    def __init__(self, comm: Comm, depth: int, bounds: Optional[Sequence[Tuple[int, int]]] = None, align: int = 8):
        self.comm = comm
        self.depth = int(depth)                       # D of the whole (padded) volume at level 0
        self.bounds = list(bounds) if bounds is not None else slab_bounds(depth, comm.world, align)
        self.d0, self.d1 = self.bounds[comm.rank]
        self.local_depth = self.d1 - self.d0
        self.stats = {"halo_exchanges": 0, "halo_bytes": 0, "all_reduces": 0, "halo_copies": 0}
        self._padded = {}        # data_ptr of an activation -> the [1, Dl+2, H, W, C] buffer it is the interior of
        # P16 form (the default): activations between layers are 16-bit twins [1, Dl, H, C/8, W, 8] allocated between
        # two spare depth slices, the convs read them through TMA, GroupNorm statistics come out of the conv epilogues
        # as partial sums and are all-reduced together with the SE pooling sums.  `p16` = the twin dtype or None.
        self.p16 = None
        self._halo_done = {}     # data_ptr of a P16 activation -> set of halo sides already received
        self._arena, self._arena_used, self._arena_dev = None, 0, None
        self._pending = []       # partial sums (fp64 statistics, fp32 pooling sums) awaiting their all-reduce

    def __enter__(self):
        from . import ops
        self._prev = current()
        _TLS.ctx = self
        if hasattr(self.comm, "begin_forward"):
            self.comm.begin_forward()
        self.p16 = None
        self._arena_used = 0
        if ops.P16["on"] and ops.USE_TC["on"]:
            self.p16 = ops._TWIN_DT.get(ops.get_conv_precision()[0])
        return self

    def __exit__(self, *a):
        _TLS.ctx = self._prev
        self._padded.clear()
        self._halo_done.clear()
        if a[0] is None and self._pending:
            self._pending = []
            raise RuntimeError("slab: partial sums were left without their all-reduce")
        self._pending = []

    def new_activation(self, shape, like: torch.Tensor) -> torch.Tensor:
        """Allocate an activation [1, Dl, H, W, C] as the interior of a buffer with one spare depth slice on each
        side, so that a later halo exchange needs no copy: the neighbours' slices are received in place."""
        shape = tuple(int(v) for v in shape)
        parent = torch.empty((1, shape[1] + 2) + shape[2:], dtype=like.dtype, device=like.device)
        view = parent[:, 1:shape[1] + 1]
        self._padded[view.data_ptr()] = parent
        return view

    # ---- geometry of a local tensor [1, Dl, H, W, C]: which level it is at, its offset in the whole volume
    def _level(self, dl: int) -> int:
        lvl, d = 0, self.local_depth
        while d != dl:
            if d < dl or d % 2:
                raise ValueError(f"slab: a tensor with {dl} depth slices is not a level of a {self.local_depth}-slice slab")
            d //= 2
            lvl += 1
        return lvl

    def geometry(self, x: torch.Tensor):
        """-> (first global depth slice, global depth) at x's resolution level."""
        if x.shape[0] != 1:
            raise ValueError("slab inference handles one volume (batch 1) at a time")
        lvl = self._level(x.shape[1])
        return self.d0 >> lvl, self.depth >> lvl

    def global_voxels(self, x: torch.Tensor) -> int:
        _, dg = self.geometry(x)
        return dg * x.shape[2] * x.shape[3]

    # ---- halo exchange
    def with_halo(self, x: torch.Tensor, before: int, after: int) -> torch.Tensor:
        """[1, Dl, H, W, C] -> [1, before + Dl + after, H, W, C] with the neighbours' boundary slices (zeros at the
        ends of the volume)."""
        c = self.comm
        dl = x.shape[1]
        parent = self._padded.get(x.data_ptr())
        if parent is not None and tuple(parent.shape) == (1, dl + 2) + tuple(x.shape[2:]) and x.is_contiguous():
            pad = parent[:, 1 - before:1 + dl + after]          # in place: x already sits between its halo slices
        else:
            pad = torch.empty((1, before + dl + after) + tuple(x.shape[2:]), dtype=x.dtype, device=x.device)
            pad[:, before:before + dl].copy_(x)
            self.stats["halo_copies"] += 1
        has_prev, has_next = c.rank > 0, c.rank < c.world - 1
        if before and not has_prev:
            pad[:, :before].zero_()
        if after and not has_next:
            pad[:, before + dl:].zero_()
        send_prev = x[:, :after] if (after and has_prev) else None             # my first slices = prev's "after" halo
        send_next = x[:, dl - before:] if (before and has_next) else None      # my last slices = next's "before" halo
        recv_prev = pad[:, :before] if (before and has_prev) else None
        recv_next = pad[:, before + dl:] if (after and has_next) else None
        c.exchange(send_prev, send_next, recv_prev, recv_next)
        self.stats["halo_exchanges"] += 1
        self.stats["halo_bytes"] += sum(t.numel() * 4 for t in (send_prev, send_next) if t is not None)
        return pad

    # ---- P16 activations
    def new_p16(self, shape5, like: torch.Tensor) -> torch.Tensor:
        """P16 twin [1, Dl, H, C/8, W, 8] of a local activation, allocated between two spare depth slices (the halo
        slices are received in place; at the ends of the volume the operand handed to the conv simply ends there and
        the loaders' zero fill is TF's 'SAME' padding, as in the un-sharded forward)."""
        _, dl, H, W_, C = (int(v) for v in shape5)
        parent = torch.empty((1, dl + 2, H, C // 8, W_, 8), dtype=self.p16, device=like.device)
        view = parent[:, 1:dl + 1]
        self._padded[view.data_ptr()] = parent
        self._halo_done[view.data_ptr()] = set()
        return view

    def with_halo_p16(self, t: torch.Tensor, before: int, after: int) -> torch.Tensor:
        """[1, Dl, H, C/8, W, 8] -> (the window of its buffer that includes the halo slices a neighbour provides, halo
        slices before, after), after receiving those that have not been received yet (a tensor read by two 3x3x3-type
        convs is exchanged once)."""
        c = self.comm
        dl = t.shape[1]
        parent = self._padded.get(t.data_ptr())
        if parent is None or tuple(parent.shape) != (1, dl + 2) + tuple(t.shape[2:]):
            raise RuntimeError("slab: a P16 operand that was not allocated by the slab context")
        done = self._halo_done[t.data_ptr()]
        need_b, need_a = bool(before) and "b" not in done, bool(after) and "a" not in done
        has_prev, has_next = c.rank > 0, c.rank < c.world - 1
        if (need_b or need_a) and c.world > 1:
            f = lambda v: v.view(_f32)
            send_prev = f(t[:, :1]) if (need_a and has_prev) else None          # my first slice = prev's "after" halo
            send_next = f(t[:, dl - 1:]) if (need_b and has_next) else None     # my last slice = next's "before" halo
            recv_prev = f(parent[:, :1]) if (need_b and has_prev) else None
            recv_next = f(parent[:, dl + 1:]) if (need_a and has_next) else None
            c.exchange(send_prev, send_next, recv_prev, recv_next)
            self.stats["halo_exchanges"] += 1
            self.stats["halo_bytes"] += sum(v.numel() * 4 for v in (send_prev, send_next) if v is not None)
        if need_b:
            done.add("b")
        if need_a:
            done.add("a")
        b_eff, a_eff = (before if has_prev else 0), (after if has_next else 0)
        return parent[:, 1 - b_eff:1 + dl + a_eff], b_eff, a_eff

    def arena(self, n: int, dtype) -> torch.Tensor:
        """n zero-initialised values (fp64 statistics / fp32 pooling sums) for a conv epilogue to accumulate into:
        slices of one buffer that is cleared ONCE per forward instead of a memset node per conv."""
        if self._arena is None:
            self._arena = torch.empty(8192, dtype=torch.float64, device=self._arena_dev)
            self._arena_used = 0
        if self._arena_used == 0:
            from . import ops
            ops._call("b3d_zero", self._arena.view(_f32))
        words = n if dtype == torch.float64 else (n + 1) // 2
        if self._arena_used + words > self._arena.numel():
            return None
        t = self._arena[self._arena_used:self._arena_used + words]
        self._arena_used += words
        return t if dtype == torch.float64 else t.view(_f32)[:n]

    def flush(self):
        """All-reduce the pending partial sums: a fp64 vector and a fp32 vector share one exchange."""
        p, self._pending = self._pending, []
        f64 = [t for t in p if t.dtype == torch.float64]
        f32 = [t for t in p if t.dtype != torch.float64]
        while f64 and f32:
            self.comm.all_reduce_sum2(f64.pop(0), f32.pop(0))
            self.stats["all_reduces"] += 1
        for t in f64 + f32:
            self.comm.all_reduce_sum(t)
            self.stats["all_reduces"] += 1

    def _conv3d_p16(self, srcs, w, bias, stride, transposed, act, want_gap, gn_groups, before, after):
        from . import ops
        dl, H, W_ = srcs[0].shape[1], srcs[0].shape[2], srcs[0].shape[4]
        xin, b_eff, a_eff = list(srcs), 0, 0
        if before + after:
            wins = [self.with_halo_p16(t, before, after) for t in srcs]
            xin, b_eff, a_eff = [w_[0] for w_ in wins], wins[0][1], wins[0][2]
        if transposed:
            cout, od = w.shape[3], (2 * dl, 2 * H, 2 * W_)
        else:
            cout = w.shape[4]
            od = (dl, H, W_) if stride == 1 else (dl // 2, H // 2, W_ // 2)
        y = torch.empty((1,) + od + (cout,), dtype=_f32, device=w.device)
        g0, dg = self.geometry(y)
        hw = od[1] * od[2]
        self._arena_dev = w.device
        stats = gap = None
        pre = 1
        if gn_groups and cout % gn_groups == 0 and (dg * hw) % gn_groups == 0:
            stats = self.arena(2 * gn_groups, torch.float64)
            if stats is None:
                stats, pre = torch.empty(2 * gn_groups, dtype=torch.float64, device=w.device), 0
            stats = stats.view(1, gn_groups, 2)
        if want_gap:
            gap = self.arena(cout, _f32) if pre else None
            if gap is None:
                if stats is not None and pre:          # mixed: let the ABI clear both
                    stats.zero_()
                gap, pre = torch.empty(cout, dtype=_f32, device=w.device), 0
            gap = gap.view(1, cout)
        wp = ops.pack_weights(w, False, stride, transposed)
        ops._call("b3d_conv3d_fwd_p16_slab", *ops._pad4(xin), w, bias, y, stride, int(transposed), int(act), b_eff, a_eff,
                  stats, gn_groups or 1, g0 * hw, dg * hw, gap, wp, pre)
        for t in (stats, gap):
            if t is not None:
                self._pending.append(t)
        return y, stats, gap

    def block_epilogue(self, res, h2, stats2, gamma2, beta2, wsp, gap_sum, w1, w2, groups, eps, keep_f32):
        """BlockEpilogueFn.forward for one slab in the P16 form (ops.block_epilogue routes here)."""
        from . import ops
        self.flush()
        F = res.shape[-1]
        R = w1.shape[1]
        hidden, chse = torch.empty((1, R), dtype=_f32, device=res.device), torch.empty((1, F), dtype=_f32, device=res.device)
        ops._call("b3d_se_fc_fwd", gap_sum, w1, w2, hidden, chse, 1.0 / self.global_voxels(res))
        has_gn = stats2 is not None
        out16 = self.new_p16(res.shape, res)
        out = torch.empty_like(res) if keep_f32 else None
        g0, dg = self.geometry(res)
        hw = res.shape[2] * res.shape[3]
        ops._call("b3d_block_epilogue_fwd", res.contiguous(), ops.materialize(h2), stats2,
                  gamma2 if has_gn else None, beta2 if has_gn else None, wsp.reshape(F), chse, out, out16, None, groups,
                  float(eps), int(has_gn), g0 * hw, dg * hw)
        if out is None:
            return ops.virtual(res.shape, res, [out16], None)
        ops._attach(out, out16, None)
        return out

    # ---- the three rerouted operations (forward only)
    def conv3d(self, x, w, bias, stride, transposed, act, want_gap, gn_groups=0):
        from . import ops
        k = w.shape[0]
        if k == 1:
            before = after = 0
        elif transposed:
            before, after = 1, 0
        elif stride == 2:
            before, after = 0, 1
        else:
            before, after = 1, 1
        srcs = ops.sources(x)
        if (self.p16 is not None and srcs is not None and len(srcs) <= 4 and all(t.dtype == self.p16 for t in srcs)
                and (not act or stride == 1) and ops.tc_supported(w, stride, transposed, False)):
            return self._conv3d_p16(srcs, w, bias, stride, transposed, act, want_gap, gn_groups, before, after)
        x = ops.materialize(x)
        ops._check(x)
        _, dl, H, W_, _ = x.shape
        xin = self.with_halo(x, before, after) if before + after else x
        if transposed:
            cout, od = w.shape[3], (2 * dl, 2 * H, 2 * W_)
        else:
            cout = w.shape[4]
            od = (dl, H, W_) if stride == 1 else (dl // 2, H // 2, W_ // 2)
        y = torch.empty((1,) + od + (cout,), dtype=_f32, device=x.device)
        gap = torch.empty((1, cout), dtype=_f32, device=x.device) if want_gap else None
        wp = None
        if ops.USE_TC["on"] and (not act or stride == 1) and ops.tc_supported(w, stride, transposed, False):
            wp = ops.pack_weights(w, False, stride, transposed)
        ops._call("b3d_conv3d_fwd_halo", xin, w, bias, y, stride, int(transposed), int(act), before, after, gap, wp)
        if gap is not None:
            self.comm.all_reduce_sum(gap)
            self.stats["all_reduces"] += 1
        return y, None, gap

    def group_norm(self, x, gamma, beta, groups, eps, relu, stats=None, operand_only=False):
        from . import ops
        x = ops.materialize(x)
        ops._check(x)
        C = x.shape[-1]
        if C < groups:      # reference group_norm.py:51-59
            raise ValueError(f"Number of groups ({groups}) cannot be more than the number of channels ({C}).")
        if C % groups != 0:
            raise ValueError(f"Number of groups ({groups}) must be a multiple of the number of channels ({C}).")
        g0, dg = self.geometry(x)
        hw = x.shape[2] * x.shape[3]
        off, total = g0 * hw, dg * hw          # the slab's voxel window of the volume
        if stats is None:
            stats = torch.empty((1, groups, 2), dtype=torch.float64, device=x.device)
            ops._call("b3d_gn_stats", x, stats, groups, off, total)
            self._pending.append(stats)
        self.flush()             # the conv epilogue's (or the kernel's above) partial sums -> whole-volume statistics
        L = total * C // groups
        if self.p16 is not None and ops.p16_ok(x.shape) and L % 8 == 0 and hw * C % 8 == 0:
            y16 = self.new_p16(x.shape, x)
            y = None if operand_only else torch.empty_like(x)
        else:
            y16, y = None, self.new_activation(x.shape, x)
        ops._call("b3d_gn_apply", x, stats, gamma, beta, y, y16, None, groups, float(eps), int(relu), off, total)
        if y16 is None:
            return y
        if y is None:
            return ops.virtual(x.shape, x, [y16], None)
        ops._attach(y, y16, None)
        return y

    def group_norm_channel(self, x, gamma, beta, groups, eps, relu, operand_only=False):
        """GroupNormalization with true channel groups (channels_first models; ops.group_norm routes here): the
        slab's channel-group sums are partial sums of the whole volume's, all-reduced in the next flush together
        with the pointwise conv's pending pooling sums; outputs as in `group_norm`."""
        from . import ops
        x = ops.materialize(x)
        ops._check(x)
        stats = torch.empty((1, groups, 2), dtype=torch.float64, device=x.device)
        ops._call("b3d_gn_channel_stats", x, stats, groups)     # raises the reference's ValueError on bad groups
        self._pending.append(stats)
        self.flush()
        nvox = self.global_voxels(x)
        if self.p16 is not None and ops.p16_ok(x.shape):
            y16 = self.new_p16(x.shape, x)
            y = None if operand_only else torch.empty_like(x)
            ops._call("b3d_gn_channel_apply_slab", x, stats, gamma, beta, y, y16, groups, float(eps), int(relu), nvox)
            if y is None:
                return ops.virtual(x.shape, x, [y16], None)
            ops._attach(y, y16, None)
            return y
        y = self.new_activation(x.shape, x)
        ops._call("b3d_gn_channel_apply_slab", x, stats, gamma, beta, y, None, groups, float(eps), int(relu), nvox)
        return y


# ------------------------------------------------------------------------------------------ drivers
def depth_axis(model) -> int:
    """Dimension of the depth axis in the model's public tensors: 2 for a channels_first model (NCDHW), else 1."""
    return 2 if getattr(model, "data_format", "channels_last") == "channels_first" else 1


def slab_forward(model, x_local: torch.Tensor, ctx: SlabContext) -> torch.Tensor:
    """This rank's slab of `model(x, training=False, inference=True)[0]` (test.py:133)."""
    with torch.no_grad(), ctx:
        return model(x_local, training=False, inference=True)[0]


def sharded_inference(model, x: torch.Tensor, comm: Comm, gather: bool = True, align: Optional[int] = None):
    """x: the WHOLE padded volume [1, D, H, W, C] ([1, C, D, H, W] for a channels_first model; every rank holds it,
    as after loading a case from disk); each rank computes its depth slab; returns the whole prediction
    (gather=True) or (slab, (d0, d1)), in the layout of x."""
    if align is None:
        align = 2 ** (len(model.encoder.levels) - 1)
    ax = depth_axis(model)
    ctx = SlabContext(comm, x.shape[ax], align=align)
    y = slab_forward(model, x.narrow(ax, ctx.d0, ctx.local_depth).contiguous(), ctx)
    if not gather:
        return y, (ctx.d0, ctx.d1)
    return comm.all_gather_cat(y, [b - a for a, b in ctx.bounds], dim=ax)


class GraphedInference:
    """`model(x, training=False, inference=True)[0]` captured once into a CUDA graph for a fixed input shape and
    replayed: the ~350 C-ABI calls of a forward become one launch.  With `comm` (a DistComm over NCCL) the input is
    this rank's depth slab and the halo exchanges / small all-reduces are captured into the graph too."""

    def __init__(self, model, x_example: torch.Tensor, comm: Optional[Comm] = None, depth: Optional[int] = None,
                 warmup: int = 2):
        self.x = x_example.clone()
        self.model = model
        self.ctx = None
        if comm is not None:
            align = 2 ** (len(model.encoder.levels) - 1)
            ax = depth_axis(model)
            self.ctx = SlabContext(comm, depth if depth is not None else x_example.shape[ax] * comm.world, align=align)
            if self.ctx.local_depth != self.x.shape[ax]:
                raise ValueError("GraphedInference: x_example must be this rank's slab")
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(warmup):
                self._run()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = self._run()

    def _run(self):
        if self.ctx is not None:
            return slab_forward(self.model, self.x, self.ctx)
        with torch.no_grad():
            return self.model(self.x, training=False, inference=True)[0]

    def __call__(self, x: Optional[torch.Tensor] = None) -> torch.Tensor:
        if x is not None:
            self.x.copy_(x, non_blocking=True)
        self.graph.replay()
        return self.out


def run_virtual_ranks(model, x: torch.Tensor, world: int, align: Optional[int] = None):
    """Single-device validation mode: `world` virtual ranks as threads sharing this device (ThreadComm).
    Returns (whole prediction, per-rank communication statistics)."""
    comms = ThreadComm.make(world)
    if align is None:
        align = 2 ** (len(model.encoder.levels) - 1)
    ax = depth_axis(model)
    bounds = slab_bounds(x.shape[ax], world, align)
    outs, stats, errs = [None] * world, [None] * world, []

    def work(r):
        try:
            if x.is_cuda:
                torch.cuda.set_device(x.device)
            ctx = SlabContext(comms[r], x.shape[ax], bounds)
            outs[r] = slab_forward(model, x.narrow(ax, bounds[r][0], bounds[r][1] - bounds[r][0]).contiguous(), ctx)
            stats[r] = ctx.stats
        except BaseException as e:     # noqa: BLE001 — release the other ranks, then re-raise in the caller
            errs.append(e)
            comms[r].sh.barrier.abort()

    ts = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    if errs:
        real = [e for e in errs if not isinstance(e, threading.BrokenBarrierError)]
        raise (real or errs)[0]
    return torch.cat(outs, dim=ax), stats
