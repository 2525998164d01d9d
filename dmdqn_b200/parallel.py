"""Multi-GPU plumbing: one process per GPU (torchrun), torch.distributed for rendezvous.

Independent networks (the reference's semantics, train.py:123-126) shard by contiguous
agent ranges with NO data-path collective: GPU r owns agents [r*N/G, (r+1)*N/G) with their
replay rings, theta, theta_tgt, Adam state (SURVEY.md section 8 E1).  Per-agent results are
bit-identical to the 1-GPU run because every kernel works on one agent's data only.

Shared parameters (BASELINE.json cfg5, not in the reference; SURVEY.md E2): every rank holds
a replica of theta/theta_tgt/m/v, draws batch/G transitions from its own rings, computes
dL/dtheta with the loss mean over the GLOBAL batch, the gradient blocks are summed and every
rank applies the same Adam step.  On GPUs the sum and the update are ONE kernel over NVLink
peer memory (``PeerExchange`` + ``dmdqn_allreduce_adam``: flag exchange, peer loads in rank
order, Adam in the same launch); the NCCL all-reduce + ``dmdqn_adam_apply`` path is kept as
the baseline it is measured against, and gloo carries the CPU tests of the host logic.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.distributed as dist


def shard_range(n_total: int, world: int, rank: int) -> tuple[int, int]:
    """Contiguous agent range of ``rank``; the first ``n_total % world`` ranks get one extra."""
    if not (0 <= rank < world) or n_total < 0:
        raise ValueError(f"bad shard request n_total={n_total} world={world} rank={rank}")
    base, extra = divmod(n_total, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def grid_neighbor_table(rows: int, cols: int):
    """Neighbour rows ``[rows*cols, 4]`` (int32, n,s,e,w; -1 = none) of a row-major ``J_r_c`` grid -- the table
    ``dmdqn_featurize`` takes instead of junction-id strings (order_lanes.py:399-404: n=(r-1,c), s=(r+1,c),
    e=(r,c+1), w=(r,c-1))."""
    import numpy as np
    r, c = np.divmod(np.arange(rows * cols), cols)
    out = np.full((rows * cols, 4), -1, np.int32)
    for k, (dr, dc) in enumerate(((-1, 0), (1, 0), (0, 1), (0, -1))):
        rr, cc = r + dr, c + dc
        ok = (rr >= 0) & (rr < rows) & (cc >= 0) & (cc < cols)
        out[ok, k] = (rr * cols + cc)[ok]
    return out


def shard_seed(seed: int, agent_global_index: int) -> int:
    """Per-agent init seed that does not depend on how agents are sharded."""
    return int(seed) + int(agent_global_index)


def allreduce_sum_(t: torch.Tensor, group=None) -> torch.Tensor:
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


class PeerExchange:
    """This rank's exchange buffer of the fused shared-parameter step and the peers' mappings of theirs.

    One device allocation per rank, float32 words: ``grads[2][stride] | loss[2][16] | flags uint32[MAX_PEERS][PEER_BLOCKS]``
    (grads / loss double-buffered by epoch parity: a peer may already write step t+1 while this rank still reads step
    t; the flags carry the epoch and are never reset).  The allocation is exported with CUDA IPC through the C ABI
    (``dmdqn_ipc_export`` / ``dmdqn_ipc_open``); torch.distributed only carries the 64-byte handles."""

    def __init__(self, grp, rank: int = 0, world: int = 1):
        from . import _native as N
        if world > N.MAX_PEERS:
            raise ValueError(f"the fused shared-parameter step serves up to {N.MAX_PEERS} ranks of one node, got {world}")
        self.N, self.grp, self.rank, self.world = N, grp, int(rank), int(world)
        self.stride = int(grp.theta.shape[-1])
        self.loss_off = 2 * self.stride
        self.flag_off = self.loss_off + 32
        self.buf = torch.zeros(self.flag_off + N.MAX_PEERS * N.PEER_BLOCKS, dtype=torch.float32, device=grp.device)
        self.loss_out = torch.zeros(1, dtype=torch.float32, device=grp.device)
        self.ptrs = [self.buf.data_ptr()] * self.world      # replaced by connect()
        self._opened = []
        self.epoch = 0

    def grads(self, epoch: int) -> torch.Tensor:
        o = (epoch & 1) * self.stride
        return self.buf[o:o + self.stride].view(1, self.stride)

    def connect(self, group=None) -> "PeerExchange":
        """Exchange IPC handles over the process group and map every peer's buffer on this device."""
        if self.world == 1:
            return self
        N, lib = self.N, self.grp.lib
        handle, off = (C.c_ubyte * 64)(), C.c_uint64()

        def agree(err):         # every rank learns about any rank's failure, so all raise together (no one is left in a collective)
            errs = [None] * self.world
            dist.all_gather_object(errs, err, group=group)
            bad = [f"rank {r}: {e}" for r, e in enumerate(errs) if e]
            if bad:
                self.close()
                raise N.NativeError("peer-memory exchange could not be set up (" + "; ".join(bad) + ")")
        with torch.cuda.device(self.grp.device):
            err, mine = None, None
            try:
                N.check(lib.dmdqn_ipc_export(self.buf.data_ptr(), handle, C.byref(off)))
                mine = (bytes(handle), int(off.value))
            except Exception as exc:
                err = str(exc)
            agree(err)
            everyone = [None] * self.world
            dist.all_gather_object(everyone, mine, group=group)
            self.ptrs = []
            try:
                for p, (h, o) in enumerate(everyone):
                    if p == self.rank:
                        self.ptrs.append(self.buf.data_ptr())
                        continue
                    out = C.c_void_p()
                    N.check(lib.dmdqn_ipc_open((C.c_ubyte * 64).from_buffer_copy(h), o, C.byref(out)))
                    self.ptrs.append(int(out.value))
                    self._opened.append((int(out.value), o))
            except Exception as exc:
                err = str(exc)
            agree(err)                      # also the barrier: nobody signals into a buffer its owner has not zeroed yet
        return self

    @staticmethod
    def connect_local(exchanges) -> None:
        """Several 'ranks' inside ONE process (tests on one GPU / one process driving several): plain pointers."""
        table = [e.buf.data_ptr() for e in exchanges]
        for e in exchanges:
            e.ptrs = list(table)

    def peers(self, epoch: int):
        P = self.N.Peers()
        for p in range(self.world):
            base = self.ptrs[p]
            P.grads[p] = base + 4 * (epoch & 1) * self.stride
            P.loss[p] = base + 4 * (self.loss_off + 16 * (epoch & 1))
            P.flags[p] = base + 4 * self.flag_off
        P.rank, P.world, P.epoch = self.rank, self.world, epoch
        return P

    def close(self) -> None:
        for ptr, off in self._opened:
            self.grp.lib.dmdqn_ipc_close(ptr, off)
        self._opened = []


class SharedParameterStep:
    """One data-parallel learn step of a shared network: local gradients -> all-reduce ->
    identical Adam on every replica.  ``local_grads(global_batch)`` returns the rank's
    gradient block (already divided by the global batch) and a [.., 8] metrics tensor whose
    column 0 is the rank's share of the loss; ``apply(grads)`` performs the update.  The two
    callables are the native calls on a GPU (``for_group``) and oracle stand-ins in the CPU
    (gloo) tests, so the same host logic is exercised in both.

    The learn decision is COLLECTIVE.  Whether a rank's rings hold its share of the batch
    (dqn_agent.py:333-335 applied to the rank's shard) differs between ranks while the rings
    fill -- ``shard_range`` gives the first ranks one agent more, masked pushes fill unevenly --
    and a replica that stepped alone would diverge for good (theta, Adam state, the
    target-sync counter).  So ``local_ready()`` flags are combined with a MIN all-reduce and
    either every rank steps or none does; ``step()`` returns None for a skipped step, like
    ``learn()`` while the buffer is short.  Rings only grow, so once every rank has been
    ready the exchange is dropped."""

    def __init__(self, local_grads, apply, local_batch: int, group=None, local_ready=None, flag_device="cpu",
                 fused_apply=None, world: int | None = None):
        self.local_grads, self.apply, self.local_batch, self.group = local_grads, apply, int(local_batch), group
        self.local_ready, self.flag_device = local_ready, flag_device
        self.fused_apply, self._world = fused_apply, world
        self._all_ready = False
        self.skipped = 0

    @property
    def world(self) -> int:
        if self._world is not None:             # ranks simulated inside one process (PeerExchange.connect_local)
            return self._world
        return dist.get_world_size(self.group) if dist.is_available() and dist.is_initialized() else 1

    def everyone_ready(self) -> bool:
        if self._all_ready:
            return True
        ready = True if self.local_ready is None else bool(self.local_ready())
        if self.world > 1 and self._world is None:
            flag = torch.tensor([1 if ready else 0], dtype=torch.int32, device=self.flag_device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
            ready = bool(flag.item())
        self._all_ready = ready
        return ready

    def step(self):
        if not self.everyone_ready():
            self.skipped += 1
            return None
        if self.fused_apply is not None:            # one kernel: flag exchange + peer loads + Adam (dmdqn_allreduce_adam)
            return self.fused_apply(self.local_batch * self.world)
        grads, metrics = self.local_grads(self.local_batch * self.world)
        allreduce_sum_(grads, self.group)           # 4*P bytes, latency bound (1.24 MB at H=512)
        loss = allreduce_sum_(metrics[..., 0].clone(), self.group)
        self.apply(grads)
        return loss

    @classmethod
    def for_group(cls, grp, group=None, fused: bool | None = None, exchange: "PeerExchange | None" = None) -> "SharedParameterStep":
        """Bind to an AgentGroup built with ``share_parameters=True``.  ``fused`` (default: whenever there is more
        than one rank) runs the all-reduce and Adam as one peer-memory kernel; ``fused=False`` is the NCCL
        all-reduce + ``dmdqn_adam_apply`` baseline.  A group with ``global_clipnorm`` takes the NCCL path and finishes with
        ``dmdqn_clip_adam_apply`` on the all-reduced block; ``fused=True`` is refused there.  ``exchange``: a PeerExchange
        already connected (tests).  A ``noisy`` group takes the NCCL path too: every rank folds the same noise (same keys and
        step counters), the effective-weight gradients are all-reduced and ``dmdqn_noisy_adam_apply`` updates mu and sigma;
        ``fused=True`` is refused there, because the peer-memory kernel does not know sigma."""
        from . import _native as N
        from .group import _ptr
        if not grp.shared:
            raise ValueError("SharedParameterStep needs share_parameters=True")
        world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        clip = grp.global_clipnorm
        if clip is not None and fused:
            raise ValueError("global_clipnorm is set: the fused peer-memory kernel (dmdqn_allreduce_adam) does not clip; "
                             "use fused=False (the NCCL all-reduce + dmdqn_clip_adam_apply path)")
        if grp.noisy and fused:
            raise ValueError("noisy=true: the fused peer-memory kernel (dmdqn_allreduce_adam) does not update sigma; use "
                             "fused=False (the NCCL all-reduce + dmdqn_noisy_adam_apply path)")
        if fused is None:
            fused = clip is None and not grp.noisy and (world > 1 or exchange is not None)
        if fused and exchange is None:
            rank = dist.get_rank(group) if world > 1 else 0
            exchange = PeerExchange(grp, rank, world).connect(group)
        grads = torch.zeros_like(grp.theta)

        def local_ready() -> bool:
            return bool(grp.active_host()[0])

        def local_grads(global_batch: int, out=None):
            out = grads if out is None else out
            if not local_ready():                   # cannot happen after everyone_ready(); never reduce a stale block
                out.zero_()
                grp.metrics.zero_()
                return out, grp.metrics
            d = grp.draw_words((1, grp.batch_size))
            with torch.cuda.device(grp.device):
                if grp.noisy:
                    N.check(grp.lib.dmdqn_learn_grads_noisy(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay),
                                                            C.byref(grp.nets), C.byref(grp.noisy_ptrs), _ptr(d), None,
                                                            int(global_batch), _ptr(out), _ptr(grp.metrics), _ptr(grp.workspace),
                                                            grp.workspace.numel(), grp._stream))
                else:
                    N.check(grp.lib.dmdqn_learn_grads(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay), C.byref(grp.nets),
                                                      _ptr(d), None, int(global_batch), _ptr(out), _ptr(grp.metrics),
                                                      _ptr(grp.workspace), grp.workspace.numel(), grp._stream))
            grp.learn_step_host += 1
            return out, grp.metrics

        def fused_begin(global_batch: int):          # this rank's gradient block of the step -> its exchange buffer
            exchange.epoch += 1
            local_grads(global_batch, out=exchange.grads(exchange.epoch))

        def fused_finish():                          # flag exchange + peer loads + Adam, one kernel
            peers = exchange.peers(exchange.epoch)
            with torch.cuda.device(grp.device):
                N.check(grp.lib.dmdqn_allreduce_adam(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), C.byref(peers),
                                                     _ptr(grp.metrics), _ptr(exchange.loss_out), _ptr(grp.workspace),
                                                     grp.workspace.numel(), grp._stream))
            return exchange.loss_out

        def fused_apply(global_batch: int):
            fused_begin(global_batch)
            return fused_finish()

        def apply(g: torch.Tensor):
            with torch.cuda.device(grp.device):
                if clip is not None:            # the norm of the all-reduced block: the same scale on every replica
                    N.check(grp.lib.dmdqn_clip_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), _ptr(g), clip,
                                                          _ptr(grp.grad_norms), _ptr(grp.workspace), grp.workspace.numel(),
                                                          grp._stream))
                    return
                if grp.noisy:
                    N.check(grp.lib.dmdqn_noisy_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets),
                                                           C.byref(grp.noisy_ptrs), _ptr(g), _ptr(grp.workspace),
                                                           grp.workspace.numel(), grp._stream))
                    return
                N.check(grp.lib.dmdqn_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), _ptr(g),
                                                 _ptr(grp.workspace), grp.workspace.numel(), grp._stream))
        step = cls(local_grads, apply, grp.batch_size, group, local_ready=local_ready, flag_device=grp.device,
                   fused_apply=fused_apply if fused else None,
                   world=exchange.world if (exchange is not None and world == 1 and exchange.world > 1) else None)
        step.exchange, step.fused_begin, step.fused_finish = exchange, fused_begin, fused_finish
        return step
