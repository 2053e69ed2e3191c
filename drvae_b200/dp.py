"""Data-parallel training of ONE model on a large minibatch (BASELINE.json configs[3], SURVEY.md §8(e)).

The reference has no distributed code; this is the B200 design for its large-batch case.  Rows of
the minibatch are sharded over ranks.  Every loss term is a sum over rows divided by a batch-level
count (DrVAE.py:612-616: N, max(1, Np), max(1, Nlab)), so a shard that is given the GLOBAL counts
produces an additive share of every loss term and of the gradient:

    counts   = all_reduce_sum([N_local, Np_local, Nlab_local])           (3 integers, before the step)
    grads_r  = drvae_grad_step(shard_r, global counts, row_offset_r)     (flat fp32 [P], C ABI)
    grads    = all_reduce_sum(grads_r)  — issued per parameter bucket on a side stream as soon as the
               backward pass has produced that bucket, overlapping the rest of backward
    drvae_adam_step(...)                                                 (replicated optimizer: 28 MB of state)

That is the NCCL path of a multi-rank step, launched eagerly.  With NVLink peer memory (PeerBackend) a step is
drvae_dp_exchange_counts + drvae_dp_train_step, which sums the gradients inside the optimizer kernel; on one rank it is
drvae_dp_train_step alone.  The plan replays drvae_dp_train_step as a CUDA graph like its other steps.

ε is keyed by the global row index (drvae_noise_t.row_offset), so the result does not depend on
the number of ranks.  The communication backend is torch.distributed (NCCL over NVLink on the
GPU box; gloo in the CPU tests of the host logic, with the oracle as the compute backend).
"""
import os

import torch
import torch.distributed as dist

from .plan import LOSS_KEYS


def shard_rows(n_rows, world, rank):
    """Contiguous, balanced row ranges: the first (n_rows % world) ranks get one extra row."""
    base, extra = divmod(int(n_rows), int(world))
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def local_counts(n, has_x2=None, has_y=None):
    np_ = int(has_x2.ne(0).sum()) if has_x2 is not None else 0
    nl = int(has_y.ne(0).sum()) if has_y is not None else 0
    return [int(n), np_, nl]


def global_counts(counts, group=None, device="cpu"):
    """Sum [N, Np, Nlab] over the ranks of `group`."""
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
        return [int(c) for c in counts]
    t = torch.tensor(counts, dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return [int(v) for v in t.tolist()]


def global_counts_device(counts, device, group=None):
    """As global_counts, but the sum stays on the device (int64 [3]): the host does not wait for the all-reduce and
    can keep enqueueing the step (drvae_hparams_t.global_counts_dev)."""
    t = torch.tensor(counts, dtype=torch.int64).pin_memory().to(device, non_blocking=True)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


class PlanBackend:
    """Compute backend over the C ABI: one single-model Plan on this rank's GPU.

    On one rank DataParallel.step is one drvae_dp_train_step, replayed by the plan as a CUDA graph.  With more ranks
    it is the eager NCCL path of the module docstring: capturing the per-bucket NCCL all-reduces as well is what a
    multi-rank step needs (a shard of a few hundred rows finishes faster than the host can enqueue ~50 launches and 7
    collectives), but that capture deadlocked when tried."""

    def __init__(self, plan):
        if plan.E != 1:
            raise ValueError("data-parallel training shards ONE model; ensembles shard by model instead")
        self.plan = plan
        self.device = plan.device
        self.comm_stream = torch.cuda.Stream(device=plan.device)

    @property
    def graphs(self):
        """CUDA-graph replays of the plan's steps so far."""
        return self.plan.graph_replays()

    def flat_grads(self):
        return self.plan.grads[0]

    def buckets(self):
        return self.plan.grad_buckets()

    def grad_step(self, batch, hp_kwargs, counts, step, eps=None, seed=0, row_offset=0):
        hp = self.plan.hparams(step=step, global_counts=counts, **hp_kwargs)
        self._hp = hp
        losses = self.plan.grad_step(batch, hp, eps=eps, seed=seed, row_offset=row_offset)
        # drvae_grad_step records one CUDA event per bucket as its gradients complete
        return losses[0], [lambda stream, k=k: self.plan.stream_wait_bucket(k, stream) for k in range(len(self.buckets()))]

    def adam_step(self):
        self.plan.adam_step(self._hp)


class PeerBackend(PlanBackend):
    """GPU backend without NCCL on the data path: every rank's flat gradient lives in symmetric memory all ranks have
    mapped (torch.distributed._symmetric_memory is used for the allocation and the pointer exchange only), and the
    all-reduce is fused into the optimizer kernel (csrc/dp_peer.cuh): cross-GPU flag barrier + ONE kernel that sums the
    ranks' gradients over NVLink in rank order and applies Adam.  The whole step — gradient kernels, barrier, optimizer —
    is one drvae_dp_train_step, replayed as one CUDA graph per set of batch buffers on every rank; per step the host
    launches the counts exchange and the step."""

    def __init__(self, plan, group=None, multicast=None):
        super().__init__(plan)
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        dev = plan.device
        n = plan.dp_grad_floats()
        self.gbuf = symm_mem.empty(n, dtype=torch.float32, device=dev)
        self.ctl = symm_mem.empty(128, dtype=torch.int64, device=dev)
        self.gbuf.zero_()
        self.ctl.zero_()
        gh = symm_mem.rendezvous(self.gbuf, self.group)
        ch = symm_mem.rendezvous(self.ctl, self.group)
        torch.cuda.synchronize(dev)
        dist.barrier(self.group)  # every control block is zero before anybody posts a flag
        if multicast is None:
            # NVLS multicast mapping (one switch-reduced load per element instead of one load per rank): measured on one
            # box at 8192 rows: 8 ranks 0.483 -> 0.442 ms per step, 4 ranks 0.471 -> 0.471 (profiles/r02_experiments.md)
            knob = os.environ.get("DRVAE_B200_DP_MULTICAST")
            multicast = (knob != "0") if knob is not None else self.world >= 8
        mc = int(getattr(gh, "multicast_ptr", 0) or 0) if multicast else 0
        self.multicast = bool(mc)
        plan.dp_attach(self.rank, self.world, list(gh.buffer_ptrs), list(ch.buffer_ptrs), mc)
        self._handles = (gh, ch)
        self.global_losses = torch.zeros(8, dtype=torch.float32, device=dev)
        self.peer = True


class DataParallel:
    """step(): one optimisation step of a row-sharded minibatch.  `backend` is a PlanBackend on the
    GPU box; the CPU tests substitute an oracle-backed object with the same four methods."""

    def __init__(self, backend, group=None):
        self.backend = backend
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.finished_training_iters = 0

    def _all_reduce(self, t):
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)

    def step(self, batch, hp_kwargs=None, eps=None, seed=0, row_offset=0, host_flags=None):
        """batch: this rank's shard (same fields as Plan.train_step).  Returns the GLOBAL losses as
        an 8-vector (RECL, KLD, PERT, YL, MMD, ELBO, CMPL, 0) identical on every rank.
        host_flags: optional dict with the CPU copies of has_x2 / has_y (what a DataLoader yields), so the local
        counts are taken on the host without a device synchronisation."""
        be = self.backend
        n = batch["x1"].shape[-2]
        flags = host_flags if host_flags is not None else batch
        local = local_counts(n, flags.get("has_x2"), flags.get("has_y"))
        hp_kwargs = dict(hp_kwargs or {})
        it = self.finished_training_iters
        if getattr(be, "peer", False):
            # the counts exchange is also the barrier that keeps a fast rank from overwriting a gradient a slow rank
            # still reads
            be.plan.dp_exchange_counts(local, it + 1)
            hp = be.plan.hparams(step=it, global_counts_ptr=be.plan.dp_counts_ptr, **hp_kwargs)
            losses = be.plan.dp_train_step(batch, hp, be.global_losses, eps=eps, seed=seed, row_offset=row_offset)
            self.finished_training_iters += 1
            return losses
        if self.world == 1 and isinstance(be, PlanBackend):
            hp = be.plan.hparams(step=it, global_counts=local, **hp_kwargs)
            losses = be.plan.dp_train_step(batch, hp, be.plan.losses[0], eps=eps, seed=seed, row_offset=row_offset)
            self.finished_training_iters += 1
            return losses
        if self.world > 1 and getattr(be, "comm_stream", None) is not None:
            counts = global_counts_device(local, be.device, self.group)  # GPU backend: no host round trip
        else:
            counts = global_counts(local, self.group, device=getattr(be, "device", "cpu"))
        losses, events = be.grad_step(batch, hp_kwargs, counts, it, eps=eps, seed=seed, row_offset=row_offset)
        flat = be.flat_grads()
        comm = getattr(be, "comm_stream", None)
        if comm is None:  # CPU backend (tests): no streams, one reduce per bucket in the same order
            for off, cnt in be.buckets():
                self._all_reduce(flat[off:off + cnt])
            self._all_reduce(losses)
        else:
            # bucket k is complete when events[k] fires; its all-reduce runs on the side stream while
            # the compute stream is still inside the backward pass of the remaining blocks
            with torch.cuda.stream(comm):
                for (off, cnt), wait in zip(be.buckets(), events):
                    wait(comm)
                    self._all_reduce(flat[off:off + cnt])
                self._all_reduce(losses)
            torch.cuda.current_stream(be.device).wait_stream(comm)
        be.adam_step()
        self.finished_training_iters += 1
        return losses

    @staticmethod
    def losses_dict(losses):
        return {k: float(losses[i]) for i, k in enumerate(LOSS_KEYS)}
