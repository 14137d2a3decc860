"""The training step / epoch of sympa/runner.py:90-122 on the fused path (host logic only; the
tensorboard / checkpoint / evaluation plumbing of the reference Runner is out of scope)."""
import torch
from torch.nn.utils import clip_grad_norm_

from . import distributed as sd
from . import ops
from .losses import AverageDistortionLoss


def train_epoch(model, optimizer, src_dst_ids, graph_distances, batch_size, max_grad_norm=50.0, grad_accum_steps=1,
                world_size=1, rank=0, epoch=0, shuffle=True, sync_stats=True, device_shuffle=False, presharded=False):
    """One pass over the training triplets (runner.py:90-122).

    src_dst_ids (T, 2) int64 and graph_distances (T,) live on the device (train.py:95-96).  Each rank
    takes the DistributedSampler shard of the triplets (train.py:105-110) in batches of
    batch_size // world_size; gradients of all parameters are averaged over the ranks before clipping
    (what DistributedDataParallel does, train.py:59) - the one collective of the path.
    Returns the mean loss per step (as runner.py:122).  sync_stats=False skips the per-step
    `.item()` host synchronisations of runner.py:108-110 and reads the loss once at the end.
    presharded=True: the triplets are already this rank's shard (sampling.PairSampler.sample with this rank): they
    are permuted locally by epoch instead of being split again; gradients are still averaged over the ranks.
    """
    loss_fn = AverageDistortionLoss()
    dev = src_dst_ids.device
    # device_shuffle: the epoch's permutation is drawn on the GPU (not DistributedSampler's CPU order)
    order = sd.shard_indices(src_dst_ids.shape[0], 0 if presharded else rank, 1 if presharded else world_size, epoch=epoch,
                             shuffle=shuffle, device=dev if device_shuffle else None).to(dev)
    per_rank = max(batch_size // world_size, 1)
    ok, point, reason = model.check_all_points()        # runner.py:91
    if not ok:
        raise AssertionError(f"Point outside manifold. Reason: {reason}\n{point}")
    model.train()
    optimizer.zero_grad(set_to_none=False)
    total = torch.zeros((), dtype=torch.float64, device=dev)
    steps = 0
    params = [p for p in model.parameters() if p.requires_grad]
    for step, start in enumerate(range(0, order.numel(), per_rank)):
        sel = order[start:start + per_rank]
        dist_m = model(src_dst_ids[sel])
        loss = loss_fn.calculate_loss(graph_distances[sel], dist_m) / grad_accum_steps
        loss.backward()
        if sync_stats:
            total += loss.item()                         # runner.py:108 (host sync, as the reference)
        else:
            total += loss.detach()
        steps += 1
        if (step + 1) % grad_accum_steps == 0:
            if world_size > 1:
                sd.allreduce_gradients([p.grad for p in params], average=True)
            clip_grad_norm_(params, max_grad_norm)       # runner.py:115
            optimizer.step()
            optimizer.zero_grad(set_to_none=False)
    ops.check_status(dev)       # the reference's per-call asserts, once per epoch
    return float(total.item()) / max(steps, 1)


class FusedEpochRunner:
    """The same epoch (runner.py:90-122: batches of the DistributedSampler shard, distortion loss, backward,
    gradient clipping at max_grad_norm, RiemannianSGD step, zero_grad) on the fused path:

        per step   sympa_distortion_step   gather + dist + loss + its derivative + scatter-add   (1 launch)
                   total gradient norm -> clipping coefficient min(1, max_norm / (norm + 1e-6))  (torch, on device)
                   sympa_rsgd_step_ex      egrad2rgrad + retr + projx per touched row, scaled by the coefficient,
                                           gradient rows zeroed in the same pass                 (1 launch)

    and - on one GPU - the whole epoch captured once in a CUDA graph and replayed: the epochs of the BASELINE
    configs are launch-bound (39 steps of ~0.1 ms of GPU work each), so removing ~40 launches and the per-step
    `.item()` synchronisation per step (runner.py:108-110) is what matters.  The loss is accumulated on the
    device and read once per epoch.  The permutation of the epoch is applied by one gather into persistent
    buffers, so the captured graph sees fixed addresses.

    Restrictions (otherwise use `train_epoch`): float64 CUDA table, grad_accum_steps == 1; the model scale must
    not be trainable (it enters the kernel as a host scalar).  The wsum weights, when the metric has them,
    are updated as Euclidean parameters with the same clipping coefficient (as geoopt's RSGD does).

    presharded=True: src_dst_ids / graph_distances are already this rank's shard (sampling.PairSampler.sample with
    this rank): every epoch permutes all of them locally instead of taking a DistributedSampler shard; gradients
    are still averaged over the ranks.  run_epoch re-gathers self.ids and self.gdist every epoch, so pairs written
    into them in place (PairSampler.sample(epoch, out=(runner.ids, runner.gdist))) are trained on at once."""

    def __init__(self, model, lr, src_dst_ids, graph_distances, batch_size, max_grad_norm=50.0, world_size=1, rank=0,
                 use_graph=True, shuffle=True, device_shuffle=False, presharded=False):
        table = model.embeddings.embeds
        if not table.is_cuda or table.dtype != torch.float64:
            raise RuntimeError("FusedEpochRunner needs a CUDA float64 embedding table (there is no CPU path)")
        if model.scale.requires_grad:
            raise RuntimeError("FusedEpochRunner: a trainable model scale is not supported, use train_epoch")
        self.model, self.lr, self.max_grad_norm = model, float(lr), float(max_grad_norm)
        self.world, self.rank, self.shuffle, self.device_shuffle = world_size, rank, shuffle, device_shuffle
        # the split run_epoch takes of self.ids: none when presharded (rank 0 of 1)
        self.split_rank, self.split_world = (0, 1) if presharded else (rank, world_size)
        self.ids, self.gdist = src_dst_ids, graph_distances
        self.per_rank = max(batch_size // world_size, 1)
        self.dev = table.device
        man = model.manifold
        self.kind = man.kind
        self.metric = "riem" if self.kind == "spd" else man.metric.name
        self.wsum = getattr(getattr(man, "metric", None), "weights", None) if self.metric == "wsum" else None
        self.count = -(-src_dst_ids.shape[0] // self.split_world)     # what shard_indices returns (padded by wrapping)
        self.idx_buf = torch.empty(self.count, 2, dtype=torch.int64, device=self.dev)
        self.gd_buf = torch.empty(self.count, dtype=torch.float64, device=self.dev)
        self.grad = torch.zeros_like(table.data)
        self.loss_acc = torch.zeros(1, dtype=torch.float64, device=self.dev)
        self.coef = torch.ones(1, dtype=torch.float64, device=self.dev)
        self.gw = torch.zeros(self.wsum.numel(), dtype=torch.float64, device=self.dev) if self.wsum is not None else None
        self.counter = torch.zeros(1, dtype=torch.int64, device=self.dev)
        self.steps = -(-self.count // self.per_rank)
        self.graph = None
        self.use_graph = use_graph and world_size == 1
        self.scale = float(model.get_scale().item())

    def _step(self, start):
        table = self.model.embeddings.embeds.data
        idx = self.idx_buf[start:start + self.per_rank]
        gd = self.gd_buf[start:start + self.per_rank]
        w = None if self.wsum is None else self.wsum.data.reshape(-1)
        ops.distortion_step(self.kind, self.metric, table, idx, gd, self.scale, self.grad, wsum_w=w, grad_wsum_w=self.gw,
                            loss_out=self.loss_acc)
        grads = [self.grad] if self.gw is None else [self.grad, self.gw]
        if self.world > 1:
            sd.allreduce_gradients(grads, average=True)
        # clip_grad_norm_ (runner.py:115): coefficient applied inside the update instead of to the gradients
        nrm = torch.linalg.vector_norm(self.grad)
        if self.gw is not None:
            nrm = torch.sqrt(nrm * nrm + self.gw.square().sum())
        torch.clamp(self.max_grad_norm / (nrm + 1e-6), max=1.0, out=self.coef[0])
        ops.rsgd_step(self.kind, table, self.grad, self.lr, lr_scale=self.coef, projected=self.counter, zero_grad=True)
        if self.gw is not None:
            self.wsum.data.sub_((self.lr * self.coef) * self.gw.reshape(self.wsum.shape))
            self.gw.zero_()

    def _all_steps(self):
        for start in range(0, self.count, self.per_rank):
            self._step(start)

    def run_epoch(self, epoch=0):
        """One epoch; returns the mean loss per step (as runner.py:122), read back once."""
        ok, point, reason = self.model.check_all_points()        # runner.py:91
        if not ok:
            raise AssertionError(f"Point outside manifold. Reason: {reason}\n{point}")
        order = sd.shard_indices(self.ids.shape[0], self.split_rank, self.split_world, epoch=epoch, shuffle=self.shuffle,
                                 device=self.dev if self.device_shuffle else None).to(self.dev)
        torch.index_select(self.ids, 0, order, out=self.idx_buf)
        torch.index_select(self.gdist, 0, order, out=self.gd_buf)
        self.loss_acc.zero_()
        if not self.use_graph:
            self._all_steps()
        else:
            if self.graph is None:
                # warm-up outside the capture (first-launch attribute calls, allocator pools), on a copy of the state
                keep = self.model.embeddings.embeds.data.clone()
                keep_w = None if self.wsum is None else self.wsum.data.clone()
                side = torch.cuda.Stream(device=self.dev)
                side.wait_stream(torch.cuda.current_stream(self.dev))
                with torch.cuda.stream(side):
                    self._step(0)
                torch.cuda.current_stream(self.dev).wait_stream(side)
                self.model.embeddings.embeds.data.copy_(keep)
                if keep_w is not None:
                    self.wsum.data.copy_(keep_w)
                self.grad.zero_()
                self.loss_acc.zero_()
                self.counter.zero_()
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    self._all_steps()
                # the capture does not execute: replay below runs the epoch
            self.graph.replay()
        man = self.model.manifold
        if hasattr(man, "_projected_counter") or self.kind != "spd":
            man._projected_counter = self.counter
        ops.check_status(self.dev)
        return float(self.loss_acc.item()) / max(self.steps, 1)
