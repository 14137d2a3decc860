#!/usr/bin/env python
"""Benchmark of the Siegel pair-distance hot path (BASELINE.json metric: pairs/s forward+backward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--n 4] [--kind upper] [--dump-outputs DIR]

Workload (config.workload) = BASELINE.json configs[4], the distance microbench: a table of 2^20 random points
and ONE BATCH OF 64M (2^26) random index pairs per step, manifold `--kind` with n x n matrices, forward +
backward through the distortion loss (sympa/losses.py:16-19).  The batch is sharded over the N ranks (strong
scaling: 2^26 / N pairs per GPU and step); a rank works through its shard in chunks of 2^23 pairs, each chunk
one call of the public API (gather -> dist -> loss -> backward -> scatter-add into the table gradient), and the
step ends with the one collective of the path, the NCCL all-reduce (average) of the table gradient.
`value` is measured with everything resident in HBM; `e2e` runs the same step with every chunk's index pairs
and graph distances copied from pinned host memory and the loss read back, inside the timed region.
A second record, `n10`, repeats the measurement for upper / fmin / n = 10 (the other size BASELINE.json's metric
names) on a smaller batch.
`--dump-outputs DIR` writes what the last timed step of the headline record returned to its caller as float64 .npy
files (see dump_outputs); the inputs depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

GLOBAL_PAIRS = 1 << 26          # BASELINE.json configs[4]: 64M random pairs per batch
CHUNK_PAIRS = 1 << 23           # pairs per API call (saved unit gradients of a chunk: 2.7 GB at n = 4)
N10_GLOBAL_PAIRS = 1 << 23      # batch of the n = 10 side record (a step is ~0.1-0.2 s on one GPU)
DUMP_SEED = 20261020            # --dump-outputs: seed of the sampled pairs and table rows
DUMP_DIST_MAX = 1 << 20         # --dump-outputs: at most this many distances (8 MB)
DUMP_GRAD_BYTES = 48 << 20      # --dump-outputs: at most this many bytes of table-gradient rows (64 MB in all)


def chunk_pairs_for(n):
    if os.environ.get("SYMPA_BENCH_CHUNK_LOG2"):          # (experiments)
        return 1 << int(os.environ["SYMPA_BENCH_CHUNK_LOG2"])
    return CHUNK_PAIRS if n <= 4 else ((1 << 21) if n <= 6 else (1 << 19))


def algorithmic_bytes_per_pair(kind, n):
    """SURVEY.md 8(d), whole step: read two rows, accumulate two gradient rows, two int64 indices, vvd out, dist
    out, upstream gradient in."""
    if kind == "spd":
        return 32 * n * n + 8 * n + 32
    return 64 * n * n + 8 * n + 32


def kernel_bytes_per_pair(kind, n):
    """the forward + unit-gradient kernel ALONE: two rows in, two index words, dist + vvd out, and the saved unit
    gradients out (packed lower triangles)"""
    blocks = 1 if kind == "spd" else 2
    rows_in = 2 * blocks * n * n * 8
    state = 2 * blocks * (n * (n + 1) // 2) * 8       # packed lower triangles, every kernel family (ABI 4)
    return rows_in + state + 16 + 8 * n + 8


def lean_flops_per_pair(n):
    return 100 * n ** 3   # SURVEY.md 8(d) yardstick F_lean


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "MEASURED_PEAKS.json"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_min_mhz": min(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "reasons": sorted(reasons), "samples": len(sm)}


def measure_fp64_peak(dev, local):
    """attainable FP64 FMA rate of this GPU in TFLOP/s (sympa_probe_fp64: pure DFMA chains, best of 20 runs of ~35 ms, CUDA events),
    with the SM clock sampled while the probe runs"""
    from sympa_b200 import _lib
    lib = _lib.load()
    out = torch.zeros(1, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    iters = 1 << 18
    best = 0.0
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(20):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        flops = lib.sympa_probe_fp64(iters, out.data_ptr(), stream)
        e1.record()
        torch.cuda.synchronize()
        if flops > 0:
            best = max(best, flops / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    clocks = sampler.stop()
    return best, clocks


def make_table(kind, n, rows, device, seed):
    """'spread' regime of SURVEY.md 8(d), scale 0.3: X = sym(0.3 N(0,1)), Y = C C^T + 0.5 I."""
    g = torch.Generator(device=device).manual_seed(seed)
    c = 0.3 * torch.randn(rows, n, n, dtype=torch.float64, device=device, generator=g)
    y = c @ c.transpose(-1, -2) + 0.5 * torch.eye(n, dtype=torch.float64, device=device)
    y = 0.5 * (y + y.transpose(-1, -2))
    if kind == "spd":
        return y.contiguous()
    x = 0.3 * torch.randn(rows, n, n, dtype=torch.float64, device=device, generator=g)
    x = 0.5 * (x + x.transpose(-1, -2))
    z = torch.stack((x, y), 1).contiguous()
    if kind == "bounded":
        from sympa_b200.manifolds import csym
        out = torch.empty_like(z)
        for s in range(0, rows, 1 << 16):
            out[s:s + (1 << 16)] = csym.to_symmetric(csym.cayley_transform(z[s:s + (1 << 16)]))
        z = out
    return z


def make_pairs(rows, b, device, seed):
    """src ~ U{0..N-1}, dst != src, graph distance ~ U{1..20} (SURVEY.md 8(d)); distances as uint8 - what
    preprocess.py:118-126 produces are small integers."""
    g = torch.Generator(device=device).manual_seed(seed)
    src = torch.randint(0, rows, (b,), device=device, generator=g)
    dst = (src + 1 + torch.randint(0, rows - 1, (b,), device=device, generator=g)) % rows   # src != dst
    gd = torch.randint(1, 21, (b,), device=device, generator=g, dtype=torch.uint8)
    return torch.stack((src, dst), 1).contiguous(), gd


def reference_loss(graph_dist, manifold_dist):
    """sympa/losses.py:16-19, the reference's torch expression"""
    return torch.abs(torch.pow(manifold_dist / graph_dist, 2) - 1).sum()


def _sample(count, keep):
    """sorted positions of a fixed, seeded sample of `keep` out of `count` (all of them when they fit)"""
    if count <= keep:
        return torch.arange(count)
    return torch.randperm(count, generator=torch.Generator().manual_seed(DUMP_SEED))[:keep].sort().values


def dump_outputs(out_dir, dists, loss, table_grad):
    """What one step of the timed path hands its caller, as float64 .npy files in out_dir:
    loss.npy        (1,)            the step's distortion loss (sum over the chunks)
    dist.npy        (m,)            manifold distances at a seeded sample of this rank's pair positions
    table_grad.npy  (r, *row shape) table.grad at a seeded sample of the table rows (after the all-reduce)
    The samples depend only on the batch and table sizes; together the files stay below 64 MB."""
    os.makedirs(out_dir, exist_ok=True)
    d = torch.cat([x.reshape(-1) for x in dists])
    d = d[_sample(d.numel(), DUMP_DIST_MAX).to(d.device)]
    rows = table_grad.shape[0]
    row_bytes = table_grad[0].numel() * 8
    g = table_grad[_sample(rows, max(1, DUMP_GRAD_BYTES // row_bytes)).to(table_grad.device)]
    arrays = {"loss": loss.reshape(1), "dist": d, "table_grad": g}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to("cpu", torch.float64).numpy())
    return sorted(arrays)


def make_manifold(kind, n, metric, dev):
    from sympa_b200 import BoundedDomainManifold, MetricType, SymmetricPositiveDefinite, UpperHalfManifold
    if kind == "spd":
        return SymmetricPositiveDefinite().to(dev)
    return {"upper": UpperHalfManifold, "bounded": BoundedDomainManifold}[kind](
        dims=n, metric=MetricType.from_str(metric)).to(dev)


def our_launches_per_chunk(kind, n, rows, b, dev, world, single_chunk=True):
    """kernels of libsympa_b200.so one chunk launches through the public API: forward + unit gradients, loss forward
    and backward, table-gradient backward (packed scatter + expansion, or the direct scatter; with the in-backward
    all-reduce of a multi-rank run the scatter is one launch per pipelined row segment); the bounded domain by rows
    adds its two row kernels.  torch's own fill / add kernels and NCCL's are not counted."""
    from sympa_b200 import ops
    sync = world > 1 and single_chunk
    by_rows = ops.bounded_by_rows(kind, n, b, rows, sync)
    kk = "upper" if by_rows else kind
    packed = ops.backward_workspace_for(kk, n, rows, dev)[1] > 0 and (2 * b >= rows or sync)
    scatter = (ops.SYNC_SEGMENTS + 1) if (sync and packed and ops.SYNC_SEGMENTS > 1) else (2 if packed else 1)
    if not single_chunk:     # gradient accumulation: scatter per chunk; expansion and row transforms once per step
        return 1 + 2 + 1
    return 1 + 2 + scatter + (2 if by_rows else 0)


def measure(kind, n, metric, rows, global_pairs, steps, warmup, rank, world, local, dev, per_kernel=True, fused=True,
            e2e=True, dump_dir=None):
    """pairs/s of one configuration: resident step, per-kernel times, fused step, end-to-end step.  dump_dir: rank 0
    writes the outputs of the last timed resident step there (dump_outputs)."""
    import torch.distributed as dist
    from sympa_b200 import _lib, ops
    from sympa_b200 import distributed as sd
    from sympa_b200.feeder import PairFeeder
    from sympa_b200.losses import AverageDistortionLoss

    man = make_manifold(kind, n, metric, dev)
    loss_fn = AverageDistortionLoss()
    table = make_table(kind, n, rows, dev, seed=1).requires_grad_(True)     # replicated on every rank
    b_rank = global_pairs // world                                          # this rank's shard of the batch
    chunk = min(chunk_pairs_for(n), b_rank)
    if chunk == b_rank and b_rank >= (1 << 22) and n >= 3 and not os.environ.get("SYMPA_BENCH_CHUNK_LOG2"):
        # a rank whose shard is a single call (8 GPUs) makes two: the scatter of the first half overlaps the forward
        # kernel of the second (TableGradAccumulator) - measured on a rank's share, 2^23 pairs: 4.96 -> 4.73 ms per step
        chunk = b_rank // 2
    n_chunks = -(-b_rank // chunk)
    idx, gd8 = make_pairs(rows, b_rank, dev, seed=100 + rank)
    gd = gd8.double()
    scale = 1.0
    mk = metric if kind != "spd" else "riem"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    # a shard of several chunks is one step with gradient accumulation (the reference's grad_accum_steps,
    # runner.py:104): the chunks share a packed gradient table, expanded (and all-reduced) once per step
    acc = man.table_grad_accumulator(table) if n_chunks > 1 else None

    def run_chunks(get_chunk, keep=None):
        """one step: every chunk through the public API; one chunk: the collective runs inside its backward on the
        packed gradient table; several chunks: they accumulate in the packed table of `acc`, and acc.finish() runs
        the collective on it and writes table.grad.  keep: a list that receives every chunk's distances"""
        table.grad = None
        total = torch.zeros((), dtype=torch.float64, device=dev)
        for c in range(n_chunks):
            idx_c, gd_c = get_chunk(c)
            if acc is not None and c == n_chunks - 1:
                acc.last_chunk()         # its scatter has no forward kernel to overlap with: whole GPU
            d = man.dist_from_table(table, idx_c, sync_grad=(world > 1 and acc is None), accumulator=acc)
            loss = loss_fn.calculate_loss(gd_c, d * scale)
            loss.backward()
            total += loss.detach()
            if keep is not None:
                keep.append(d.detach())
        if acc is not None:
            acc.finish(sync_grad=world > 1)
        return total

    def resident_chunk(c):
        return idx[c * chunk:(c + 1) * chunk], gd[c * chunk:(c + 1) * chunk]

    last = {}       # with dump_dir: the distances and loss of the latest resident step

    def step_resident():
        if dump_dir is None:
            return run_chunks(resident_chunk)
        last.clear()
        last["dist"] = []
        last["loss"] = run_chunks(resident_chunk, last["dist"])
        return last["loss"]

    host_ms = {}

    def timed(fn, k, tag=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        if tag:      # host time to ENQUEUE the steps (no synchronisation inside): must stay below the device time
            host_ms[tag] = (time.perf_counter() - t0) * 1e3 / k
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    for _ in range(warmup):
        step_resident()
    ops.check_status(dev)
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.2)
    ms_total = timed(step_resident, steps, tag="resident")
    clocks = sampler.stop()
    if dump_dir is not None:
        if rank == 0:
            names = dump_outputs(dump_dir, last["dist"], last["loss"], table.grad)
            print(f"bench: wrote {', '.join(names)} of the last timed step to {dump_dir}", file=sys.stderr)
        last.clear()
    res = {"value": global_pairs * steps / (ms_total * 1e-3), "ms_per_step": ms_total / steps, "clocks": clocks,
           "host_enqueue_ms_per_step": round(host_ms.get("resident", 0.0), 3),
           "pairs_per_gpu_per_step": b_rank, "chunk_pairs": chunk, "chunks_per_step": n_chunks}
    lpc = our_launches_per_chunk(kind, n, rows, chunk, dev, world, single_chunk=(n_chunks == 1))
    per_step_extra = 0 if n_chunks == 1 else (1 + (2 if kind == "bounded" else 0))     # expansion (+ row transforms) once per step
    res["gpu_launches"] = (lpc * n_chunks + per_step_extra) * steps
    res["launches_per_chunk"] = lpc

    lib = _lib.load()
    if per_kernel:   # the kernels of one chunk timed alone, CUDA events on the launching (current) stream
        fwd_ms, bwd_ms, rows_ms = [], [], []
        ci, cg = resident_chunk(0)
        cb = ci.shape[0]
        # the route the step takes: bounded by rows = row transform + the UPPER-half pair kernel on the transformed table
        by_rows = ops.bounded_by_rows(kind, n, cb, rows, world > 1 and n_chunks == 1)
        kk = "upper" if by_rows else kind
        ktable = table.detach()
        if by_rows:
            ktable = torch.empty_like(ktable)
            gz = torch.empty_like(ktable)
        ws, ws_bytes = ops.backward_workspace_for(kk, n, rows, dev)
        gt = torch.empty_like(table)
        stream = torch.cuda.current_stream().cuda_stream
        torch.cuda.synchronize()
        for it in range(min(steps, 10) + 1):      # (the first pass is a warm-up: its allocations can fall between the events)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(8)]
            if by_rows:
                ev[4].record()
                _lib.check(lib.sympa_bounded_rows_to_upper(n, rows, table.data_ptr(), ktable.data_ptr(),
                                                           ops.status_word(dev).data_ptr(), stream))
                ev[5].record()
            with torch.no_grad():
                ev[0].record()
                dd, vv, saved = ops.forward_raw(kk, mk, table=ktable, idx=ci, wsum_w=None, want_grad=True)
                ev[1].record()
            g1 = torch.ones_like(dd)
            ev[2].record()   # the backward of the table path as the autograd Function issues it (workspace, overwrite)
            _lib.check(lib.sympa_dist_backward_table(_lib.KIND[kk], n, _lib.METRIC["riem"], cb, g1.data_ptr(),
                                                     saved.data_ptr(), gt.data_ptr(), rows, ci.data_ptr(), None, None, None,
                                                     None if ws is None else ws.data_ptr(), ws_bytes, 1,
                                                     torch.cuda.current_stream().cuda_stream))
            ev[3].record()
            if by_rows:
                ev[6].record()
                _lib.check(lib.sympa_bounded_rows_backward(n, rows, table.data_ptr(), gt.data_ptr(), gz.data_ptr(), 1, stream))
                ev[7].record()
            torch.cuda.synchronize()
            if it == 0:
                del saved, dd, vv
                continue
            fwd_ms.append(ev[0].elapsed_time(ev[1]))
            bwd_ms.append(ev[2].elapsed_time(ev[3]))
            if by_rows:
                rows_ms.append(ev[4].elapsed_time(ev[5]) + ev[6].elapsed_time(ev[7]))
            del saved, dd, vv
        del gt
        res["kernel_ms"] = statistics.median(fwd_ms)
        res["backward_ms"] = statistics.median(bwd_ms)
        res["kernel_pairs"] = cb
        res["kernel_kind"] = kk
        if by_rows:
            res["bounded_rows_ms"] = statistics.mean(rows_ms)
            del ktable, gz

    if fused:    # one launch per chunk (on-device loss): sympa_distortion_step
        gtab = torch.zeros_like(table)
        loss_out = torch.zeros(1, dtype=torch.float64, device=dev)

        def step_fused():
            gtab.zero_()
            loss_out.zero_()
            for c in range(n_chunks):
                ic, gc = resident_chunk(c)
                ops.distortion_step(kind, mk, table.detach(), ic, gc, scale, gtab, loss_out=loss_out)
            if world > 1:
                sd.allreduce_gradients([gtab], average=True)
        for _ in range(2):
            step_fused()
        k = max(2, steps // 2)
        ms_fused = timed(step_fused, k) / k
        res["fused_step"] = {"pairs_per_s": global_pairs / (ms_fused * 1e-3), "ms_per_step": ms_fused,
                             "launches_per_chunk": 1}
        del gtab

    if e2e:
        # host-resident inputs: node ids as int32, graph distances as uint8 (9 bytes per pair on the wire), widened
        # on the device by the feeder; every chunk of every step crosses PCIe inside the timed region
        idx_h = idx.to(torch.int32).cpu().pin_memory()
        gd_h = gd8.cpu().pin_memory()
        loss_h = torch.empty(2, dtype=torch.float64).pin_memory()    # two slots: the host reads step k - 1 while step k runs
        loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
        losses = []
        feeder = PairFeeder(dev)

        def submit(c):
            feeder.submit(idx_h[c * chunk:(c + 1) * chunk], gd_h[c * chunk:(c + 1) * chunk])

        def step_e2e(more_steps):
            first = [True]

            def get(c):
                if not first[0]:
                    feeder.done()           # the kernels that read the previous chunk are enqueued
                first[0] = False
                ic, gc = feeder.next()
                if c + 1 < n_chunks:        # the copy of the next chunk overlaps this chunk's compute
                    submit(c + 1)
                elif more_steps:
                    submit(0)
                return ic, gc
            total = run_chunks(get)
            feeder.done()
            k = step_no[0] % 2
            loss_h[k:k + 1].copy_(total.reshape(1), non_blocking=True)      # this step's result, device -> host
            loss_ev[k].record()
            if step_no[0] > 0:      # block on the PREVIOUS step's read-back: the host stays one step ahead of the device
                loss_ev[1 - k].synchronize()
                losses.append(float(loss_h[1 - k]))
            step_no[0] += 1

        step_no = [0]

        def run_e2e(k):
            step_no[0] = 0
            submit(0)                       # first chunk: its copy is exposed, and inside the timed region
            for s in range(k):
                step_e2e(s + 1 < k)
            last = (k - 1) % 2              # the last step's loss: the host waits for it inside the timed region
            loss_ev[last].synchronize()
            losses.append(float(loss_h[last]))

        run_e2e(2)
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        run_e2e(steps)
        t1.record()
        barrier()
        ms_e2e = max_over_ranks(t0.elapsed_time(t1))
        res["e2e"] = {"value": global_pairs * steps / (ms_e2e * 1e-3), "unit": "pairs/s",
                      "h2d_bytes_per_step": int((idx_h.numel() * idx_h.element_size() + gd_h.numel() * gd_h.element_size()) * world),
                      "d2h_bytes_per_step": 8 * world,
                      "ms_per_step": ms_e2e / steps,
                      "how": "per step and rank: every chunk = manifold.dist_from_table + AverageDistortionLoss + backward "
                             "through the public API; the chunk's index pairs (int32 on the host, widened on the device) and "
                             "graph distances (uint8 on the host) are copied from pinned host memory by "
                             "sympa_b200.feeder.PairFeeder (the copy of chunk k+1 overlaps the compute of chunk k on a side "
                             "stream; the first copy is exposed); every step's loss is copied device -> host, the host waits for the read-back of "
                             "step k - 1 after enqueueing step k (and for the last step's before the timed region ends)"}
        del idx_h, gd_h
    ops.check_status(dev)
    del table, idx, gd
    torch.cuda.empty_cache()
    return res


def roofline_of(kind, n, res, fp64_peak, fp64_clocks, peaks, peak_src, rows):
    """roofline object of the dominant kernel (forward + unit gradients) from its live-timed duration"""
    b = res["kernel_pairs"]
    k_s = res["kernel_ms"] * 1e-3
    lean_tf = lean_flops_per_pair(n) * b / k_s / 1e12
    kb = kernel_bytes_per_pair(kind, n) * b
    step_b = res["pairs_per_gpu_per_step"]
    step_s = res["ms_per_step"] * 1e-3
    kk = res.get("kernel_kind", kind)
    coop = n > {"upper": 7, "bounded": 7, "spd": 10}[kk]
    kname = (f"coop_kernel<{n},{kk},fwd+unit-grad>" if coop else f"pair_kernel<{n},{kk},fwd+unit-grad>")
    fp64_bound = n >= 3
    traffic = scatter = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        rec = tj.get(f"{kind}_n{n}_fwdsave")
        if rec:
            traffic = rec["bytes_per_pair"] * b     # ncu dram bytes per pair x pairs of one launch
        rec = tj.get(f"{kind}_n{n}_backward")
        if rec:   # the backward of a chunk: its DRAM traffic (ncu) over its live-timed duration
            sbytes = rec["scatter_bytes_per_pair"] * b + rec["expand_bytes_per_row"] * rows
            alg = (3 * 16 * n * (n + 1) + 24) * b + 48 * n * n * rows
            scatter = {"kernel": rec["kernel"], "bound": "hbm", "traffic": sbytes, "algorithmic_bytes": alg,
                       "achieved": round(alg / (res["backward_ms"] * 1e-3) / 1e9, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                       "frac": round(alg / (res["backward_ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                       "traffic_over_algorithmic": round(sbytes / alg, 3)}
    fp64 = {"bound": "fp64", "achieved": round(lean_tf, 3), "peak": round(fp64_peak, 2), "unit": "TFLOP/s",
            "frac": round(lean_tf / max(fp64_peak, 1e-9), 4), "peak_nominal": 37.2,
            "peak_source": "sympa_probe_fp64 (pure DFMA chains) timed with CUDA events in this run - MEASURED_PEAKS.json "
                           "has no FP64 entry", "peak_clocks": fp64_clocks,
            "how": "algorithmic flops 100 n^3 per pair (SURVEY.md 8(d) F_lean) x pairs of one launch / kernel time"}
    hbm = {"bound": "hbm", "achieved": round(kb / k_s / 1e9, 2), "peak": peaks["hbm_gbs"], "unit": "GB/s",
           "frac": round(kb / k_s / 1e9 / peaks["hbm_gbs"], 4), "algorithmic_bytes": kb, "peak_source": peak_src,
           "how": "the kernel's OWN algorithmic bytes (rows in, indices, dist + vvd, saved unit gradients out) / kernel time"}
    main = dict(fp64 if fp64_bound else hbm)
    main.update({"kernel": kname, "kernel_ms": round(res["kernel_ms"], 4), "pairs_per_launch": b, "traffic": traffic,
                 "traffic_source": "ncu --set full capture, profiles/r02_traffic.json" if traffic else None,
                 "other_bound": hbm if fp64_bound else fp64,
                 "whole_step": {
                     "fp64_frac": round(lean_flops_per_pair(n) * step_b / step_s / 1e12 / max(fp64_peak, 1e-9), 4),
                     "hbm_frac": round(algorithmic_bytes_per_pair(kind, n) * step_b / step_s / 1e9 / peaks["hbm_gbs"], 4),
                     "how": "F_lean resp. SURVEY.md 8(d) bytes (64n^2+8n+32) x this GPU's pairs of a step / device time of the "
                            "whole step (forward, loss, backward scatter + expansion, gradient accumulation, collective)"},
                 "backward_ms": round(res["backward_ms"], 4)})
    if "bounded_rows_ms" in res:
        main["bounded_rows_ms"] = round(res["bounded_rows_ms"], 4)
        main["note"] = ("bounded domain by rows: the inverse Cayley transform runs once per table row and chunk "
                        "(sympa_bounded_rows_to_upper / _backward, bounded_rows_ms), the pairs run the upper-half kernel")
    if scatter is not None:
        main["scatter"] = scatter
    return main


def parity_check(rank, world, dev):
    """N > 1, inside the warm-up: the table gradient after the in-backward NCCL all-reduce (pairs sharded over the
    ranks as DistributedSampler does, train.py:105-110) must equal the full-batch gradient of one GPU divided by
    the number of ranks (DDP averages, train.py:59).  40 960 pairs, upper n = 4 and bounded n = 3 (by-rows route);
    also a rank with an EMPTY shard joins the collective.  Every rank checks; the verdict is the AND over ranks."""
    import torch.distributed as dist
    from sympa_b200 import distributed as sd
    out = {"ok": True, "max_rel": 0.0, "pairs": 40960, "cases": []}
    for kind, n, metric in (("upper", 4, "riem"), ("bounded", 3, "fone"), ("upper", 10, "fmin")):
        rows, pairs = 4096, 40960
        man = make_manifold(kind, n, metric, dev)
        table = make_table(kind, n, rows, dev, seed=7)
        idx, gd8 = make_pairs(rows, pairs, dev, seed=11)          # same batch on every rank
        gd = gd8.double()

        def grad_of(sel, sync):
            t = table.clone().requires_grad_(True)
            d = man.dist_from_table(t, idx[sel].contiguous(), sync_grad=sync)
            reference_loss(gd[sel], d).backward()
            return t.grad

        shard = sd.shard_indices(pairs, rank, world, shuffle=True, seed=3).to(dev)
        avg = grad_of(shard, True)
        everyone = torch.cat([sd.shard_indices(pairs, r, world, shuffle=True, seed=3) for r in range(world)]).to(dev)
        full = grad_of(everyone, False) / world
        rel = float((avg - full).abs().max() / full.abs().max())
        # ragged: the last rank has nothing this step
        sel = shard if rank < world - 1 else shard[:0]
        avg2 = grad_of(sel, True)
        part = torch.cat([sd.shard_indices(pairs, r, world, shuffle=True, seed=3) for r in range(world - 1)]).to(dev)
        full2 = grad_of(part, False) / world
        rel2 = float((avg2 - full2).abs().max() / full2.abs().max())
        # the route of a multi-chunk step (N = 1, 2, 4 of the scaling run): the shard in three calls that accumulate
        # into one packed table (scatter on the side stream), ONE all-reduce in finish()
        t3 = table.clone().requires_grad_(True)
        acc = man.table_grad_accumulator(t3)
        cuts = [0, len(shard) // 3, len(shard) // 3 + 1, len(shard)]
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            sel3 = shard[lo:hi]
            reference_loss(gd[sel3], man.dist_from_table(t3, idx[sel3].contiguous(), accumulator=acc)).backward()
        acc.finish(sync_grad=True)
        rel3 = float((t3.grad - full).abs().max() / full.abs().max())
        out["cases"].append({"kind": kind, "n": n, "max_rel": rel, "max_rel_empty_rank": rel2, "max_rel_accumulated": rel3})
        out["max_rel"] = max(out["max_rel"], rel, rel2, rel3)
    out["ok"] = bool(out["max_rel"] < 1e-9)
    flag = torch.tensor([1.0 if out["ok"] else 0.0, out["max_rel"]], dtype=torch.float64, device=dev)
    ok = flag[:1].clone()
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    mx = flag[1:].clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    out["ok"] = bool(ok.item() > 0.5)
    out["max_rel"] = float(mx.item())
    out["how"] = ("dist_from_table(sync_grad=True) on each rank's DistributedSampler shard vs the full-batch gradient of one "
                  "GPU / world - in one call, with an empty rank, and accumulated over three calls with the all-reduce in "
                  "TableGradAccumulator.finish(sync_grad=True) -, max |diff| / max |grad|, worst rank; tolerance 1e-9")
    return out


def run_ours(args):
    import torch.distributed as dist
    from sympa_b200 import distributed as sd

    # rank 0 prints ONE JSON line on stdout.  NCCL writes its version banner to stdout when the environment sets
    # NCCL_DEBUG=VERSION/WARN (the GPU boxes do): rather than silencing NCCL, file descriptor 1 points at stderr
    # until the line is printed, so every library's chatter is kept - on stderr.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = sd.init_process_group()
    assert world == args.gpus, f"launched with WORLD_SIZE={world} but --gpus {args.gpus}"
    dev = torch.device("cuda", local)
    # pinned host buffers NUMA-local to this rank's GPU (SYMPA_BENCH_NO_NUMA=1 switches it off for an A/B)
    # - only with several ranks: one rank keeps every host core for the CPU baseline it also times
    numa = None if (os.environ.get("SYMPA_BENCH_NO_NUMA") or world == 1) else sd.bind_to_gpu_numa_node(local)
    if os.environ.get("SYMPA_SPLIT_PATH"):          # tuning experiments only
        from sympa_b200 import _lib
        _lib.check(_lib.load().sympa_set_option(_lib.OPT_SPLIT_PATH, int(os.environ["SYMPA_SPLIT_PATH"])))
    if os.environ.get("SYMPA_SCATTER_PASS_MB"):     # tuning experiments only
        from sympa_b200 import _lib
        _lib.check(_lib.load().sympa_set_option(_lib.OPT_SCATTER_PASS_MB, int(os.environ["SYMPA_SCATTER_PASS_MB"])))
    kind, n, rows = args.kind, args.n, args.rows
    global_pairs = args.pairs if args.pairs else GLOBAL_PAIRS
    warmup = max(args.warmup, 3)
    pcheck = parity_check(rank, world, dev) if world > 1 else None

    res = measure(kind, n, args.metric, rows, global_pairs, args.steps, warmup, rank, world, local, dev,
                  dump_dir=args.dump_outputs)
    peaks, peak_src = load_peaks()
    fp64_peak, fp64_clocks = measure_fp64_peak(dev, local)
    roofline = roofline_of(kind, n, res, fp64_peak, fp64_clocks, peaks, peak_src, rows)
    par = (f"dp{world}: the batch sharded over the ranks ({res['pairs_per_gpu_per_step']} pairs per GPU and step), table "
           "replicated, one NCCL all-reduce (average) of the table gradient per step")
    out = {
        "metric": "Siegel dist pairs/s fwd+bwd", "value": res["value"], "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"distance microbench (BASELINE.json configs[4]): {kind} n={n} metric={args.metric}, table "
                               f"2^{rows.bit_length() - 1} rows, one batch of {global_pairs} random pairs per step (sharded "
                               f"over {world} GPU(s), chunks of {res['chunk_pairs']} pairs per API call), fwd+bwd through "
                               "AverageDistortionLoss",
                   "global_pairs_per_step": global_pairs, "pairs_per_gpu_per_step": res["pairs_per_gpu_per_step"],
                   "chunk_pairs": res["chunk_pairs"], "rows": rows, "n": n, "kind": kind, "metric": args.metric,
                   "l2": "table (268 MB at n=4) + saved unit gradients + indices of a chunk exceed the 126 MB L2 many times "
                         "over (no explicit flush needed)",
                   "parallelism": par,
                   "host_numa": (f"rank 0 runs on the {numa['cpus']} CPUs of NUMA node {numa['node']} (its GPU's node): pinned "
                                 "buffers are first-touched there" if numa else "not bound (topology unreadable or switched off)")},
        "e2e": res["e2e"],
        "gpu_launches": res["gpu_launches"],
        "gpu_launches_how": f"{res['launches_per_chunk']} kernels of libsympa_b200.so per chunk x {res['chunks_per_step']} "
                            f"chunks x {args.steps} steps (forward + unit gradients, loss forward, loss backward, table-gradient "
                            "scatter [+ expansion, once per step when the chunks accumulate]); torch's fill kernels and NCCL's are not "
                            "counted",
        "fused_step": res["fused_step"],
        "host_enqueue_ms_per_step": res["host_enqueue_ms_per_step"],
        "clocks": res["clocks"],
        "roofline": roofline,
    }
    if pcheck is not None:
        out["parity_check"] = pcheck
    if not args.no_n10:   # the other matrix size named by BASELINE.json's metric, as a record of its own
        r10 = measure("upper", 10, "fmin", rows, N10_GLOBAL_PAIRS, max(3, min(args.steps, 5)), 3, rank, world, local, dev,
                      fused=False)
        out["n10"] = {"metric": "Siegel dist pairs/s fwd+bwd", "value": r10["value"], "unit": "pairs/s",
                      "ms_per_step": r10["ms_per_step"], "steps": max(3, min(args.steps, 5)), "warmup": 3,
                      "config": {"workload": f"distance microbench: upper n=10 metric=fmin, table 2^{rows.bit_length() - 1} rows, one "
                                             f"batch of {N10_GLOBAL_PAIRS} random pairs per step (sharded over {world} GPU(s), "
                                             f"chunks of {r10['chunk_pairs']}), fwd+bwd through AverageDistortionLoss",
                                 "global_pairs_per_step": N10_GLOBAL_PAIRS, "rows": rows, "n": 10, "kind": "upper",
                                 "metric": "fmin"},
                      "e2e": r10["e2e"], "clocks": r10["clocks"], "gpu_launches": r10["gpu_launches"],
                      "roofline": roofline_of("upper", 10, r10, fp64_peak, fp64_clocks, peaks, peak_src, rows)}
    if not args.no_extras:
        out["also"] = extras(args, world, rank, dev)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(kind, n, args.metric, budget_s=args.cpu_budget)
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    if rank == 0:
        print(json.dumps(out), flush=True)
    os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def quick_pairs_per_s(kind, n, metric, pairs, rows, dev, world, steps=5):
    """resident fwd+bwd pairs/s of another configuration (one chunk per rank and step)."""
    import torch.distributed as dist
    from sympa_b200.losses import AverageDistortionLoss
    man = make_manifold(kind, n, metric, dev)
    loss_fn = AverageDistortionLoss()
    table = make_table(kind, n, rows, dev, seed=2).requires_grad_(True)
    idx, gd8 = make_pairs(rows, pairs, dev, seed=300)
    gd = gd8.double()

    def step():
        table.grad = None
        d = man.dist_from_table(table, idx, sync_grad=world > 1)
        loss_fn.calculate_loss(gd, d).backward()

    for _ in range(3):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    return world * pairs * steps / (ms * 1e-3)


def dropin_pairs_per_s(dev, n=4, pairs=1 << 21, rows=1 << 20, steps=5):
    """The literal drop-in path of the north star - the reference's model.py / losses.py unchanged around the
    replaced manifold: two torch gathers (sympa/embeddings.py:29-34), manifold.dist(z1, z2) on MATERIALISED operands
    (model.py:32-38), the reference's loss expression (losses.py:16-19), autograd backward with torch's dense
    index_put gather-backward into the (N, 2, n, n) gradient."""
    man = make_manifold("upper", n, "riem", dev)
    table = make_table("upper", n, rows, dev, seed=3).requires_grad_(True)
    idx, gd8 = make_pairs(rows, pairs, dev, seed=301)
    gd = gd8.double()

    def step():
        table.grad = None
        d = man.dist(table[idx[:, 0]], table[idx[:, 1]])
        reference_loss(gd, d).backward()

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    return pairs * steps / (e0.elapsed_time(e1) * 1e-3)


def _epoch_model(config, dev):
    from types import SimpleNamespace
    from sympa_b200.graphs import balanced_tree_triplets, grid_triplets, product_cartesian_triplets
    from sympa_b200.model import Model
    torch.manual_seed(0)
    if config == 1:     # BASELINE configs[0]: grid 20x20 (400 nodes, 79 800 pairs), upper / riem / n=2
        idx, gd, nodes = grid_triplets(20, 2)
        a = dict(manifold="upper", metric="riem", dims=2)
    elif config == 2:   # BASELINE configs[1]: balanced tree branching 3 height 5 (364 nodes, 66 066 pairs), bounded / fone / n=3
        idx, gd, nodes = balanced_tree_triplets(3, 5)
        a = dict(manifold="bounded", metric="fone", dims=3)
    else:               # BASELINE configs[2]: product-cartesian tree x grid with the reference's CLI defaults (preprocess.py:
        # tree 3/3 x grid 5x5x5 = 5000 nodes, 12 497 500 pairs), upper / finf / n=6
        idx, gd, nodes = product_cartesian_triplets(3, 3, 5, 3)
        a = dict(manifold="upper", metric="finf", dims=6)
    args = SimpleNamespace(num_points=nodes, scale_init=1.0, scale_coef=1.0, train_scale=False, **a)
    return Model(args).to(dev), idx.to(dev), gd.to(dev)


EPOCH_BATCH = {1: 2048, 2: 2048, 3: 131072}     # configs 1-2: the reference's batch; config 3: 96 steps per epoch


def epoch_seconds(dev, world, rank, epochs=3, fused=True, sync_stats=True, config=1):
    """Seconds per training epoch (runner.py:90-122 semantics, per-step loss.item() kept), RiemannianSGD."""
    from sympa_b200.optim import RiemannianSGD
    from sympa_b200.runner import train_epoch
    model, idx, gd = _epoch_model(config, dev)
    bs = EPOCH_BATCH[config]
    opt = RiemannianSGD(model.parameters(), lr=1e-2 * world, fused=fused)
    dshuf = config == 3      # 12.5 M pairs: the permutation is drawn on the GPU (0.2 s per epoch on the CPU)
    train_epoch(model, opt, idx, gd, bs, world_size=world, rank=rank, epoch=0, sync_stats=sync_stats, device_shuffle=dshuf)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for ep in range(1, epochs + 1):
        loss = train_epoch(model, opt, idx, gd, bs, world_size=world, rank=rank, epoch=ep, sync_stats=sync_stats,
                           device_shuffle=dshuf)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / epochs, loss


def fused_epoch_seconds(dev, world, rank, epochs=5, config=1):
    """The same epochs on sympa_b200.runner.FusedEpochRunner: two launches per step (fused distortion step, fused
    optimizer row kernel with clipping and zero_grad), the epoch replayed from a CUDA graph on one rank, the loss
    read back once per epoch."""
    from sympa_b200.runner import FusedEpochRunner
    model, idx, gd = _epoch_model(config, dev)
    runner = FusedEpochRunner(model, 1e-2 * world, idx, gd, EPOCH_BATCH[config], world_size=world, rank=rank,
                              device_shuffle=(config == 3))
    runner.run_epoch(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for ep in range(1, epochs + 1):
        loss = runner.run_epoch(ep)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / epochs, loss


def cfg4_step(kind, n, metric, dev, world, rank, rows=1 << 20, global_pairs=1 << 22, steps=3, owner_computes=False):
    """BASELINE configs[3]: a 1M-node table, one TRAINING STEP (forward, distortion loss, backward, the gradient
    collective, fused Riemannian SGD update of the table) on a batch of sampled pairs sharded over the ranks.
    Returns (ms per step, pairs per step, loss of the last step)."""
    from sympa_b200 import distributed as sd
    from sympa_b200.embeddings import ManifoldParameter
    from sympa_b200.losses import AverageDistortionLoss
    from sympa_b200.optim import RiemannianSGD
    man = make_manifold(kind, n, metric, dev)
    table = ManifoldParameter(make_table(kind, n, rows, dev, seed=5), manifold=man)
    opt = RiemannianSGD([table], lr=1e-3 * world, fused=True)
    loss_fn = AverageDistortionLoss()
    b_rank = global_pairs // world
    chunk = min(chunk_pairs_for(n), b_rank)
    n_chunks = -(-b_rank // chunk)
    idx, gd8 = make_pairs(rows, b_rank, dev, seed=500 + rank)
    gd = gd8.double()

    from sympa_b200 import ops
    lr = 1e-3 * world

    # several calls per step accumulate in one packed gradient table (expanded - and all-reduced - once per step)
    acc = man.table_grad_accumulator(table) if n_chunks > 1 else None

    def step():
        table.grad = None
        total = torch.zeros((), dtype=torch.float64, device=dev)
        in_backward = world > 1 and n_chunks == 1 and not owner_computes
        for c in range(n_chunks):
            sl = slice(c * chunk, (c + 1) * chunk)
            if acc is not None and c == n_chunks - 1:
                acc.last_chunk()
            d = man.dist_from_table(table, idx[sl], sync_grad=in_backward, accumulator=acc)
            loss = loss_fn.calculate_loss(gd[sl], d)
            loss.backward()
            total += loss.detach()
        if acc is not None:
            acc.finish(sync_grad=world > 1 and not owner_computes)
        if owner_computes and world > 1:
            # SURVEY.md 8(f) rank 2: reduce-scatter by row owner, fused update of the owned rows, all-gather
            sd.sharded_rsgd_step(table, lr, lambda t, g, s: ops.rsgd_step(kind, t, g.contiguous(), s))
            return total
        if world > 1 and not in_backward and acc is None:
            sd.allreduce_gradients([table.grad], average=True)
        opt.step()
        return total

    step()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = t.item()
    out = (ms, global_pairs, float(loss.item()))
    del table, opt, idx, gd
    torch.cuda.empty_cache()
    return out


def extras(args, world, rank, dev):
    """Side measurements: other sizes, the literal drop-in path, BASELINE.json's epoch-time leg (configs 1-3)."""
    out = {}
    try:
        out["upper_n2_riem_pairs_per_s"] = quick_pairs_per_s("upper", 2, "riem", 1 << 22, 1 << 20, dev, world)
        out["upper_n6_finf_pairs_per_s"] = quick_pairs_per_s("upper", 6, "finf", 1 << 20, 1 << 20, dev, world)
        out["spd_n10_pairs_per_s"] = quick_pairs_per_s("spd", 10, "riem", 1 << 18, 1 << 18, dev, world)
        out["bounded_n3_fone_pairs_per_s"] = quick_pairs_per_s("bounded", 3, "fone", 1 << 22, 1 << 20, dev, world)
        if world == 1:
            out["dropin_pairs_per_s"] = dropin_pairs_per_s(dev)
            out["dropin_how"] = ("upper n=4, 2^21 pairs/step: table[idx] gathers + manifold.dist(z1, z2) on materialised operands "
                                 "+ the reference's loss expression + torch's dense index_put backward (model.py:16-38, "
                                 "losses.py:16-19 as shipped)")
        # configs 1-2 (79 800 / 66 066 pairs in batches of 2048) do not shard - a 256-pair shard per rank is pure launch
        # latency: with N > 1 every rank trains its own replica on the whole graph, no collective (DESIGN.md section 4)
        for cfg, name in ((1, "config1_grid400_upper_riem_n2"), (2, "config2_tree_b3h5_bounded_fone_n3")):
            tag = "" if world == 1 else "_replica_per_rank"
            sec, loss = epoch_seconds(dev, 1, 0, fused=True, sync_stats=True, config=cfg)
            out[f"train_epoch_sec_{name}_b2048{tag}"] = sec
            out[f"train_epoch_final_loss_{name}"] = loss
            sec_g, loss_g = fused_epoch_seconds(dev, 1, 0, config=cfg)
            out[f"train_epoch_sec_{name}_fused_graph{tag}"] = sec_g
            out[f"train_epoch_final_loss_{name}_fused_graph"] = loss_g
        sec_h, _ = epoch_seconds(dev, 1, 0, fused=False, sync_stats=True)
        out["train_epoch_sec_config1_host_optimizer"] = sec_h
        # config 3: product-cartesian graph, 12.5M pairs per epoch, pairs sharded over the ranks, batch 131072
        name = "config3_product_tree3x3_grid5x5x5_5000nodes_upper_finf_n6_b131072"
        sec, loss = epoch_seconds(dev, world, rank, epochs=2, fused=True, sync_stats=True, config=3)
        out[f"train_epoch_sec_{name}_sharded_dp{world}"] = sec
        out[f"train_epoch_final_loss_{name}"] = loss
        sec_g, loss_g = fused_epoch_seconds(dev, world, rank, epochs=2, config=3)
        out[f"train_epoch_sec_{name}_fused_sharded_dp{world}"] = sec_g
        out[f"train_epoch_final_loss_{name}_fused"] = loss_g
        # config 4: 1M-node table, one training step on 2^22 sampled pairs (sharded), optimizer included
        for kind, metric, key in (("upper", "fmin", "cfg4_1Mnodes_upper_fmin_n10"), ("spd", "riem", "cfg4_1Mnodes_spd_n10")):
            ms, pairs, loss = cfg4_step(kind, 10, metric, dev, world, rank)
            out[f"{key}_train_step_ms_dp{world}"] = ms
            out[f"{key}_pairs_per_step"] = pairs
            out[f"{key}_pairs_per_s"] = pairs / (ms * 1e-3)
            out[f"{key}_loss"] = loss
            if world > 1:   # the same step with the owner-computes optimizer (reduce-scatter, update of N/P rows, all-gather)
                ms2, _, loss2 = cfg4_step(kind, 10, metric, dev, world, rank, owner_computes=True)
                out[f"{key}_train_step_ms_dp{world}_owner_computes"] = ms2
                out[f"{key}_loss_owner_computes"] = loss2
    except Exception as e:  # noqa: BLE001 - extras must never take the headline line down
        out["error"] = repr(e)
    return out


# ------------------------------------------------------------------------------------------ CPU legs
def _reference_dist_fn(kind, n, metric):
    """manifold.dist of the UNMODIFIED reference when oracle/_ref holds a copy of its package (made by
    oracle/make_ref.py in the build container; git-ignored, travels to the GPU box), else the oracle port.
    Returns (callable(z1, z2) -> dist, kind_label)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    ref_root = os.path.join(ROOT, "oracle", "_ref")
    if kind != "spd" and os.path.isdir(os.path.join(ref_root, "sympa")):
        try:
            os.environ["SYMPA_REFERENCE_ROOT"] = ref_root
            import import_reference
            import_reference.REFERENCE_ROOT = ref_root
            import_reference.import_reference()
            from sympa.manifolds import BoundedDomainManifold, UpperHalfManifold
            from sympa.manifolds.metrics import MetricType
            torch.set_default_dtype(torch.float64)      # what sympa/config.py:17-18 does
            man = (UpperHalfManifold if kind == "upper" else BoundedDomainManifold)(dims=n, metric=MetricType.from_str(metric))
            return (lambda z1, z2: man.dist(z1, z2)), "reference"
        except Exception:  # noqa: BLE001
            pass
    import siegel_oracle as so
    return (lambda z1, z2: so.dist(kind, z1, z2, metric if kind != "spd" else "riem")), "port"


def _cpu_step_fn(kind, n, metric, rows, b):
    dist_fn, label = _reference_dist_fn(kind, n, metric)
    table = make_table(kind, n, rows, torch.device("cpu"), seed=1).requires_grad_(True)
    idx, gd8 = make_pairs(rows, b, torch.device("cpu"), seed=100)
    gd = gd8.double()

    def step():
        table.grad = None
        d = dist_fn(table[idx[:, 0]], table[idx[:, 1]])      # gathers + dist, as Model.forward (model.py:16-38)
        reference_loss(gd, d).backward()                      # losses.py:16-19 + autograd, dense index_put backward
    return step, label


def cpu_baseline(kind, n, metric, budget_s=15.0, threads=None):
    """The reference's own CPU implementation of the path timed on the host cores: gather -> dist -> distortion loss
    -> autograd backward, float64, on a bounded sample of the workload."""
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    rows, b = 1 << 14, 1 << 14
    step, label = _cpu_step_fn(kind, n, metric, rows, b)
    step()
    t0 = time.perf_counter()
    reps = 0
    while True:
        step()
        reps += 1
        el = time.perf_counter() - t0
        if el > budget_s or reps >= 2000:
            break
    return {"value": b * reps / el, "unit": "pairs/s", "cores": threads, "kind": label,
            "sample": f"{reps} steps x {b} pairs of the same workload ({kind} n={n} metric={metric}, table 2^14 rows), "
                      f"torch CPU float64, {el:.1f} s"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind, n = args.kind, args.n
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    rows, b = 1 << 14, 1 << 13
    step, label = _cpu_step_fn(kind, n, args.metric, rows, b)
    warmup = max(1, args.warmup)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    el = time.perf_counter() - t0
    value = b * args.steps / el
    sample = (f"each step = {b} pairs (a bounded sample of the 2^26-pair batch), table 2^14 rows, gather -> manifold.dist -> "
              f"losses.py expression -> autograd backward, torch CPU float64, {threads} threads")
    out = {
        "impl": "reference", "metric": "Siegel dist pairs/s fwd+bwd", "value": value, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup, "ms_per_step": el / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"distance microbench (BASELINE.json configs[4]): {kind} n={n} metric={args.metric}; this CPU arm "
                               f"runs a bounded sample per step: {b} pairs on a table of {rows} rows",
                   "pairs_per_step": b, "rows": rows, "n": n, "kind": kind, "metric": args.metric},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": threads, "kind": label, "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kind", default="upper", choices=["upper", "bounded", "spd"])
    ap.add_argument("--n", type=int, default=4)
    ap.add_argument("--metric", default="riem")
    ap.add_argument("--rows", type=int, default=1 << 20)
    ap.add_argument("--pairs", type=int, default=0, help="pairs of the whole batch per step (default 2^26)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the side measurements (other sizes, epoch times)")
    ap.add_argument("--no-n10", action="store_true", help="skip the n = 10 record")
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, a sample of the distances and a sample of the table gradient of the last timed "
                         "step of the headline record as float64 .npy files into DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
