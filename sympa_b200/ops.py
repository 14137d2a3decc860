"""Host side of the hot path: torch.autograd Functions over the C ABI.

PyTorch is used for device memory, streams and autograd plumbing only; all arithmetic of
`dist` happens in libsympa_b200.so.  Tensors must be CUDA float64 and contiguous.
"""
import collections
import os

import torch

from . import _lib

# bounded domain on the table path: transform the rows once instead of both operands of every pair when the
# batch covers the table densely (set to False to force the per-pair bounded kernels)
BOUNDED_BY_ROWS = True
# largest matrix size of that route (the row kernels are unrolled register code for every n since round 2;
# round 1 stopped at 7: its rolled local-memory row kernels made bounded n = 10 slower, 18.9 -> 8.2 M pairs/s)
BOUNDED_BY_ROWS_MAX_N = 10

_status_words = {}
_scratch = {}


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def status_word(device):
    """Per-device uint32 word the kernels OR their SYMPA_STATUS_* bits into."""
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    w = _status_words.get(key)
    if w is None:
        w = torch.zeros(1, dtype=torch.int32, device=device)
        _status_words[key] = w
    return w


def scratch_for(kind, n, num_pairs, device):
    """Per-device scratch buffer (grown on demand, reused by every call on that device - calls are
    stream-ordered) for the three-kernel path of the larger matrix sizes."""
    nbytes = _lib.load().sympa_scratch_bytes(_lib.KIND[kind], n, num_pairs)
    if nbytes <= 0:
        return None, 0
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    buf = _scratch.get(key)
    if buf is None or buf.numel() * 8 < nbytes:
        buf = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=device)
        _scratch[key] = buf
    return buf, buf.numel() * 8


_bwd_workspace = {}


def backward_workspace_for(kind, n, num_rows, device):
    """Per-device workspace of the table-gradient backward (packed gradient table; grown on demand and
    reused - calls are stream-ordered)."""
    nbytes = _lib.load().sympa_backward_workspace_bytes(_lib.KIND[kind], n, num_rows)
    if nbytes <= 0:
        return None, 0
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    buf = _bwd_workspace.get(key)
    if buf is None or buf.numel() * 8 < nbytes:
        buf = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=device)
        _bwd_workspace[key] = buf
    return buf, buf.numel() * 8


def check_status(device=None, reset=True):
    """Host-synchronising check of the device status word (call once per step / epoch; the
    reference asserted synchronously inside every dist call, siegel_manifold.py:65-66)."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    w = status_word(device)
    v = int(w.item()) & 0xFFFFFFFF
    if reset:
        w.zero_()
    if v:
        reasons = [msg for bit, msg in _lib.STATUS_BITS.items() if v & bit]
        raise AssertionError("sympa_b200 status 0x%x: %s" % (v, "; ".join(reasons)))
    return v


CHECK_REASONS = {1: {"upper": "Matrices are not symmetric", "bounded": "Matrices are not symmetric",
                     "spd": "`x != x.transpose` with atol={atol}, rtol={rtol}"},
                 2: {"upper": "'x' determinant is not > 0",
                     "bounded": "'Id - conj(Z) Z' is not hermitian (is not definite positive)",
                     "spd": "eigenvalues of x are not all greater than 0."}}


def check_points(kind, table, atol=1e-5, rtol=1e-5):
    """Embeddings.check_all_points (sympa/embeddings.py:41-47) as one launch over the table: returns (True, None,
    None) or (False, index of the first offending row, reason) with the reference's reason strings.  One host
    synchronisation (the 8-byte verdict)."""
    table = _require(table, "table")
    n = table.shape[-1]
    _check_n(n)
    if tuple(table.shape[1:]) != _point_shape(kind, n):
        raise ValueError(f"table must have shape (N, {_point_shape(kind, n)})")
    with torch.cuda.device(table.device):
        verdict = torch.empty(1, dtype=torch.int64, device=table.device)
        _lib.check(_lib.load().sympa_check_points(_lib.KIND[kind], n, table.shape[0], _ptr(table), float(atol), float(rtol),
                                                  _ptr(verdict), _stream()))
        v = int(verdict.item()) & 0xFFFFFFFFFFFFFFFF
    if v == 0xFFFFFFFFFFFFFFFF:
        return True, None, None
    return False, v >> 8, CHECK_REASONS[v & 0xFF][kind].format(atol=atol, rtol=rtol)


def _require(t, name, dtype=torch.float64):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a tensor")
    if not t.is_cuda:
        raise RuntimeError(f"sympa_b200: {name} must be a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"sympa_b200: {name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def _point_shape(kind, n):
    return (n, n) if kind == "spd" else (2, n, n)


def _check_n(n):
    if not 1 <= n <= _lib.MAX_N:
        raise NotImplementedError(f"sympa_b200 supports matrix sizes 1..{_lib.MAX_N}, got {n}")


def forward_raw(kind, metric, z1=None, z2=None, table=None, idx=None, wsum_w=None, want_grad=False,
                want_vvd=True):
    """One forward launch.  Returns (dist, vvd or None, saved_state or None)."""
    lib = _lib.load()
    if table is not None:
        table = _require(table, "table")
        idx = _require(idx, "idx", torch.int64)
        if idx.dim() != 2 or idx.shape[1] != 2:
            raise ValueError("idx must have shape (num_pairs, 2)")
        n = table.shape[-1]
        if tuple(table.shape[1:]) != _point_shape(kind, n):
            raise ValueError(f"table must have shape (N, {_point_shape(kind, n)})")
        b, dev = idx.shape[0], table.device
    else:
        z1 = _require(z1, "z1")
        z2 = _require(z2, "z2")
        if z1.shape != z2.shape:
            raise ValueError("z1 and z2 must have the same shape")
        n = z1.shape[-1]
        if tuple(z1.shape[1:]) != _point_shape(kind, n):
            raise ValueError(f"points must have shape (b, {_point_shape(kind, n)}), got {tuple(z1.shape)}")
        b, dev = z1.shape[0], z1.device
    _check_n(n)
    if metric == "wsum" and kind != "spd":
        wsum_w = _require(wsum_w, "wsum_w").reshape(-1)
        if wsum_w.numel() != n:
            raise ValueError("wsum weights must have n entries")
    else:
        wsum_w = None
    with torch.cuda.device(dev):
        dist = torch.empty(b, dtype=torch.float64, device=dev)
        vvd = torch.empty(b, n, dtype=torch.float64, device=dev) if want_vvd else None
        saved = None
        if b == 0:   # nothing to launch (an empty tensor has a null data pointer)
            if want_grad:
                saved = torch.empty(0, dtype=torch.float64, device=dev)
            return dist, vvd, saved
        if want_grad:
            nbytes = lib.sympa_workspace_bytes(_lib.KIND[kind], n, b)
            saved = torch.empty(nbytes // 8, dtype=torch.float64, device=dev)
        scratch, scratch_bytes = scratch_for(kind, n, b, dev)
        _lib.check(lib.sympa_dist_forward(
            _lib.KIND[kind], n, _lib.METRIC[metric], b, _ptr(z1), _ptr(z2), _ptr(table),
            0 if table is None else table.shape[0], _ptr(idx), _ptr(wsum_w), _ptr(dist), _ptr(vvd), _ptr(saved),
            _ptr(scratch), scratch_bytes, _ptr(status_word(dev)), _stream()))
    return dist, vvd, saved


class _DistFn(torch.autograd.Function):
    """dist(z1, z2) on materialised (b, 2, n, n) / (b, n, n) operands - what the reference's
    Model.distance calls (sympa/model.py:32-38)."""

    @staticmethod
    def forward(ctx, z1, z2, wsum_w, kind, metric):
        need = any(ctx.needs_input_grad[:3])
        dist, vvd, saved = forward_raw(kind, metric, z1=z1, z2=z2, wsum_w=wsum_w, want_grad=need)
        ctx.kind, ctx.metric, ctx.shape = kind, metric, z1.shape
        ctx.save_for_backward(saved, vvd, wsum_w if metric == "wsum" else None)
        ctx.mark_non_differentiable(vvd)
        return dist, vvd

    @staticmethod
    def backward(ctx, grad_dist, _grad_vvd):
        saved, vvd, wsum_w = ctx.saved_tensors
        lib = _lib.load()
        grad_dist = _require(grad_dist, "grad_dist")
        b, n = vvd.shape
        dev = vvd.device
        if b == 0:
            z = torch.zeros(ctx.shape, dtype=torch.float64, device=dev)
            return z, z.clone(), (None if wsum_w is None else torch.zeros_like(wsum_w)), None, None
        with torch.cuda.device(dev):
            g1 = torch.empty(ctx.shape, dtype=torch.float64, device=dev)
            g2 = torch.empty(ctx.shape, dtype=torch.float64, device=dev)
            gw = None
            w_flat = None
            if wsum_w is not None and ctx.needs_input_grad[2]:
                gw = torch.zeros(n, dtype=torch.float64, device=dev)
                w_flat = wsum_w.contiguous().reshape(-1)
            _lib.check(lib.sympa_dist_backward(
                _lib.KIND[ctx.kind], n, _lib.METRIC[ctx.metric], b, _ptr(grad_dist), _ptr(saved), _ptr(g1), _ptr(g2),
                None, 0, None, _ptr(vvd), _ptr(w_flat), _ptr(gw), _stream()))
        if gw is not None:
            gw = gw.reshape(wsum_w.shape)
        return g1, g2, gw, None, None


def _world_size():
    import torch.distributed as dist
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def bounded_by_rows(kind, n, num_pairs, num_rows, sync_grad):
    """Route choice of the bounded domain on the table path (see _TableDistFn).  With sync_grad in a
    multi-process group the choice must not depend on rank-local state - the ranks put their result into ONE
    all-reduced buffer, and the by-rows route accumulates the gradient with respect to the TRANSFORMED rows -
    so there it depends on (kind, n) only; a single process also looks at how densely the batch covers the table."""
    if not (BOUNDED_BY_ROWS and kind == "bounded" and n <= BOUNDED_BY_ROWS_MAX_N and num_rows > 0):
        return False
    if sync_grad and _world_size() > 1:
        return True
    return 2 * num_pairs >= num_rows


# SMs the scatter of an accumulated chunk confines itself to while it runs on the accumulator's side stream next to
# the forward kernel of the following chunk (0: no overlap, the scatter runs on the caller's stream on all SMs)
ACC_SCATTER_SMS = int(os.environ.get("SYMPA_ACC_SCATTER_SMS", "48"))


class TableGradAccumulator:
    """Gradient accumulation over the dist_from_table calls of ONE step (the reference's grad_accum_steps,
    runner.py:104): the backward of every call scatter-adds into one packed gradient table, and finish() - once
    per step - runs the collective on it (optional), expands it into table.grad and zeroes it for the next step.
    Saves, per call after the first, the zeroing and expansion passes over the table and autograd's dense
    accumulation (0.26 ms of a 5.1 ms chunk at n = 4 and 2^20 rows), keeps the all-reduce of a multi-chunk step on
    the packed bytes, and - bounded domain by rows - transforms the table once per step instead of once per call
    (the transformed table is cached until finish(), or until the table is modified in place).

        acc = manifold.table_grad_accumulator(table)
        for idx_c, gd_c in chunks:
            loss_fn.calculate_loss(gd_c, manifold.dist_from_table(table, idx_c, accumulator=acc)).backward()
        acc.finish(sync_grad=world_size > 1)       # table.grad is ready (accumulated into if it already existed)
    """

    def __init__(self, kind, table, scatter_sms=None):
        lib = _lib.load()
        # the scatter of a chunk is bound by L2 atomics / DRAM and the forward kernel of the next chunk by the FP64
        # pipes: the scatter goes to a high-priority side stream and keeps to `scatter_sms` SMs (the two kernels
        # cannot share an SM: the pair kernel's two CTAs own the register file), finish() joins the streams
        # (n = 2 is bound by HBM, not by the FP64 pipes: its forward kernel is shorter than a scatter on a third of
        # the SMs, measured 8.9 -> 7.5 G pairs/s with the partition - no overlap there unless asked for)
        self.scatter_sms = (ACC_SCATTER_SMS if table.shape[-1] >= 3 else 0) if scatter_sms is None else int(scatter_sms)
        self.stream = torch.cuda.Stream(device=table.device, priority=-1) if self.scatter_sms > 0 else None
        self.tickets = torch.zeros(4, dtype=torch.int32, device=table.device)
        self._pending = False
        self._hold = None
        self._last = False
        self.table = table
        self.n, self.rows = table.shape[-1], table.shape[0]
        _check_n(self.n)
        self.by_rows = bool(BOUNDED_BY_ROWS and kind == "bounded" and self.n <= BOUNDED_BY_ROWS_MAX_N)
        self.kind = "upper" if self.by_rows else kind
        self.nbytes = lib.sympa_backward_workspace_bytes(_lib.KIND[self.kind], self.n, self.rows)
        self.ws = torch.zeros(self.nbytes // 8, dtype=torch.float64, device=table.device)
        self._src = self._src_of = None
        self._src_version = -1

    def source(self):
        """the table the pair kernels read: the table itself, or its inverse Cayley transform (cached per version)"""
        if not self.by_rows:
            return _require(self.table, "table").detach()
        if self._src is None or self._src_version != self.table._version:
            t = _require(self.table, "table").detach()
            src = torch.empty_like(t) if self._src is None else self._src
            with torch.cuda.device(t.device):
                _lib.check(_lib.load().sympa_bounded_rows_to_upper(self.n, self.rows, _ptr(t), _ptr(src),
                                                                   _ptr(status_word(t.device)), _stream()))
            self._src, self._src_of, self._src_version = src, t, self.table._version
        return self._src

    def scatter_add(self, kind, n, b, grad_dist, saved, idx):
        """this chunk's contribution into the packed table (called by the backward of dist_from_table)"""
        lib = _lib.load()
        k = _lib.KIND[kind]
        cur = torch.cuda.current_stream()
        self._join(cur)
        if self.stream is None or self._last:      # nothing to overlap with: the whole GPU, on the caller's stream
            _lib.check(lib.sympa_table_grad_scatter_add(k, n, b, _ptr(grad_dist), _ptr(saved), self.rows, _ptr(idx), _ptr(self.ws),
                                                        self.nbytes, 0, None, _stream()))
            return
        self.stream.wait_stream(cur)            # grad_dist and the saved state are ready, the table zeroed
        with torch.cuda.stream(self.stream):
            _lib.check(lib.sympa_table_grad_scatter_add(k, n, b, _ptr(grad_dist), _ptr(saved), self.rows, _ptr(idx), _ptr(self.ws),
                                                        self.nbytes, self.scatter_sms, _ptr(self.tickets), self.stream.cuda_stream))
        # The tensors the side stream reads belong to the caller's stream as far as the caching allocator knows.  They
        # are kept alive here until the caller's stream has waited for the scatter (_join: at the next chunk's
        # backward, by which time the scatter - overlapped with that chunk's forward - is over), so their memory
        # is reused in stream order.  (tensor.record_stream instead would leave every chunk's 2.7 GB state
        # unreusable for a host that enqueues many steps ahead: the allocator then grows until it has to
        # synchronise and free - measured: 1.88 -> 1.50 G pairs/s over 25 steps.)
        self._hold = (grad_dist, saved, idx)
        self._pending = True

    def _join(self, cur):
        if self._pending:
            cur.wait_stream(self.stream)
            self._pending = False
        self._hold = None

    def last_chunk(self):
        """hint: the next backward is the last one before finish() - no forward kernel follows it, so its scatter
        should use the whole GPU instead of the partition (optional; results do not depend on it)"""
        self._last = True

    def finish(self, sync_grad=False):
        lib = _lib.load()
        dev = self.table.device
        self._last = False
        self._join(torch.cuda.current_stream(dev))
        with torch.cuda.device(dev):
            if sync_grad:
                _allreduce_avg(self.ws)
            gt = torch.empty(self.table.shape, dtype=torch.float64, device=dev)
            _lib.check(lib.sympa_table_grad_expand(_lib.KIND[self.kind], self.n, self.rows, _ptr(self.ws), _ptr(gt), 1, _stream()))
            if self.by_rows:
                src_of = self._src_of if self._src_of is not None else _require(self.table, "table").detach()
                gz = torch.empty_like(gt)
                _lib.check(lib.sympa_bounded_rows_backward(self.n, self.rows, _ptr(src_of), _ptr(gt), _ptr(gz), 1, _stream()))
                gt = gz
            self.ws.zero_()
        self._src_version = -1      # an optimizer step follows (the fused one writes through raw pointers: no version bump)
        if self.table.grad is None:
            self.table.grad = gt
        else:
            self.table.grad.add_(gt)
        return self.table.grad


class _TableDistFn(torch.autograd.Function):
    """dist(table[idx[:,0]], table[idx[:,1]]) with the gather fused into the forward kernel and the
    gather backward (dense index_put in the reference, sympa/embeddings.py:29-34) fused into an
    atomic scatter-add."""

    @staticmethod
    def forward(ctx, table, idx, wsum_w, kind, metric, sync_grad=False, by_rows=None, acc=None):
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[2]
        ctx.acc = acc
        if acc is not None:     # gradient accumulation over the calls of a step: see TableGradAccumulator
            if acc.table is not table:
                raise ValueError("the accumulator was made for another table")
            dist, vvd, saved = forward_raw(acc.kind, metric, table=acc.source(), idx=idx, wsum_w=wsum_w, want_grad=need)
            ctx.kind, ctx.metric, ctx.tshape, ctx.sync_grad, ctx.by_rows = acc.kind, metric, table.shape, False, False
            ctx.save_for_backward(saved, vvd, idx, wsum_w if metric == "wsum" else None, None)
            ctx.mark_non_differentiable(vvd)
            return dist, vvd
        # bounded domain, batch covering the table densely: the inverse Cayley transform is applied once per
        # table row (sympa_bounded_rows_to_upper) and the pairs run the upper-half kernels on the result
        # (break-even in flops is 2 pairs per row)
        if by_rows is None:
            by_rows = table.is_cuda and idx.dim() == 2 and bounded_by_rows(kind, table.shape[-1], idx.shape[0],
                                                                           table.shape[0], sync_grad)
        by_rows = bool(by_rows) and kind == "bounded"
        src = table
        t = None
        if by_rows:
            t = _require(table, "table").detach()
            src = torch.empty_like(t)
            with torch.cuda.device(t.device):
                _lib.check(_lib.load().sympa_bounded_rows_to_upper(t.shape[-1], t.shape[0], _ptr(t), _ptr(src),
                                                                   _ptr(status_word(t.device)), _stream()))
        kk = "upper" if by_rows else kind
        dist, vvd, saved = forward_raw(kk, metric, table=src, idx=idx, wsum_w=wsum_w, want_grad=need)
        ctx.kind, ctx.metric, ctx.tshape, ctx.sync_grad, ctx.by_rows = kk, metric, table.shape, sync_grad, by_rows
        # (the contiguous copy `t`, not `table`: the backward hands its raw pointer to the row kernel)
        ctx.save_for_backward(saved, vvd, idx, wsum_w if metric == "wsum" else None, t)
        ctx.mark_non_differentiable(vvd)
        return dist, vvd

    @staticmethod
    def backward(ctx, grad_dist, _grad_vvd):
        saved, vvd, idx, wsum_w, ztable = ctx.saved_tensors
        lib = _lib.load()
        grad_dist = _require(grad_dist, "grad_dist")
        b, n = vvd.shape
        dev = vvd.device
        if ctx.acc is not None:
            acc = ctx.acc
            gw = None
            with torch.cuda.device(dev):
                k, m = _lib.KIND[ctx.kind], _lib.METRIC[ctx.metric]
                if b > 0:
                    acc.scatter_add(ctx.kind, n, b, grad_dist, saved, idx.contiguous())
                if wsum_w is not None and ctx.needs_input_grad[2]:
                    gw = torch.zeros(n, dtype=torch.float64, device=dev)
                    if b > 0:
                        _lib.check(lib.sympa_dist_backward(k, n, m, b, _ptr(grad_dist), _ptr(saved), None, None, None, 0, None,
                                                           _ptr(vvd), _ptr(wsum_w.contiguous().reshape(-1)), _ptr(gw), _stream()))
                    gw = gw.reshape(wsum_w.shape)
            return None, None, gw, None, None, None, None, None      # the table gradient arrives with acc.finish()
        with torch.cuda.device(dev):
            # every decision below depends on (kind, n, rows, sync_grad) only, never on the local batch: with
            # sync_grad all ranks must enter the same collectives on buffers of the same size, a rank with an
            # empty shard included
            gt = torch.empty(ctx.tshape, dtype=torch.float64, device=dev)     # written, not accumulated (overwrite=1)
            gw = None
            w_flat = None
            if wsum_w is not None and ctx.needs_input_grad[2]:
                gw = torch.zeros(n, dtype=torch.float64, device=dev)
                w_flat = wsum_w.contiguous().reshape(-1)
            ws, ws_bytes = backward_workspace_for(ctx.kind, n, ctx.tshape[0], dev)
            k, m, rows = _lib.KIND[ctx.kind], _lib.METRIC[ctx.metric], ctx.tshape[0]
            if ctx.sync_grad and ws is not None:
                # data-parallel backward: scatter into the packed gradient table, all-reduce (average) THAT - the
                # one collective of the path, on 62 % of the dense bytes at n = 4 - then write the dense rows
                need = lib.sympa_backward_workspace_bytes(k, n, rows)
                if _pipelined_sync():
                    # scatter the rows in SYNC_SEGMENTS ranges and start the all-reduce of a range as soon as it is
                    # complete: NCCL works on its own stream while the next range is scattered, so only the last
                    # range's collective is exposed (the segment count depends on nothing rank-local)
                    per_s = need // 8 // rows
                    seg = -(-rows // SYNC_SEGMENTS)
                    idx_c = idx.contiguous() if b > 0 else None
                    works = []
                    for lo in range(0, rows, seg):
                        hi = min(lo + seg, rows)
                        _lib.check(lib.sympa_table_grad_scatter_rows(
                            k, n, b, _ptr(grad_dist) if b > 0 else None, _ptr(saved) if b > 0 else None, rows, _ptr(idx_c),
                            lo, hi, _ptr(ws), ws_bytes, _stream()))
                        works.append(_allreduce_avg(ws[lo * per_s: hi * per_s], async_op=True))
                    if gw is not None and b > 0:
                        _lib.check(lib.sympa_dist_backward(k, n, m, b, _ptr(grad_dist), _ptr(saved), None, None, None, 0, None,
                                                           _ptr(vvd), _ptr(w_flat), _ptr(gw), _stream()))
                    for w in works:
                        if w is not None:
                            w.wait()
                else:
                    if b > 0:
                        _lib.check(lib.sympa_table_grad_scatter(k, n, m, b, _ptr(grad_dist), _ptr(saved), rows,
                                                                _ptr(idx.contiguous()), _ptr(vvd), _ptr(w_flat), _ptr(gw), _ptr(ws),
                                                                ws_bytes, _stream()))
                    else:
                        ws[: need // 8].zero_()
                    _allreduce_avg(ws[: need // 8])
                _lib.check(lib.sympa_table_grad_expand(k, n, rows, _ptr(ws), _ptr(gt), 1, _stream()))
            else:
                if b > 0:
                    _lib.check(lib.sympa_dist_backward_table(
                        k, n, m, b, _ptr(grad_dist), _ptr(saved), _ptr(gt), rows, _ptr(idx.contiguous()), _ptr(vvd), _ptr(w_flat),
                        _ptr(gw), _ptr(ws), ws_bytes, 1, _stream()))
                else:
                    gt.zero_()
                if ctx.sync_grad:
                    _allreduce_avg(gt)
            if ctx.sync_grad and gw is not None:
                _allreduce_avg(gw)
            if ctx.by_rows:   # gt is the gradient with respect to the transformed rows: back through the transform
                gz = torch.empty_like(gt)
                _lib.check(lib.sympa_bounded_rows_backward(n, rows, _ptr(ztable), _ptr(gt), _ptr(gz), 1, _stream()))
                gt = gz
        if gw is not None:
            gw = gw.reshape(wsum_w.shape)
        return gt, None, gw, None, None, None, None, None


def dist(kind, metric, z1, z2, wsum_w=None):
    """Differentiable distance and (non-differentiable) ascending vector-valued distance."""
    return _DistFn.apply(z1, z2, wsum_w, kind, metric)


# ranges the in-backward all-reduce of the packed table gradient is pipelined over (see _TableDistFn.backward).
# 1 = one scatter, one all-reduce.  Measured on 8 x B200 (n = 4, 2^23 pairs per rank, 168 MB packed table): with 4
# segments the step took 6.53 ms against 5.1 ms of compute - restricting the scatter to a row range makes every
# pass walk all (pair, element) work items again (1.4 -> 2.0 ms for four passes), which costs more than hiding
# three quarters of a 0.5 ms all-reduce gains.  The pipeline pays only where the scatter of a range is cheap.
SYNC_SEGMENTS = 1


def _pipelined_sync():
    import torch.distributed as dist
    return (SYNC_SEGMENTS > 1 and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
            and dist.get_backend() == "nccl")


def _allreduce_avg(t, async_op=False):
    """average over the ranks (what DDP does with the table gradient, train.py:59); no-op in a single process.
    async_op (NCCL only): returns the work handle - the collective is ordered after the kernels already enqueued
    on the current stream, later kernels do not wait for it until handle.wait()."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        if dist.get_backend() == "nccl":
            return dist.all_reduce(t, op=dist.ReduceOp.AVG, async_op=async_op)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        t.div_(dist.get_world_size())
    return None


def table_dist(kind, metric, table, idx, wsum_w=None, sync_grad=False, by_rows=None, accumulator=None):
    """sync_grad=True: the backward also averages the table gradient (and dL/dw of wsum) over the ranks of
    the default process group - on the packed gradient table where there is one - so the caller must NOT
    all-reduce table.grad again.  Every rank of the group must make the call (an empty local batch included).
    by_rows: force / forbid the bounded-domain row route (None: bounded_by_rows decides)."""
    if accumulator is not None and sync_grad:
        raise ValueError("with an accumulator the collective runs in accumulator.finish(sync_grad=True)")
    return _TableDistFn.apply(table, idx, wsum_w, kind, metric, bool(sync_grad), by_rows, accumulator)


def distortion_step(kind, metric, table, idx, graph_dist, scale, grad_table, wsum_w=None, grad_wsum_w=None,
                    grad_scale=None, loss_out=None, dist_out=None):
    """Fused training step of the distortion objective: accumulates into grad_table (and
    grad_wsum_w, grad_scale, loss_out when given).  Returns loss_out (a 1-element tensor)."""
    lib = _lib.load()
    table = _require(table, "table")
    idx = _require(idx, "idx", torch.int64)
    graph_dist = _require(graph_dist, "graph_dist")
    n = table.shape[-1]
    _check_n(n)
    dev = table.device
    if grad_table.shape != table.shape or not grad_table.is_contiguous():
        raise ValueError("grad_table must be a contiguous tensor shaped like table")
    if metric == "wsum" and kind != "spd":
        wsum_w = _require(wsum_w, "wsum_w").reshape(-1)
    else:
        wsum_w = None
    with torch.cuda.device(dev):
        scratch, scratch_bytes = scratch_for(kind, n, idx.shape[0], dev)
        if loss_out is None:
            loss_out = torch.zeros(1, dtype=torch.float64, device=dev)
        _lib.check(lib.sympa_distortion_step(
            _lib.KIND[kind], n, _lib.METRIC[metric], idx.shape[0], _ptr(table), table.shape[0], _ptr(idx),
            _ptr(graph_dist), float(scale), _ptr(wsum_w), _ptr(grad_table), _ptr(grad_wsum_w), _ptr(grad_scale),
            _ptr(loss_out), _ptr(dist_out), _ptr(scratch), scratch_bytes, _ptr(status_word(dev)), _stream()))
    return loss_out


_idx_workspace = {}


def dist_matrix(kind, metric, table, row_begin=0, row_count=None, wsum_w=None, chunk_pairs=1 << 24, out=None):
    """Rows [row_begin, row_begin + row_count) of the all-pairs distance matrix of `table` (forward only,
    zeros on the diagonal): sympa_dist_matrix.  The index workspace (16 bytes per pair of a chunk) is
    kept per device and reused.  out: an optional contiguous (row_count, N) float64 tensor on the table's
    device to write into (a streaming caller reuses one block buffer)."""
    lib = _lib.load()
    table = _require(table, "table").detach()
    n = table.shape[-1]
    _check_n(n)
    rows = table.shape[0]
    row_count = rows - row_begin if row_count is None else row_count
    if row_begin < 0 or row_count < 0 or row_begin + row_count > rows:
        raise ValueError("row range outside the table")
    if metric == "wsum" and kind != "spd":
        wsum_w = _require(wsum_w, "wsum_w").reshape(-1)
    else:
        wsum_w = None
    dev = table.device
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty(row_count, rows, dtype=torch.float64, device=dev)
        elif (out.dtype != torch.float64 or out.device != dev or tuple(out.shape) != (row_count, rows)
              or not out.is_contiguous()):
            raise ValueError(f"out must be a contiguous float64 ({row_count}, {rows}) tensor on {dev}")
        if row_count == 0 or rows == 0:
            return out
        chunk = max(1, min(chunk_pairs, row_count * rows))
        ws = _idx_workspace_for(dev, chunk)
        _lib.check(lib.sympa_dist_matrix(_lib.KIND[kind], n, _lib.METRIC[metric], _ptr(table), rows, row_begin, row_count,
                                         _ptr(wsum_w), _ptr(out), _ptr(ws), chunk, _ptr(status_word(dev)), _stream()))
    return out


def _idx_workspace_for(dev, chunk):
    """the per-device index workspace of dist_matrix and dist_rows, grown to 2 * chunk int64 on demand"""
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    ws = _idx_workspace.get(key)
    if ws is None or ws.numel() < 2 * chunk:
        ws = torch.empty(2 * chunk, dtype=torch.int64, device=dev)
        _idx_workspace[key] = ws
    return ws


def dist_rows(kind, metric, table, queries, wsum_w=None, out=None, chunk_pairs=1 << 24):
    """Rows queries[0], queries[1], ... of the all-pairs distance matrix of `table` (forward only): sympa_dist_rows,
    each row bit-identical to the same row of dist_matrix.  queries: 1-D int64 node ids on the table's device, in
    [0, N) (checked here, one host synchronisation), repeats allowed.  Returns the (Q, N) float64 block; `out` a
    contiguous (Q, N) float64 tensor to write into.  The index workspace is dist_matrix's, shared per device."""
    lib = _lib.load()
    table = _require(table, "table").detach()
    queries = _require(queries, "queries", torch.int64)
    n = table.shape[-1]
    _check_n(n)
    rows = table.shape[0]
    dev = table.device
    if queries.dim() != 1 or queries.device != dev:
        raise ValueError(f"queries must be a 1-D tensor on {dev}")
    q = queries.numel()
    if q and (rows == 0 or int(queries.min()) < 0 or int(queries.max()) >= rows):
        raise ValueError(f"queries must lie in [0, {rows})")
    if metric == "wsum" and kind != "spd":
        wsum_w = _require(wsum_w, "wsum_w").reshape(-1)
    else:
        wsum_w = None
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty(q, rows, dtype=torch.float64, device=dev)
        elif out.dtype != torch.float64 or out.device != dev or tuple(out.shape) != (q, rows) or not out.is_contiguous():
            raise ValueError(f"out must be a contiguous float64 ({q}, {rows}) tensor on {dev}")
        if q == 0:
            return out
        chunk = max(1, min(chunk_pairs, q * rows))
        ws = _idx_workspace_for(dev, chunk)
        _lib.check(lib.sympa_dist_rows(_lib.KIND[kind], n, _lib.METRIC[metric], _ptr(table), rows, _ptr(queries), q,
                                       _ptr(wsum_w), _ptr(out), _ptr(ws), chunk, _ptr(status_word(dev)), _stream()))
    return out


_topk_workspace = {}
TOPK_MAX_K = 1024


def row_topk(dist_block, k, exclude=None, out=None):
    """The k smallest entries of every row of the (R, M) float64 block `dist_block`: sympa_row_topk.  Entries
    compare by value (-0.0 equal to +0.0), then by column; column exclude[r] (1-D int64 on the block's device, -1
    for none) is left out of row r; NaN entries are never selected (they set the non-finite status bit).  Returns
    (ids (R, k) int64, values (R, k) float64), ascending, a row with fewer than k selectable entries padded with
    (-1, NaN): row r equals torch.sort(row, stable=True) with the excluded column removed, cut to k, NaN entries
    replaced by (-1, NaN).  1 <= k <= 1024.  `out` = (ids, values) to write into.  The workspace (16 bytes per
    candidate of a column slice) is kept per device and reused."""
    lib = _lib.load()
    dist_block = _require(dist_block, "dist_block")
    if dist_block.dim() != 2:
        raise ValueError("dist_block must be (rows, columns)")
    rows, cols = dist_block.shape
    dev = dist_block.device
    k = int(k)
    if not 1 <= k <= TOPK_MAX_K:
        raise ValueError(f"k must lie in [1, {TOPK_MAX_K}]")
    if exclude is not None:
        exclude = _require(exclude, "exclude", torch.int64)
        if exclude.device != dev or tuple(exclude.shape) != (rows,):
            raise ValueError(f"exclude must be a ({rows},) tensor on {dev}")
    if out is None:
        out = (torch.empty(rows, k, dtype=torch.int64, device=dev), torch.empty(rows, k, dtype=torch.float64, device=dev))
    else:
        ids, vals = out
        if (ids.dtype != torch.int64 or ids.device != dev or tuple(ids.shape) != (rows, k) or not ids.is_contiguous()
                or vals.dtype != torch.float64 or vals.device != dev or tuple(vals.shape) != (rows, k)
                or not vals.is_contiguous()):
            raise ValueError(f"out must be contiguous int64 and float64 ({rows}, {k}) tensors on {dev}")
        out = (ids, vals)
    if rows == 0:
        return out
    with torch.cuda.device(dev):
        nbytes = lib.sympa_row_topk_workspace_bytes(rows, cols, k)
        if nbytes < 0:
            raise ValueError(f"at most 2^31 - 1 rows per call, got {rows}")
        key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
        ws = _topk_workspace.get(key)
        if ws is None or ws.numel() * 8 < nbytes:
            ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=dev)
            _topk_workspace[key] = ws
        _lib.check(lib.sympa_row_topk(rows, cols, _ptr(dist_block), _ptr(exclude), k, _ptr(out[0]), _ptr(out[1]), _ptr(ws),
                                      ws.numel() * 8, _ptr(status_word(dev)), _stream()))
    return out


_rank_workspace = {}


def target_ranks(dist_block, queries, targets, filter_adj, out=None):
    """Filtered ranks of held-out targets among all N nodes: sympa_target_ranks.  dist_block: the (R, N) float64 block
    of the distance rows of `queries` ((R,) int64; what dist_rows returns).  targets = (ptr, idx): int64, ptr with
    R + 1 entries, the targets of block row r are idx[ptr[r]:ptr[r + 1]].  filter_adj = (ptr, idx): the CSR adjacency
    of all N nodes whose row u lists the known neighbours of u (graphs.adjacency_csr), left out of the competitors.
    All on the block's device.  Returns (lt, le): int64 tensors shaped like targets' idx, entry i the number of
    competitors strictly closer than, and at most as far as, the target idx[i] (definition in include/sympa_b200.h);
    -1 for every pair of a row with a NaN distance (which sets the non-finite status bit).  Only the entries
    [ptr[0], ptr[R]) are written; `out` = (lt, le) to write into, otherwise they are allocated filled with -1.  The
    workspace (8 bytes per row and 24 per entry of idx) is kept per device and reused."""
    lib = _lib.load()
    dist_block = _require(dist_block, "dist_block")
    if dist_block.dim() != 2:
        raise ValueError("dist_block must be (rows, N)")
    rows, n_cols = dist_block.shape
    dev = dist_block.device
    queries = _require(queries, "queries", torch.int64)
    t_ptr, t_idx = (_require(t, name, torch.int64) for t, name in zip(targets, ("targets ptr", "targets idx")))
    f_ptr, f_idx = (_require(t, name, torch.int64) for t, name in zip(filter_adj, ("filter ptr", "filter idx")))
    if any(t.device != dev for t in (queries, t_ptr, t_idx, f_ptr, f_idx)):
        raise ValueError("queries, targets and the filter must be on the distance block's device")
    if tuple(queries.shape) != (rows,):
        raise ValueError(f"queries must have shape ({rows},)")
    if t_ptr.dim() != 1 or t_ptr.numel() != rows + 1 or t_idx.dim() != 1:
        raise ValueError(f"targets ptr must have R + 1 = {rows + 1} entries and idx must be 1-D")
    if f_ptr.dim() != 1 or f_ptr.numel() != n_cols + 1 or f_idx.dim() != 1:
        raise ValueError(f"filter ptr must have N + 1 = {n_cols + 1} entries and idx must be 1-D")
    if out is None:
        out = (torch.full_like(t_idx, -1), torch.full_like(t_idx, -1))
    else:
        lt, le = out
        if any(o.dtype != torch.int64 or o.device != dev or o.shape != t_idx.shape or not o.is_contiguous()
               for o in (lt, le)):
            raise ValueError(f"out must be two contiguous int64 ({t_idx.numel()},) tensors on {dev}")
    if rows == 0 or n_cols == 0:
        return out
    with torch.cuda.device(dev):
        nbytes = lib.sympa_target_ranks_workspace_bytes(rows, t_idx.numel())
        key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
        ws = _rank_workspace.get(key)
        if ws is None or ws.numel() * 8 < nbytes:
            ws = torch.empty(nbytes // 8, dtype=torch.float64, device=dev)
            _rank_workspace[key] = ws
        dummy = None
        if t_idx.numel() == 0 or f_idx.numel() == 0:
            dummy = torch.zeros(1, dtype=torch.int64, device=dev)      # no entries: any valid pointer
        _lib.check(lib.sympa_target_ranks(rows, n_cols, _ptr(dist_block), _ptr(queries), _ptr(t_ptr),
                                          _ptr(t_idx if t_idx.numel() else dummy), _ptr(f_ptr),
                                          _ptr(f_idx if f_idx.numel() else dummy), _ptr(out[0] if out[0].numel() else dummy),
                                          _ptr(out[1] if out[1].numel() else dummy), _ptr(ws), ws.numel() * 8,
                                          _ptr(status_word(dev)), _stream()))
    return out


_ap_workspace = {}


def average_precision(dist_block, row_begin, adj, out=None):
    """Graph-reconstruction average precision of rows [row_begin, row_begin + R) of a distance matrix, given as
    the (R, N) block `dist_block` of those rows (what dist_matrix returns): sympa_average_precision.
    adj = (ptr, idx): the CSR adjacency of all N nodes on the block's device (graphs.adjacency_csr).  Returns
    (R,) float64, NaN for a node without neighbours; `out` (R,) to write into.  The workspace (16 bytes per row
    and per adjacency entry) is kept per device and reused.  Parity with the reference's metric code is
    unpinned (it is not available): the definition is the one in include/sympa_b200.h."""
    lib = _lib.load()
    dist_block = _require(dist_block, "dist_block")
    if dist_block.dim() != 2:
        raise ValueError("dist_block must be (rows, N)")
    ptr, idx = adj
    ptr = _require(ptr, "adjacency ptr", torch.int64)
    idx = _require(idx, "adjacency idx", torch.int64)
    rows, n_cols = dist_block.shape
    dev = dist_block.device
    if ptr.device != dev or idx.device != dev:
        raise ValueError("the adjacency must be on the distance block's device")
    if ptr.dim() != 1 or ptr.numel() != n_cols + 1 or idx.dim() != 1:
        raise ValueError(f"adjacency ptr must have N + 1 = {n_cols + 1} entries and idx must be 1-D")
    if row_begin < 0 or row_begin + rows > n_cols:
        raise ValueError("row range outside the matrix")
    if out is None:
        out = torch.empty(rows, dtype=torch.float64, device=dev)
    elif out.dtype != torch.float64 or out.device != dev or tuple(out.shape) != (rows,) or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous float64 ({rows},) tensor on {dev}")
    if rows == 0:
        return out
    with torch.cuda.device(dev):
        nbytes = lib.sympa_average_precision_workspace_bytes(rows, idx.numel())
        key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
        ws = _ap_workspace.get(key)
        if ws is None or ws.numel() * 8 < nbytes:
            ws = torch.empty(nbytes // 8, dtype=torch.float64, device=dev)
            _ap_workspace[key] = ws
        if idx.numel() == 0:
            idx = torch.zeros(1, dtype=torch.int64, device=dev)     # no entries: any valid pointer
        _lib.check(lib.sympa_average_precision(row_begin, rows, n_cols, _ptr(dist_block), _ptr(ptr), _ptr(idx), _ptr(out),
                                               _ptr(ws), ws.numel() * 8, _ptr(status_word(dev)), _stream()))
    return out


_hop_workspace = {}


def hop_distances(adj, row_begin, row_count, out=None):
    """Hop distances from the sources [row_begin, row_begin + row_count) to every node of the undirected graph
    adj = (ptr, idx) (the CSR adjacency of graphs.adjacency_csr, on a CUDA device), by breadth-first search on
    the device: sympa_hop_distances.  Returns the (row_count, N) int32 block, 0 on the diagonal and -1 where a
    node is unreachable; `out` to write into.  The workspace (one queue of N int32 per resident CTA, independent
    of row_count) is kept per device and reused."""
    lib = _lib.load()
    ptr, idx = adj
    ptr = _require(ptr, "adjacency ptr", torch.int64)
    idx = _require(idx, "adjacency idx", torch.int64)
    dev = ptr.device
    if idx.device != dev:
        raise ValueError("adjacency ptr and idx must be on the same device")
    if ptr.dim() != 1 or ptr.numel() < 1 or idx.dim() != 1:
        raise ValueError("adjacency ptr must be 1-D with N + 1 entries and idx must be 1-D")
    n_nodes = ptr.numel() - 1
    if row_begin < 0 or row_count < 0 or row_begin + row_count > n_nodes:
        raise ValueError("row range outside the graph")
    if out is None:
        out = torch.empty(row_count, n_nodes, dtype=torch.int32, device=dev)
    elif (out.dtype != torch.int32 or out.device != dev or tuple(out.shape) != (row_count, n_nodes)
          or not out.is_contiguous()):
        raise ValueError(f"out must be a contiguous int32 ({row_count}, {n_nodes}) tensor on {dev}")
    if row_count == 0:
        return out
    with torch.cuda.device(dev):
        nbytes = lib.sympa_hop_distances_workspace_bytes(n_nodes)
        if nbytes < 0:
            raise ValueError(f"graphs of {n_nodes} nodes are not supported (int32 node ids)")
        key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
        ws = _hop_workspace.get(key)
        if ws is None or ws.numel() * 8 < nbytes:
            ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=dev)
            _hop_workspace[key] = ws
        if idx.numel() == 0:
            idx = torch.zeros(1, dtype=torch.int64, device=dev)     # no entries: any valid pointer
        _lib.check(lib.sympa_hop_distances(row_begin, row_count, n_nodes, _ptr(ptr), _ptr(idx), _ptr(out), _ptr(ws),
                                           ws.numel() * 8, _ptr(status_word(dev)), _stream()))
    return out


_sample_workspace = {}


def sample_pairs(adj, sources, k, seed, epoch, out=None):
    """K = k training pairs per source of the undirected graph adj = (ptr, idx) (graphs.adjacency_csr, on a CUDA
    device), drawn uniformly with replacement from the nodes each source reaches, with their hop distances, by
    breadth-first search on the device: sympa_sample_pairs.  The draws are a fixed function of (seed, epoch, source,
    draw number), defined in include/sympa_b200.h.  sources: 1-D int64 node ids on adj's device.  Returns
    (src_dst_ids (S k, 2) int64, graph_distances (S k,) float64), the pairs of sources[i] in rows i k .. i k + k - 1:
    the tensors the trainers take.  out = (ids, gd) to write into.  A source outside [0, N) sets the status bit of
    an out-of-range index, one that reaches no other node its own bit (check_status); both get k pairs (u, u) at
    distance 0.  The workspace (about 8.25 bytes per node per resident CTA, independent of S and k) is kept per
    device and reused."""
    lib = _lib.load()
    ptr, idx = adj
    ptr = _require(ptr, "adjacency ptr", torch.int64)
    idx = _require(idx, "adjacency idx", torch.int64)
    sources = _require(sources, "sources", torch.int64)
    dev = ptr.device
    if idx.device != dev or sources.device != dev:
        raise ValueError("adjacency ptr, idx and sources must be on the same device")
    if ptr.dim() != 1 or ptr.numel() < 1 or idx.dim() != 1:
        raise ValueError("adjacency ptr must be 1-D with N + 1 entries and idx must be 1-D")
    if sources.dim() != 1:
        raise ValueError("sources must be 1-D")
    k, seed, epoch = int(k), int(seed), int(epoch)
    if k < 0:
        raise ValueError("k must be >= 0")
    if not (0 <= seed < 1 << 64 and 0 <= epoch < 1 << 64):
        raise ValueError("seed and epoch must lie in [0, 2^64)")
    n_nodes, s = ptr.numel() - 1, sources.numel()
    if s >= 1 << 31:
        raise ValueError("at most 2^31 - 1 sources per call")
    if n_nodes >= 1 << 31:
        raise ValueError(f"graphs of {n_nodes} nodes are not supported (int32 node ids)")
    if out is None:
        out = (torch.empty(s * k, 2, dtype=torch.int64, device=dev), torch.empty(s * k, dtype=torch.float64, device=dev))
    else:
        ids, gd = out
        if (ids.dtype != torch.int64 or ids.device != dev or tuple(ids.shape) != (s * k, 2) or not ids.is_contiguous()
                or gd.dtype != torch.float64 or gd.device != dev or tuple(gd.shape) != (s * k,) or not gd.is_contiguous()):
            raise ValueError(f"out must be contiguous int64 ({s * k}, 2) and float64 ({s * k},) tensors on {dev}")
        out = (ids, gd)
    if s * k == 0:
        return out
    with torch.cuda.device(dev):
        nbytes = lib.sympa_sample_pairs_workspace_bytes(n_nodes)
        key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
        ws = _sample_workspace.get(key)
        if ws is None or ws.numel() * 8 < nbytes:
            ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=dev)
            _sample_workspace[key] = ws
        if idx.numel() == 0:
            idx = torch.zeros(1, dtype=torch.int64, device=dev)     # no entries: any valid pointer
        _lib.check(lib.sympa_sample_pairs(n_nodes, _ptr(ptr), _ptr(idx), s, _ptr(sources), k, seed, epoch, _ptr(out[0]),
                                          _ptr(out[1]), _ptr(ws), ws.numel() * 8, _ptr(status_word(dev)), _stream()))
    return out


DistortionRows = collections.namedtuple("DistortionRows", "sum count max min")
DistortionRows.__doc__ = """Per-row distortion terms (sympa_distortion_rows): over the pairs (u, w > u) connected in the
graph, sum of |s d - g| / g (float64), the number of pairs (int64) and the extremes of s d / g (float64;
-inf / +inf for a row without pairs, NaN for a row with a NaN distance)."""


def distortion_rows(dist_block, hop_block, row_begin, scale, out=None, full=False):
    """Graph-reconstruction distortion terms of rows [row_begin, row_begin + R) of a distance matrix, from the
    (R, N) float64 block `dist_block` of those rows (dist_matrix) and the (R, N) int32 hop block of the same
    rows (hop_distances): sympa_distortion_rows over the columns w > u, or with full=True
    sympa_distortion_rows_full over every column w != u.  `scale` multiplies every distance (the model scale).
    Returns a DistortionRows of (R,) tensors; `out` a DistortionRows to write into.  A row's values are
    bit-identical whatever block it comes in.  Parity with the reference's metric code is unpinned (it is not
    available): the definition is the one in include/sympa_b200.h."""
    lib = _lib.load()
    dist_block = _require(dist_block, "dist_block")
    hop_block = _require(hop_block, "hop_block", torch.int32)
    if dist_block.dim() != 2:
        raise ValueError("dist_block must be (rows, N)")
    rows, n_cols = dist_block.shape
    dev = dist_block.device
    if hop_block.device != dev or tuple(hop_block.shape) != (rows, n_cols):
        raise ValueError(f"hop_block must be ({rows}, {n_cols}) on {dev}")
    if row_begin < 0 or row_begin + rows > n_cols:
        raise ValueError("row range outside the matrix")
    dtypes = DistortionRows(torch.float64, torch.int64, torch.float64, torch.float64)
    if out is None:
        out = DistortionRows(*(torch.empty(rows, dtype=t, device=dev) for t in dtypes))
    else:
        out = DistortionRows(*out)
        for o, t in zip(out, dtypes):
            if o.dtype != t or o.device != dev or tuple(o.shape) != (rows,) or not o.is_contiguous():
                raise ValueError(f"out must hold contiguous ({rows},) tensors on {dev} of dtypes {tuple(dtypes)}")
    if rows == 0:
        return out
    with torch.cuda.device(dev):
        fn = lib.sympa_distortion_rows_full if full else lib.sympa_distortion_rows
        _lib.check(fn(row_begin, rows, n_cols, _ptr(dist_block), _ptr(hop_block), float(scale),
                      *(_ptr(o) for o in out), _ptr(status_word(dev)), _stream()))
    return out


def rsgd_step(kind, table, grad, lr, lr_scale=None, projected=None, zero_grad=False):
    """In-place Riemannian SGD update of a CUDA table (one launch); see sympa_rsgd_step in the header.
    zero_grad=True also zeroes the gradient rows it applied."""
    lib = _lib.load()
    if not table.is_cuda or table.dtype != torch.float64 or not table.is_contiguous():
        raise RuntimeError("sympa_b200: rsgd_step needs a contiguous CUDA float64 table (there is no CPU path)")
    grad = _require(grad, "grad")
    n = table.shape[-1]
    _check_n(n)
    with torch.cuda.device(table.device):
        _lib.check(lib.sympa_rsgd_step_ex(_lib.KIND[kind], n, table.shape[0], table.data_ptr(), grad.data_ptr(), float(lr),
                                          _ptr(lr_scale), _ptr(projected), int(bool(zero_grad)), _stream()))
    return table
