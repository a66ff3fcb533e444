"""Grid points across the GPUs of one box (SURVEY 8e): every point is independent
(reference pmlib.py:229-242 reads only shared read-only inputs), so ranks take
disjoint, equally heavy shares and the (N, 5) result table is assembled with one
all-gather.  No collective runs during the compute.

One process per GPU, launched by torchrun; ``torch.distributed`` only does the
plumbing (NCCL on GPUs, gloo in the CPU tests)."""
import numpy as np


def _dist():
    try:
        import torch.distributed as dist
    except ImportError:
        return None
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


def shard_indices(border, world_size, rank):
    """Indices of the points rank ``rank`` computes: points sorted by search radius
    (work per point ~ (2*border+1)^2) and dealt round-robin, so every rank gets the
    same mix of cheap and expensive points."""
    border = np.asarray(border, dtype=np.float64)
    order = np.argsort(-border, kind='stable')
    return np.sort(order[rank::world_size])


def gather_rows(local_rows, local_idx, n_total, dist, device=None):
    """All-gather the per-rank (n_r, 5) tables (padded to equal length) and scatter
    them back to the original point order.  One collective."""
    import torch
    world = dist.get_world_size()
    n_max = -(-n_total // world)
    pack = torch.full((n_max, 6), float('nan'), dtype=torch.float64)
    pack[:len(local_idx), 0] = torch.from_numpy(np.asarray(local_idx, dtype=np.float64))
    pack[:len(local_idx), 1:] = torch.from_numpy(np.ascontiguousarray(local_rows, dtype=np.float64))
    if device is not None:
        pack = pack.to(device)
    gathered = torch.empty((world * n_max, 6), dtype=torch.float64, device=pack.device)
    dist.all_gather_into_tensor(gathered, pack)
    g = gathered.cpu().numpy()
    keep = ~np.isnan(g[:, 0])
    out = np.full((n_total, 5), np.nan, dtype=np.float64)
    out[g[keep, 0].astype(np.int64)] = g[keep, 1:]
    return out


def _collective_device(dist, device=None):
    """Device the gather tensors live on: the compute context's GPU on NCCL (NOT torch's current device, which is
    cuda:0 in every rank unless the caller set it), None / CPU on gloo."""
    if dist.get_backend() != 'nccl':
        return None
    import torch
    from . import _lib
    return torch.device('cuda', _lib.default_context(device).device)


def _refuse_uncertainty(kwargs, name):
    if kwargs.get('uncertainty'):
        raise ValueError("uncertainty=True runs on one GPU: it is not supported by %s (use pmlib.use_mcc_batch)" % name)


def use_mcc_batch_sharded(c1, r1, c2fg, r2fg, border, img1, img2, img_size, alpha0, compute=None, **kwargs):
    """``use_mcc_batch`` over all ranks of an initialised process group (falls back to
    a plain single-GPU call when there is none).  Every rank passes the same inputs
    and receives the full table.  ``compute`` is the per-shard function (the GPU
    batch by default; the CPU tests inject a stand-in)."""
    _refuse_uncertainty(kwargs, 'use_mcc_batch_sharded')
    if compute is None:
        from .pmlib import use_mcc_batch as compute
    dist = _dist()
    n = len(c1)
    if dist is None or n == 0:
        return compute(c1, r1, c2fg, r2fg, border, img1, img2, img_size, alpha0, **kwargs) if n else np.zeros((0, 5))
    rank, world = dist.get_rank(), dist.get_world_size()
    idx = shard_indices(border, world, rank)
    arrs = [np.asarray(a, dtype=np.float64)[idx] for a in (c1, r1, c2fg, r2fg, border)]
    local = compute(*arrs, img1, img2, img_size, alpha0, **kwargs) if len(idx) else np.zeros((0, 5))
    return gather_rows(local, idx, n, dist, _collective_device(dist, kwargs.get('device')))


# ---------------------------------------------------------------------------------------------------------
# north_star's multi-GPU data plane for ONE pair: every rank uploads one row slab of each image, an in-place
# all-gather over NVLink completes the padded image buffers on every GPU (replaces the fork / copy-on-write
# replication of the reference's Pool, pmlib.py:430-448), the points are dealt by search radius, the kernel writes
# its rows straight into its slab of a result buffer, and ONE all-gather assembles the table.

class SplitPlan(object):
    """Row slabs of an image of ``rows`` lines over ``world`` ranks (equal slabs, the last one padded)."""

    def __init__(self, rows, cols, world):
        from . import _lib
        self.rows, self.cols, self.world = int(rows), int(cols), int(world)
        self.pitch, self.bytes = _lib.pair_layout(rows, cols)
        self.rows_per = -(-self.rows // self.world)
        self.slab = self.rows_per * self.pitch                       # bytes every rank contributes
        self.gather_bytes = self.slab * self.world                   # >= rows * pitch
        self.alloc_bytes = max(self.bytes, self.gather_bytes) + 256  # tail slack of the layout included

    def row_range(self, rank):
        r0 = min(self.rows, rank * self.rows_per)
        return r0, min(self.rows, r0 + self.rows_per)


_split_buffers = {}


def _split_buffer(key, plan, device):
    """Cached zero-initialised device buffer (torch uint8, 256-byte aligned by the allocator)."""
    import torch
    buf = _split_buffers.get(key)
    if buf is None or buf.numel() < plan.alloc_bytes or buf.device != device:
        buf = torch.zeros(plan.alloc_bytes, dtype=torch.uint8, device=device)
        _split_buffers[key] = buf
    return buf


def replicate_pair(img1, img2, dist, ctx=None, device=None):
    """Make ``img1`` / ``img2`` resident on EVERY rank's GPU while each rank transfers only 1/world of them over
    PCIe: rank r copies rows ``SplitPlan.row_range(r)`` of both images host -> device into its slab of the padded
    buffers (one asynchronous 2-D copy per image on the compute stream), then one in-place
    ``all_gather_into_tensor`` per image fills the rest over NVLink -- image 1's all-gather runs while image 2's
    slab is still uploading.  The context adopts the buffers without a copy (``sid_adopt_pair_device``).  Returns
    (bytes this rank uploaded, [(buffer, plan), (buffer, plan)])."""
    import torch
    from . import _lib
    ctx = ctx or _lib.default_context(device)
    rank, world = dist.get_rank(), dist.get_world_size()
    nccl = dist.get_backend() == 'nccl'
    dev = torch.device('cuda', ctx.device) if nccl else torch.device('cpu')
    uploaded = 0
    bufs = []
    for k, img in enumerate((img1, img2)):
        img = _lib.as_u8_image(img)
        plan = SplitPlan(img.shape[0], img.shape[1], world)
        buf = _split_buffer((ctx.device if nccl else 'cpu', k), plan, dev)
        r0, r1 = plan.row_range(rank)
        mine = buf[rank * plan.slab:(rank + 1) * plan.slab]
        if nccl:
            uploaded += ctx.upload_rows(mine.data_ptr(), plan.pitch, img[r0:r1])
        elif r1 > r0:
            mine.view(plan.rows_per, plan.pitch)[:r1 - r0, :plan.cols].copy_(torch.from_numpy(img[r0:r1]))
            uploaded += (r1 - r0) * plan.cols
        whole = buf[:plan.gather_bytes]
        # in place: NCCL's all-gather is in place when the send buffer is the rank's own slot of the receive buffer
        dist.all_gather_into_tensor(whole, mine if nccl else mine.clone())
        bufs.append((buf, plan))
    if nccl:
        (b1, p1), (b2, p2) = bufs
        ctx.adopt_pair_device(b1.data_ptr(), (p1.rows, p1.cols), p1.pitch, b1.numel(),
                              b2.data_ptr(), (p2.rows, p2.cols), p2.pitch, b2.numel())
    return uploaded, bufs


def shard_all(border, world):
    """``shard_indices`` of every rank from ONE sort."""
    border = np.asarray(border, dtype=np.float64)
    if border.size and border.min() == border.max():             # uniform radius: the stable sort is the identity
        return [np.arange(r, border.size, world) for r in range(world)]
    order = np.argsort(-border, kind='stable')
    return [np.sort(order[r::world]) for r in range(world)]


def use_mcc_batch_split(c1, r1, c2fg, r2fg, border, img1, img2, img_size, alpha0, **kwargs):
    """``use_mcc_batch`` for ONE pair over all ranks of the NCCL process group (north_star's split): the pair is
    replicated by :func:`replicate_pair` (1/world of it per PCIe link + one all-gather over NVLink), the points are
    dealt by :func:`shard_indices`, every rank's kernel writes its rows into its slab of the result buffer and one
    ``all_gather_into_tensor`` assembles the (N, 5) table on every rank.  Everything is enqueued on torch's current
    stream (slab copies, collectives, kernels), so the only host synchronisation is the final read-back.  Every rank
    passes the same arguments.  Falls back to :func:`use_mcc_batch_sharded` (each rank uploads the whole pair)
    without NCCL."""
    _refuse_uncertainty(kwargs, 'use_mcc_batch_split')
    dist = _dist()
    n = len(c1)
    if dist is None or dist.get_backend() != 'nccl' or n == 0:
        return use_mcc_batch_sharded(c1, r1, c2fg, r2fg, border, img1, img2, img_size, alpha0, **kwargs)
    import torch
    from . import _lib
    ctx = _lib.default_context(kwargs.get('device'))
    dev = torch.device('cuda', ctx.device)
    rank, world = dist.get_rank(), dist.get_world_size()
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)
    try:
        replicate_pair(img1, img2, dist, ctx)
        border = np.asarray(border, dtype=np.float64)
        parts = shard_all(border, world)
        idx = parts[rank]
        n_max = -(-n // world)
        pts = np.full((5, n_max), np.nan, dtype=np.float64)           # padding rows: rejected up front, NaN out
        for k, arr in enumerate((c1, r1, c2fg, r2fg, border)):
            pts[k, :len(idx)] = np.asarray(arr, dtype=np.float64)[idx]
        d_pts = torch.from_numpy(pts).to(dev, non_blocking=True)
        table = torch.empty((world, n_max, 5), dtype=torch.float64, device=dev)
        flags = _lib.flags_from_options(kwargs)
        ctx.run_device(n_max, *[d_pts[k].data_ptr() for k in range(5)], int(np.nanmax(border)), img_size,
                       list(kwargs.get('angles', [-3, 0, 3])), alpha0, table[rank].data_ptr(),
                       rot_order=kwargs.get('rot_order', 0), flags=flags, mtype=kwargs.get('mtype', _lib.SID_TM_CCOEFF_NORMED))
        dist.all_gather_into_tensor(table.view(world * n_max, 5), table[rank])        # in place, the ONE result collective
        host_t = _staging('split_recv', (world, n_max, 5), dev)
        host_t.copy_(table, non_blocking=True)
        stream.synchronize()
        host = host_t.numpy()
    finally:
        ctx.set_stream(None)
    out = np.empty((n, 5), dtype=np.float64)
    uniform = border.min() == border.max()
    for r in range(world):
        if uniform:
            out[r::world] = host[r, :len(parts[r])]                   # strided slab: a plain strided copy
        else:
            out[parts[r]] = host[r, :len(parts[r])]
    return out


def shard_pairs(n_pairs, world_size, rank):
    """Indices of the image pairs of a time series that rank ``rank`` processes (BASELINE configs[4]: whole
    pairs are dealt round-robin, so no image is replicated and nothing is exchanged during the compute)."""
    return list(range(rank, n_pairs, world_size))


def use_mcc_series(pairs, img_size, alpha0=0.0, n_contexts=1, compute=None, gather=True, **kwargs):
    """Pattern matching for a time series of image pairs: the batched form of calling the reference's
    ``pattern_matching`` Pool section (pmlib.py:430-448) once per pair.

    ``pairs`` is a sequence whose items are ``(img1, img2, c1, r1, c2fg, r2fg, border)`` tuples or zero-argument
    callables returning one (lazy loading: a rank only ever touches its own pairs).  Pairs are dealt round-robin
    to the ranks of the process group (``shard_pairs``); inside a rank every pair goes through
    ``Context.run_pair`` (banded upload overlapped with the kernels).  ``n_contexts`` > 1 lets several contexts work
    through the rank's pairs concurrently (threads); measured on B200 this is SLOWER than one context (9.4 vs
    11.0 ms per EW pair for 1 / 2 contexts at the end of round 2, 13.2 / 14.0 / 16.8 ms for 1 / 2 / 3 in round 1: the
    persistent kernels and band uploads of two pairs only delay each other), so the default is 1.  Returns the list of (n_k, 5) tables ``[c2, r2, angle, r, h]`` in pair order -- complete on
    every rank when ``gather`` is true (one all-gather of the padded tables); with ``gather='root'`` only rank 0
    reads the gathered tables back (the other ranks keep ``None`` for foreign pairs, as with ``gather=False``) --
    the cheaper choice when one process writes the products, since the read-back is host-memory bound.

    ``compute(ctx_slot, img1, img2, c1, r1, c2fg, r2fg, border)`` is the per-pair function (the GPU
    ``Context.run_pair`` by default; the CPU tests inject a stand-in)."""
    import queue
    import threading
    _refuse_uncertainty(kwargs, 'use_mcc_series')
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
    mine = shard_pairs(len(pairs), world, rank)
    results = [None] * len(pairs)
    n_contexts = max(1, min(int(n_contexts), max(1, len(mine))))
    if compute is None:
        from . import _lib
        # the reference's own defaults (pmlib.py:36, 118-121): hes_norm=True, hes_smth=False, mcc_norm=False
        flags = _lib.flags_from_options(kwargs)
        angles = kwargs.get('angles', [-3, 0, 3])
        rot_order = kwargs.get('rot_order', 0)
        mtype = kwargs.get('mtype', _lib.SID_TM_CCOEFF_NORMED)
        ctxs = [_lib.default_context()] + [_lib.Context(_lib.default_context().device) for _ in range(n_contexts - 1)]

        def compute(slot, img1, img2, c1, r1, c2fg, r2fg, border):
            return ctxs[slot].run_pair(img1, img2, c1, r1, c2fg, r2fg, border, img_size, angles, alpha0,
                                       rot_order=rot_order, flags=flags, mtype=mtype)
    work = queue.Queue()
    for k in mine:
        work.put(k)
    errors = []

    def worker(slot):
        while True:
            try:
                k = work.get_nowait()
            except queue.Empty:
                return
            try:
                item = pairs[k]() if callable(pairs[k]) else pairs[k]
                results[k] = np.asarray(compute(slot, *item), dtype=np.float64).reshape(-1, 5)
            except BaseException as exc:      # surfaced on the calling thread
                errors.append(exc)
                return

    threads = [threading.Thread(target=worker, args=(s,)) for s in range(1, n_contexts)]
    for t in threads:
        t.start()
    worker(0)
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    if dist is None or not gather:
        return results
    return _gather_series(results, mine, len(pairs), dist, root_only=(gather == 'root'))


_pinned = {}


def _staging(name, shape, device):
    """Cached page-locked float64 staging buffer (NCCL path only; plain tensors on CPU/gloo)."""
    import torch
    if device.type != 'cuda':
        return torch.empty(shape, dtype=torch.float64)
    n = int(np.prod(shape))
    buf = _pinned.get(name)
    if buf is None or buf.numel() < n:
        buf = torch.empty((max(n, 1),), dtype=torch.float64).pin_memory()
        _pinned[name] = buf
    return buf[:n].view(*shape)


def _gather_series(results, mine, n_pairs, dist, root_only=False):
    """Exchange the per-pair tables: one all-gather of the table lengths, one of the NaN-padded tables.  On
    NCCL the tables travel host -> device -> all ranks -> host through cached pinned staging buffers."""
    import torch
    world = dist.get_world_size()
    device = _collective_device(dist) or torch.device('cpu')
    per_rank = -(-n_pairs // world)
    sizes = torch.full((per_rank,), -1, dtype=torch.int64)
    for j, k in enumerate(mine):
        sizes[j] = results[k].shape[0]
    all_sizes = torch.empty((world * per_rank,), dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(all_sizes, sizes.to(device))
    all_sizes = all_sizes.cpu().numpy().reshape(world, per_rank)
    n_max = max(1, int(all_sizes.max()))
    pack = _staging('send', (per_rank, n_max, 5), device)
    for j in range(per_rank):
        n_j = results[mine[j]].shape[0] if j < len(mine) else 0
        if n_j:
            pack[j, :n_j] = torch.from_numpy(results[mine[j]])
        pack[j, n_j:] = float('nan')
    gathered = torch.empty((world * per_rank, n_max, 5), dtype=torch.float64, device=device)
    dist.all_gather_into_tensor(gathered, pack.to(device, non_blocking=True))
    if root_only and dist.get_rank() != 0:
        return results                      # the exchange on the device is collective; only rank 0 reads it back
    host = _staging('recv', (world, per_rank, n_max, 5), device)
    host.copy_(gathered.view(world, per_rank, n_max, 5), non_blocking=True)
    if device.type == 'cuda':
        torch.cuda.current_stream(device).synchronize()
    g = host.numpy()
    out = [None] * n_pairs
    for r in range(world):
        for j, k in enumerate(shard_pairs(n_pairs, world, r)):
            # own tables are returned as they are; foreign ones are copied out of the reusable staging buffer
            out[k] = results[k] if results[k] is not None else g[r, j, :int(all_sizes[r, j])].copy()
    return out


def bind_rank_to_gpu(device):
    """Restrict the calling process to the CPU cores that are local to CUDA device ``device`` (NVML's CPU
    affinity of the GPU), so that page-locked host buffers allocated afterwards -- the image pairs that
    ``run_pair`` uploads every step -- live on the GPU's own NUMA node.  For one-process-per-GPU jobs; call it
    before allocating pinned memory.  Returns the sorted core list, or None when NVML / the affinity API is not
    available or the result would be empty (nothing is changed then)."""
    import os
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(device).uuid)
        if not uuid.startswith("GPU-"):
            uuid = "GPU-" + uuid
        handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (ncpu + 63) // 64)
        cpus = {64 * w + bit for w, mask in enumerate(words) for bit in range(64) if (int(mask) >> bit) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except Exception:       # no NVML, no permission, unknown device: leave the affinity alone
        return None
