"""Multi-GPU searches: one process per GPU (``torch.distributed``, NCCL over NVLink).

Two ways to shard, both with one exchange step at most (SURVEY.md 8e):

* **orientations** (``sharded_search``): the orientation list -- the reference's only
  parallel axis (``Pool.imap`` over angles, core.py:180-183) -- is split contiguously over
  the ranks; every rank holds the whole DEM and its own best state.  The exchange is the
  per-pixel best-SNR merge.  Default: an all-to-all of row bands (rank r receives every
  rank's candidates for band r and folds them on the device), after which each rank owns the
  merged result of its band and decodes / downloads only that; 12 bytes per pixel cross the
  links once.  ``merge_best_state`` is the replicated alternative (two all-reduces on packed
  keys and winner amplitudes), after which every rank holds the whole merged state.
* **rows** (``spatial_search``): the raster is cut into row bands with a halo
  (BASELINE config 5); a rank holds only its band of the DEM and of the best state, runs the
  whole orientation x age search on it, and no pixel data is exchanged at all -- only three
  scalars so that every band packs with the same curvature scale and learns about a NaN
  held by another band.

Stream rule: the plan's kernels run on the plan's stream, ``torch.distributed`` on torch's
current stream.  Unless they are the same stream (``Plan(stream=torch.cuda.current_stream()
.cuda_stream)``) every hand-over between the two is fenced with a host-side synchronise.
"""
import numpy as np


def shard_bounds(n_items, world_size, rank):
    """Contiguous shard [lo, hi) of ``n_items`` for ``rank`` (sizes differ by <= 1)."""
    base, extra = divmod(n_items, world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def _world(group):
    import torch.distributed as dist
    if not dist.is_initialized():
        return 1, 0
    return dist.get_world_size(group), dist.get_rank(group)


class _Fence(object):
    """Orders work between the plan's stream and torch's current stream on ``device``."""

    def __init__(self, plan, device):
        import torch
        self.plan = plan
        self.cuda = device is not None and torch.device(device).type == "cuda"
        self.same = False
        if self.cuda:
            self.torch_stream = torch.cuda.current_stream(device)
            self.same = int(self.torch_stream.cuda_stream) == plan.stream_handle

    def plan_done(self):
        """Plan kernels issued so far finish before torch work issued next starts."""
        if self.cuda and not self.same:
            self.plan.sync()

    def torch_done(self):
        """Torch work issued so far finishes before plan kernels issued next start."""
        if self.cuda and not self.same:
            self.torch_stream.synchronize()


class _DevView(object):
    """``__cuda_array_interface__`` over a raw device pointer (borrowed from the plan)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def _as_tensor(ptr, n, kind, device):
    """Zero-copy torch tensor over plan memory (CUDA), or over host memory for the CPU
    emulator build used by the gloo tests."""
    import torch
    dtype, typestr, ctype = {"f4": (torch.float32, "<f4", np.float32), "i4": (torch.int32, "<i4", np.int32)}[kind]
    if device is not None and torch.device(device).type == "cuda":
        return torch.as_tensor(_DevView(ptr, n, typestr), device=device)
    import ctypes
    buf = (ctypes.c_byte * (4 * n)).from_address(int(ptr))
    return torch.from_numpy(np.frombuffer(buf, dtype=ctype))


def merge_best_state(plan, device, group=None):
    """Replicated merge of state 0: all ranks end with the same merged best state in ``plan``
    (all-reduce MAX on packed keys, all-reduce SUM on the winners' amplitudes)."""
    import torch
    import torch.distributed as dist
    fence = _Fence(plan, device)
    n = (plan.row_hi - plan.row_lo) * plan.nx
    keys = torch.empty(n, dtype=torch.int64, device=device)
    amp = torch.empty(n, dtype=torch.float32, device=device)
    fence.torch_done()                       # the allocator may hand out memory torch still uses
    plan.best_pack(keys.data_ptr())
    fence.plan_done()
    dist.all_reduce(keys, op=dist.ReduceOp.MAX, group=group)
    fence.torch_done()
    plan.best_select(keys.data_ptr(), amp.data_ptr())
    fence.plan_done()
    dist.all_reduce(amp, op=dist.ReduceOp.SUM, group=group)
    fence.torch_done()
    plan.best_unpack(keys.data_ptr(), amp.data_ptr())
    fence.plan_done()                        # keys / amp may be freed by the caller
    return keys, amp


def merge_best_bands(plan, device, group=None, state=0):
    """Banded merge: rank r receives every rank's candidates for row band r (one all-to-all
    per plane) and folds them into its own best state there.  Afterwards this rank's best
    state is the merged result on rows ``shard_bounds(ny, world, rank)`` (other rows keep
    its own partial result).  Returns that band ``(row_lo, row_hi)``."""
    import torch
    import torch.distributed as dist
    world, rank = _world(group)
    ny, nx = plan.row_hi - plan.row_lo, plan.nx
    bands = [shard_bounds(ny, world, r) for r in range(world)]
    lo, hi = bands[rank]
    lo, hi = lo + plan.row_lo, hi + plan.row_lo
    if world == 1:
        return lo, hi
    fence = _Fence(plan, device)
    ps, pa, pi = plan.best_state_pointers(state)
    n = ny * nx
    send = [nx * (b - a) for a, b in bands]
    mine = nx * (hi - lo)
    recv = [mine] * world
    outs = []
    fence.plan_done()                        # the sweep's last writes to the best state
    for ptr, kind, dtype in ((ps, "f4", torch.float32), (pa, "f4", torch.float32), (pi, "i4", torch.int32)):
        src = _as_tensor(ptr, n, kind, device)
        dst = torch.empty(world * mine, dtype=dtype, device=device)
        dist.all_to_all_single(dst, src, output_split_sizes=recv, input_split_sizes=send, group=group)
        outs.append(dst)
    fence.torch_done()
    plan.best_merge(state, (lo, hi), world, outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr())
    fence.plan_done()                        # the candidate buffers are released on return
    return lo, hi


def merge_region_bands(plan, device, group=None):
    """Banded merge of the region planes after ``region_sweep`` over this rank's share: rank r
    receives every rank's planes for row band r (one all-to-all per plane) and replaces its own
    there by their fold (``Plan.region_merge``: counts summed, age ranks min / max, orientation
    words OR-ed -- NCCL has no OR reduction, so no all-reduce can do this).  Afterwards this rank's
    region planes are the merged result on rows ``shard_bounds(ny, world, rank)``; returns that band
    ``(row_lo, row_hi)``.  Bands, fences and receive buffer as ``merge_best_bands``; the buffer holds
    4 * (3 + words) B per pixel of the plan's rows."""
    import torch
    import torch.distributed as dist
    world, rank = _world(group)
    ny, nx = plan.row_hi - plan.row_lo, plan.nx
    bands = [shard_bounds(ny, world, r) for r in range(world)]
    lo, hi = bands[rank]
    lo, hi = lo + plan.row_lo, hi + plan.row_lo
    if world == 1:
        return lo, hi
    fence = _Fence(plan, device)
    ptr, n_planes = plan.region_planes()
    n = ny * nx
    send = [nx * (b - a) for a, b in bands]
    mine = nx * (hi - lo)
    recv = [mine] * world
    src = _as_tensor(ptr, n_planes * n, "i4", device).view(n_planes, n)
    dst = torch.empty((n_planes, world * mine), dtype=torch.int32, device=device)     # [plane][cand][row][nx]
    fence.plan_done()                        # the region pass's last writes to the planes
    for p in range(n_planes):
        dist.all_to_all_single(dst[p], src[p], output_split_sizes=recv, input_split_sizes=send, group=group)
    fence.torch_done()
    plan.region_merge((lo, hi), world, dst.data_ptr())
    fence.plan_done()                        # the candidate buffer is released on return
    return lo, hi


def _region_args(plan, name, ages, angles, snr_ratio):
    """Checked float64 ages and the region tables of a fit region; one best state."""
    from . import params as P
    from .core import search_args
    ages = search_args(name, ages, snr_ratio, max_ages=None, angles=angles)
    if plan.states != 1:
        plan.set_states(1)
    return ages, P.region_tables(ages, angles)


def _age_range_args(plan, name, ages, snr_ratio):
    """Checked float64 ages of an age range; one best state per age."""
    from .core import search_args
    ages = search_args(name, ages, snr_ratio)
    if plan.states != len(ages):
        plan.set_states(len(ages))
    return ages


def sharded_fit_region(plan, spec, scale, ages, angles, snr_ratio, device=None, group=None):
    """``core.fit_region`` over ranks sharing the orientation x age templates (DESIGN.md section 15),
    on ``plan`` over the whole raster (DEM already set, e.g. with ``set_dem_sharded``): this rank
    sweeps its share, the best states are merged replicated (every pixel's threshold needs the
    merged best), the region pass runs over the same share and the region planes are merged by row
    band.  Returns ``(row_lo, row_hi, stack)``, ``stack`` the (9, row_hi - row_lo, nx) rows of
    ``core.fit_region``'s result, bit for bit.  Raises ``core.fit_region``'s ``ValueError`` before any
    device work or collective."""
    ages, tables = _region_args(plan, "sharded_fit_region", ages, angles, snr_ratio)
    world, rank = _world(group)
    share = (rank, world) if world > 1 else None
    a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, "age_major", template_share=share)
    plan.reset()
    plan.sweep(a_rec, t_rec)
    if world > 1:
        merge_best_state(plan, device, group)
    plan.region_sweep(a_rec, t_rec, snr_ratio, tables)
    band = merge_region_bands(plan, device, group)
    return band + (plan.region_finalize(age_of, angle_of, tables, rows=band),)


def sharded_age_range(plan, spec, scale, ages, angles, snr_ratio, device=None, group=None):
    """``core.age_range`` over ranks sharing the orientation x age templates (DESIGN.md section 15):
    this rank sweeps its share with one best state per age, every state is merged by row band
    (``merge_best_bands``) and this rank reduces its band.  Returns ``(row_lo, row_hi, stack)``,
    ``stack`` the (6, row_hi - row_lo, nx) rows of ``core.age_range``'s result, bit for bit.  Raises
    ``core.age_range``'s ``ValueError`` before any device work or collective."""
    ages = _age_range_args(plan, "sharded_age_range", ages, snr_ratio)
    world, rank = _world(group)
    share = (rank, world) if world > 1 else None
    a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, "age_major", template_share=share,
                                                     state_per_age=True)
    plan.reset()
    plan.sweep(a_rec, t_rec)
    band = (plan.row_lo, plan.row_hi)
    for s in range(len(ages)):
        band = merge_best_bands(plan, device, group, state=s)
    return band + (plan.age_range(age_of, angle_of, snr_ratio, rows=band),)


def set_dem_sharded(plan, z, device, group=None):
    """``plan.set_dem(z)`` for an orientation-sharded search, where every rank needs the whole
    raster: rank r copies only rows ``shard_bounds(ny, world, r)`` host -> device and the ranks
    all-gather the rest over NVLink (one NCCL all-gather, in place) -- 1 / world of the PCIe
    traffic per rank.  ``z``: the same host float64 (ny, nx) raster on every rank, a NumPy array
    or a CPU ``torch.Tensor`` (a page-locked tensor makes the copy fast and asynchronous; it must
    not change before the search that follows has returned).  The device buffer stays with the
    plan."""
    import torch
    import torch.distributed as dist
    world, rank = _world(group)
    ny, nx = plan.ny, plan.nx
    if world == 1 or (plan.row_lo, plan.row_hi) != (0, ny):
        plan.set_dem(z)
        return
    if not isinstance(z, torch.Tensor):
        z = torch.from_numpy(np.ascontiguousarray(z, dtype=np.float64))
    if tuple(z.shape) != (ny, nx) or z.dtype != torch.float64 or z.device.type != "cpu" or not z.is_contiguous():
        raise ValueError("DEM: expected a contiguous host float64 raster of shape %r" % ((ny, nx),))
    per = -(-ny // world)                        # equal chunks for the all-gather; the tail is padding
    buf = plan.__dict__.get("_dem_shared")
    if buf is None or buf.device != torch.device(device):
        buf = plan.__dict__["_dem_shared"] = torch.zeros((world * per, nx), dtype=torch.float64, device=device)
    fence = _Fence(plan, device)
    fence.plan_done()                            # kernels of the last search may still read the buffer
    lo, hi = rank * per, min((rank + 1) * per, ny)
    if hi > lo:
        buf[lo:hi].copy_(z[lo:hi], non_blocking=True)
    dist.all_gather_into_tensor(buf.view(-1), buf[rank * per:(rank + 1) * per].view(-1), group=group)
    fence.torch_done()
    plan.set_dem_device(buf.data_ptr())


def sharded_search(plan, spec, scale, ages, angles, order="age_major", device=None,
                   group=None, finalize=True, merge="replicated"):
    """Run this rank's shard of the orientation search on ``plan`` (DEM already set), merge
    across ranks and decode.

    ``merge="replicated"``: every rank ends with the whole merged state and (with
    ``finalize``) returns the (4, ny, nx) stack.  ``merge="bands"``: rank r ends with the
    merged rows of band r and returns ``(row_lo, row_hi, stack)`` with ``stack`` of shape
    (4, row_hi - row_lo, nx) -- the distributed form of the result: nothing is decoded or
    downloaded twice.  ``finalize=False`` leaves the merged state in the plan."""
    world, rank = _world(group)
    # shares of the orientation-major template list that differ by at most one template (whole
    # orientations would differ by one orientation: 4 % at 181 over 8)
    a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, order,
                                                     template_share=(rank, world))
    plan.reset()
    plan.sweep(a_rec, t_rec)
    if merge == "bands":
        band = merge_best_bands(plan, device, group) if world > 1 else (plan.row_lo, plan.row_hi)
        if not finalize:
            return band + (None,)
        return band + (plan.finalize(age_of, angle_of, rows=band),)
    if world > 1:
        merge_best_state(plan, device, group)
    if not finalize:
        return None
    return plan.finalize(age_of, angle_of)


# ---------------------------------------------------------------------------
# spatial sharding
# ---------------------------------------------------------------------------
def slab_halo(spec, scale, ages, angles, nx, ny, de):
    """Rows of halo a band needs on either side: the largest template support along y over
    the whole search, plus the curvature stencil (dem.py:88-99) and one row of slack."""
    from . import params as P
    scales = [scale] if np.ndim(scale) == 0 else list(scale)
    need = 0
    for sc in scales:
        x, y = P.axis_vectors(nx, ny, de)
        recs = P.template_records(spec, sc, np.atleast_1d(np.asarray(ages, dtype=np.float64)),
                                  np.asarray(angles, dtype=np.float64), nx, ny, de, x, y,
                                  np.arange(len(angles)), np.zeros((len(angles), np.size(ages)), dtype=np.int64))
        need = max(need, int(-recs["sy_lo"].min()), int(recs["sy_hi"].max()))
    return need + 3


def share_dem_stats(plan, device=None, group=None):
    """Sum the curvature statistics of all bands (3 scalars; SUM carries a NaN) and hand the
    totals to the plan: every band then packs curv**2 with the same power of two and knows
    about a NaN anywhere in the raster (dem.py:105 through the reference's full-raster fft2)."""
    import torch
    import torch.distributed as dist
    world, _ = _world(group)
    s, n = plan.curv_stats()
    if world > 1:
        t = torch.tensor([s, n], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        s, n = (float(v) for v in t.tolist())
    plan.set_curv_stats(s, n)


def spatial_plan(ny, nx, dx, dy, spec, scale, ages, angles, group=None, **plan_kwargs):
    """This rank's plan for a raster sharded by row bands: ``(plan, (row_lo, row_hi))``.
    Upload the band with ``plan.set_dem`` (whole raster or just ``plan.dem_rows()``) or
    ``plan.set_dem_device``, then call ``share_dem_stats`` and ``spatial_search``."""
    from .engine import Plan
    world, rank = _world(group)
    lo, hi = shard_bounds(ny, world, rank)
    halo = slab_halo(spec, scale, ages, angles, nx, ny, dx)
    plan = Plan(ny, nx, dx, dy, slab=(lo, hi, halo), **plan_kwargs)
    return plan, (lo, hi)


def spatial_search(plan, spec, scale, ages, angles, order="age_major", finalize=True):
    """The whole orientation x age search on this rank's band (DEM set, statistics shared).
    Returns ``(row_lo, row_hi, stack)``; no data-path collective."""
    a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, order)
    plan.reset()
    plan.sweep(a_rec, t_rec)
    if not finalize:
        return plan.row_lo, plan.row_hi, None
    return plan.row_lo, plan.row_hi, plan.finalize(age_of, angle_of)


def spatial_fit_region(plan, spec, scale, ages, angles, snr_ratio):
    """``core.fit_region`` on this rank's band (DEM set, statistics shared): both passes on the slab
    plan.  Returns ``(row_lo, row_hi, stack)`` with ``stack`` of shape (9, row_hi - row_lo, nx); no
    data-path collective."""
    ages, tables = _region_args(plan, "spatial_fit_region", ages, angles, snr_ratio)
    a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles)
    plan.reset()
    plan.sweep(a_rec, t_rec)
    plan.region_sweep(a_rec, t_rec, snr_ratio, tables)
    return plan.row_lo, plan.row_hi, plan.region_finalize(age_of, angle_of, tables)


def spatial_age_range(plan, spec, scale, ages, angles, snr_ratio):
    """``core.age_range`` on this rank's band (DEM set, statistics shared; create the plan with
    ``spatial_plan(..., states=len(ages))`` to avoid a reallocation).  Returns ``(row_lo, row_hi,
    stack)`` with ``stack`` of shape (6, row_hi - row_lo, nx); no data-path collective."""
    ages = _age_range_args(plan, "spatial_age_range", ages, snr_ratio)
    a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, "age_major", state_per_age=True)
    plan.reset()
    plan.sweep(a_rec, t_rec)
    return plan.row_lo, plan.row_hi, plan.age_range(age_of, angle_of, snr_ratio)
