"""Device-side coverage step: grid-resident state and the calls into libmfgp_b200's cov_* / choi_* entry points.

`CoverageGrid` keeps the environment grid (coordinates, ground truth) in HBM for the whole simulation and owns the
output / workspace buffers of `cov_assign_reduce`; `BoundedVoronoi` is the host-side polygon set the reference gets
from scipy/Qhull (simulator.py:154-191), flattened for the device.
"""
import ctypes
import itertools
import math

import numpy as np
import torch
from scipy.spatial import Voronoi

from . import _native as nat

EPS = 0.1            # boundary cushion, simulator.py:33
TIE_TOL = 1e-9       # |d2_second - d2_best| below which the exact crossings test decides membership
AMAX_REL = 1e-10     # arg-max ties: |dvar| <= AMAX_REL * (k(0) - var) counts as tied, first index wins (argmax.cuh)


def host_array_key(arr):
    """Identity key of a host array for the device-copy caches (predict's x_star, the free coverage functions' truth_arr):
    address, shape, strides plus a checksum of a strided sample of <= 257 rows, so an in-place edit of the array between
    two calls is noticed in all but contrived cases (O(1): the reference's loops pass the same million-point array every
    iteration)."""
    arr = np.asarray(arr)
    n = arr.shape[0] if arr.ndim else 0
    step = max(1, n // 256)
    sample = arr[::step]
    return (arr.__array_interface__["data"][0], arr.shape, arr.strides, hash(sample.tobytes()))


def in_box(points, bounding_box):
    """simulator.py:139-151."""
    return np.logical_and(np.logical_and(bounding_box[0] - EPS <= points[:, 0], points[:, 0] <= bounding_box[1] + EPS),
                          np.logical_and(bounding_box[2] - EPS <= points[:, 1], points[:, 1] <= bounding_box[3] + EPS))


class BoundedVoronoi:
    """Bounded Voronoi partition as the reference builds it (simulator.py:154-191): seeds inside the cushioned box are
    mirrored across its four sides, Qhull computes the diagram of the 5A points and the first A regions are the
    bounded cells.  Keeps the reference's attribute names (`vertices`, `filtered_points`, `filtered_regions`)."""

    def __init__(self, points, bounding_box):
        points = np.asarray(points, dtype=np.float64)
        keep = in_box(points, bounding_box)
        c = points[keep, :]
        left = np.copy(c)
        left[:, 0] = bounding_box[0] - (left[:, 0] - bounding_box[0] + EPS)
        right = np.copy(c)
        right[:, 0] = bounding_box[1] + (bounding_box[1] - right[:, 0] + EPS)
        down = np.copy(c)
        down[:, 1] = bounding_box[2] - (down[:, 1] - bounding_box[2] + EPS)
        up = np.copy(c)
        up[:, 1] = bounding_box[3] + (bounding_box[3] - up[:, 1] + EPS)
        pts = np.concatenate((c, left, right, down, up), axis=0)
        vor = Voronoi(pts)
        self.vertices = vor.vertices
        self.filtered_points = c
        self.filtered_regions = [list(vor.regions[r]) for r in vor.point_region[:vor.npoints // 5]]
        self.bounding_box = np.asarray(bounding_box, dtype=np.float64)
        # the argmin fast path equals the polygon test only when every seed lies inside the domain box proper
        self.seeds_inside = bool(np.all((c[:, 0] >= bounding_box[0]) & (c[:, 0] <= bounding_box[1]) &
                                        (c[:, 1] >= bounding_box[2]) & (c[:, 1] <= bounding_box[3])))
        self._flat = None

    def __len__(self):
        return len(self.filtered_regions)

    def cell_vertices(self, i):
        return self.vertices[self.filtered_regions[i], :]

    def areas(self):
        """Shoelace area per cell (simulator.py:127-136): 0.5 |x . roll(y,1) - y . roll(x,1)|, cached.  All cells at once
        on the flat vertex list (two segmented dot products, then the difference -- the reference's order of operations)."""
        if getattr(self, "_areas", None) is None:
            _, poly, off = self.flat()
            A = len(self)
            if A == 0 or poly.shape[0] == 0:
                self._areas = np.zeros(A)
            else:
                x, y = poly[:, 0], poly[:, 1]
                prev = np.arange(poly.shape[0]) - 1
                prev[off[:-1]] = off[1:] - 1                      # roll(., 1) inside every cell
                a = np.add.reduceat(x * y[prev], off[:-1])
                b = np.add.reduceat(y * x[prev], off[:-1])
                self._areas = 0.5 * np.abs(a - b)
        return self._areas

    def flat(self):
        """(seeds[A,2], poly_xy[nvert,2], poly_off[A+1]) as contiguous host arrays."""
        if self._flat is None:
            regs = self.filtered_regions
            A = len(regs)
            lens = np.fromiter((len(r) for r in regs), dtype=np.int64, count=A)
            off = np.zeros(A + 1, dtype=np.int32)
            np.cumsum(lens, out=off[1:])
            idx = np.fromiter(itertools.chain.from_iterable(regs), dtype=np.intp, count=int(off[-1]))
            poly = np.ascontiguousarray(self.vertices[idx], dtype=np.float64) if A else np.empty((0, 2))
            self._flat = (np.ascontiguousarray(self.filtered_points, dtype=np.float64), poly, off)
        return self._flat


class ClippedVoronoi:
    """Bounded Voronoi partition built ON THE DEVICE by half-plane clipping (cov_voronoi_clip): same cells as
    BoundedVoronoi up to ~1e-13 in the vertices, no host Qhull call and nothing to upload but the seeds.  Host views
    (`vertices`, `filtered_regions`, `areas()`) are fetched lazily, only if somebody asks."""

    def __init__(self, points, bounding_box, device=None, reuse=None):
        """`reuse`: a ClippedVoronoi of an earlier iteration whose device buffers may be overwritten (same cell count)."""
        if reuse is not None:
            self.device = reuse.device
        else:
            nat.require_cuda()
            self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        points = np.asarray(points, dtype=np.float64)
        bb = np.asarray(bounding_box, dtype=np.float64)
        c = np.ascontiguousarray(points[in_box(points, bb), :])
        self.filtered_points = c
        self.bounding_box = bb
        self.A = int(c.shape[0])
        self.seeds_inside = bool(np.all((c[:, 0] >= bb[0]) & (c[:, 0] <= bb[1]) & (c[:, 1] >= bb[2]) & (c[:, 1] <= bb[3])))
        self.nvert = 7 * self.A + 16                       # capacity (planar bound ~6A + corners); actual count = off[A]
        f64 = dict(dtype=torch.float64, device=self.device)
        self._stale = False
        if reuse is not None and reuse.A == self.A:
            reuse._stale = True      # its device buffers now belong to this object
            self.seeds, self.poly, self.off, self.dev_areas, self.flag, self._stage, self._cwork = \
                reuse.seeds, reuse.poly, reuse.off, reuse.dev_areas, reuse.flag, reuse._stage, reuse._cwork
            # page-locked staging + asynchronous copy: the host never waits for what is already queued on the stream
            # (the previous user of the staging buffer is long done: its iteration ended with a synchronising copy home)
            self._stage.numpy()[:] = c.reshape(-1)
            self.seeds.copy_(self._stage, non_blocking=True)
        else:
            self._stage = torch.empty(max(2 * self.A, 1), dtype=torch.float64, pin_memory=True)
            self._stage.numpy()[:2 * self.A] = c.reshape(-1)
            self.seeds = self._stage[:2 * self.A].to(self.device, non_blocking=True)
            self.poly = torch.empty(2 * self.nvert, **f64)
            self.off = torch.empty(self.A + 2, dtype=torch.int32, device=self.device)
            self.dev_areas = torch.empty(max(self.A, 1), **f64)
            self.flag = torch.empty(1, dtype=torch.int32, device=self.device)
            self._cwork = torch.empty(int(nat.lib().cov_voronoi_clip_workspace_bytes(max(self.A, 1))) // 8 + 8, **f64)
        if self.A:
            nat.check(nat.lib().cov_voronoi_clip(nat.ptr(self.seeds), self.A, bb[0], bb[1], bb[2], bb[3], EPS,
                                                 nat.ptr(self.poly), nat.ptr(self.off), self.nvert, nat.ptr(self.dev_areas),
                                                 nat.ptr(self.flag), nat.ptr(self._cwork), self._cwork.numel() * 8,
                                                 nat.stream_ptr()), "cov_voronoi_clip")
        self._host = None
        self._areas_host = None

    def __len__(self):
        return self.A

    def _fetch(self):
        if self._host is None and self._stale:
            raise RuntimeError("this partition's device buffers were recycled by a later iteration (ClippedVoronoi reuse=)")
        if self._host is None:
            if int(self.flag.item()):
                raise RuntimeError("cov_voronoi_clip: polygon capacity exceeded")
            off = self.off[:self.A + 1].cpu().numpy()
            poly = self.poly.cpu().numpy().reshape(-1, 2)[:off[-1]]
            self._host = (poly, off, self.dev_areas[:self.A].cpu().numpy())
        return self._host

    @property
    def vertices(self):
        return self._fetch()[0]

    @property
    def filtered_regions(self):
        off = self._fetch()[1]
        return [list(range(off[i], off[i + 1])) for i in range(self.A)]

    def cell_vertices(self, i):
        poly, off, _ = self._fetch()
        return poly[off[i]:off[i + 1]]

    def areas(self):
        """Host copy of the device shoelace areas (one small copy; the vertices stay on the device)."""
        if self._host is not None:
            return self._host[2]
        if getattr(self, "_areas_host", None) is None and self._stale:
            raise RuntimeError("this partition's device buffers were recycled by a later iteration (ClippedVoronoi reuse=)")
        if getattr(self, "_areas_host", None) is None:
            h = torch.empty(self.A + 1, dtype=torch.float64, pin_memory=True)
            h[:self.A].copy_(self.dev_areas[:self.A], non_blocking=True)
            h[self.A:].copy_(self.flag.to(torch.float64), non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            if h[self.A] != 0:
                raise RuntimeError("cov_voronoi_clip: polygon capacity exceeded")
            self._areas_host = h.numpy()[:self.A]
        return self._areas_host


class HybridVoronoi(ClippedVoronoi):
    """The default partition object of the drop-in (`simulator.voronoi_bounded`): the cells are clipped on the DEVICE at
    construction (nothing to wait for, nothing to upload), and scipy/Qhull -- what the reference calls,
    simulator.py:154-191 -- runs on the host only on demand:
      * when a coverage pass reports grid points within TIE_TOL of a bisector (cov_assign_reduce's tie counter): their
        membership is decided by the reference's crossings test against the polygon VERTICES, and tie parity is defined
        by live Qhull (SURVEY 7.4), so that pass is repeated with Qhull's polygons;
      * when the host reads `vertices` / `filtered_regions` / `cell_vertices` (plotting, the reference's attribute names).
    With no tie point the result of a pass depends on the cells only through nearest-seed membership (identical) and the
    cell areas (device shoelace vs Qhull shoelace: 1e-11 relative, tests/test_gpu_coverage.py)."""

    def __init__(self, points, bounding_box, device=None, reuse=None):
        super().__init__(points, bounding_box, device=device, reuse=reuse)
        self._points = np.array(points, dtype=np.float64, copy=True)
        self._qhull = None

    def qhull(self):
        if self._qhull is None:
            self._qhull = BoundedVoronoi(self._points, self.bounding_box)
        return self._qhull

    @property
    def vertices(self):
        return self.qhull().vertices

    @property
    def filtered_regions(self):
        return self.qhull().filtered_regions

    def cell_vertices(self, i):
        return self.qhull().cell_vertices(i)

    def areas(self):
        if self._qhull is None and self._stale and self._areas_host is None:
            self.qhull()             # the device buffers went to a later iteration: Qhull rebuilds the cells from the seeds
        return self._qhull.areas() if self._qhull is not None else super().areas()


def polygon_partition(seeds, polygons):
    """A partition from explicit polygons (list of [n_i,2] arrays); used for in_polygon / sample clustering."""
    bv = BoundedVoronoi.__new__(BoundedVoronoi)
    verts = np.concatenate(polygons, axis=0) if polygons else np.empty((0, 2))
    regions, o = [], 0
    for p in polygons:
        regions.append(list(range(o, o + len(p))))
        o += len(p)
    bv.vertices = verts
    bv.filtered_points = np.asarray(seeds, dtype=np.float64).reshape(-1, 2)
    bv.filtered_regions = regions
    bv.seeds_inside = False
    bv._flat = None
    return bv


class _DevPartition:
    """Seeds, polygon vertices and polygon offsets of one partition on the device (ONE packed upload)."""

    def __len__(self):
        return self.A

    def __init__(self, vor, device):
        seeds, poly, off = vor.flat()
        self.A = int(seeds.shape[0])
        self.nvert = int(off[-1])
        nb_s, nb_p = self.A * 16, max(self.nvert, 1) * 16
        # staged in page-locked memory (torch's caching host allocator) and copied asynchronously: a pageable upload
        # would make the host wait for everything queued on the stream before it (the posterior kernels)
        stage = torch.zeros(nb_s + nb_p + (self.A + 2) // 2 * 8, dtype=torch.uint8, pin_memory=True)
        host = stage.numpy()
        host[:nb_s] = seeds.reshape(-1).view(np.uint8)
        if self.nvert:
            host[nb_s:nb_s + self.nvert * 16] = poly.reshape(-1).view(np.uint8)
        host[nb_s + nb_p:nb_s + nb_p + (self.A + 1) * 4] = off.view(np.uint8)
        buf = stage.to(device, non_blocking=True)
        self.seeds = buf[:nb_s].view(torch.float64)
        self.poly = buf[nb_s:nb_s + nb_p].view(torch.float64)
        self.off = buf[nb_s + nb_p:].view(torch.int32)


def seeds_summary(points, bounding_box):
    """(number of cells, seeds_inside) of the partition BoundedVoronoi would build from `points` -- without building it
    (the seeds kept are those inside the cushioned box, simulator.py:139-151)."""
    points = np.asarray(points, dtype=np.float64).reshape(-1, 2)
    bb = bounding_box
    c = points[in_box(points, bb), :]
    inside = bool(np.all((c[:, 0] >= bb[0]) & (c[:, 0] <= bb[1]) & (c[:, 1] >= bb[2]) & (c[:, 1] <= bb[3])))
    return int(c.shape[0]), inside


def partition_capacity(A):
    """Vertex capacity of a packed partition buffer (planar bound ~6A + the box corners, with slack)."""
    return 8 * A + 32


def partition_doubles(A):
    """Size of one packed partition: seeds 2A | areas A (+pad) | offsets (A+1 int32, padded) | vertices 2 cap."""
    return 2 * A + (A + 1) // 2 * 2 + (A + 2) // 2 * 2 + 2 * partition_capacity(A)


def pack_partition(vor, out):
    """Write a BoundedVoronoi into `out` (numpy float64 view of partition_doubles(A) entries)."""
    seeds, poly, off = vor.flat()
    A = seeds.shape[0]
    cap = partition_capacity(A)
    if int(off[-1]) > cap:
        raise RuntimeError("pack_partition: polygon capacity exceeded")
    o_ar = 2 * A
    o_off = o_ar + (A + 1) // 2 * 2
    o_poly = o_off + (A + 2) // 2 * 2
    out[:] = 0.0
    out[:2 * A] = seeds.reshape(-1)
    out[o_ar:o_ar + A] = vor.areas()
    out[o_off:o_poly].view(np.int32)[:A + 1] = off
    out[o_poly:o_poly + 2 * int(off[-1])] = poly.reshape(-1)


class PackedPartition:
    """A partition that lives in a packed device buffer (pack_partition layout): what CoverageGrid.assign_reduce needs
    (seeds, polygons, offsets) plus the cell areas, without any host geometry -- e.g. received through a broadcast."""

    def __init__(self, buf, A, seeds_inside):
        cap = partition_capacity(A)
        o_ar = 2 * A
        o_off = o_ar + (A + 1) // 2 * 2
        o_poly = o_off + (A + 2) // 2 * 2
        self.A, self.nvert, self.seeds_inside = int(A), cap, bool(seeds_inside)      # nvert: capacity, the count is off[A]
        self.seeds = buf[:2 * A]
        self.dev_areas = buf[o_ar:o_ar + A]
        self.off = buf[o_off:o_poly].view(torch.int32)
        self.poly = buf[o_poly:o_poly + 2 * cap]

    def __len__(self):
        return self.A

    def areas(self):
        """Host copy of the cell areas (one small device->host copy, cached)."""
        if getattr(self, "_areas", None) is None:
            self._areas = self.dev_areas.cpu().numpy()
        return self._areas


class CoverageGrid:
    """Grid points xy[G,2] (+ optional truth f[G]) resident on the device, with reusable output buffers."""

    def __init__(self, xy_host, f_host=None, device=None, base_index=0, axes=None):
        """`axes`: TensorAxes of the FULL grid when xy_host is a contiguous slice [base_index, base_index+G) of a
        tensor-product grid (grid sharding); detected automatically when xy_host is itself a whole tensor grid."""
        nat.require_cuda()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        xy = np.ascontiguousarray(xy_host, dtype=np.float64).reshape(-1, 2)
        self.G = int(xy.shape[0])
        self.base_index = int(base_index)
        self.xy = torch.from_numpy(xy).to(self.device)
        self.f = None if f_host is None else torch.from_numpy(
            np.ascontiguousarray(f_host, dtype=np.float64).reshape(-1)).to(self.device)
        self._work = None
        self._work_key = None
        self._fin = None
        self.use_sweep = True        # tensor-product grids: column-sweep kernel (cov_assign_reduce_grid)
        if axes is None and base_index == 0:
            from ._engine import TensorAxes, detect_tensor_grid
            t = detect_tensor_grid(xy)
            axes = TensorAxes(t[0], t[1], self.device) if t is not None else None
        self.axes = axes

    def _workspace(self, Ac, Ap):
        need = int(nat.lib().cov_workspace_bytes(self.G, max(Ac, 1), Ap))
        if self._work is None or self._work.numel() * 8 < need:
            self._work = torch.empty(need // 8 + 8, dtype=torch.float64, device=self.device)
        return self._work

    def upload(self, vor):
        """Device copy of a partition (BoundedVoronoi / polygon_partition); pass the result to assign_reduce to reuse it."""
        if isinstance(vor, ClippedVoronoi) and vor._stale and not (isinstance(vor, HybridVoronoi)):
            raise RuntimeError("this partition's device buffers were recycled by a later iteration (ClippedVoronoi reuse=)")
        if isinstance(vor, HybridVoronoi) and (not vor.seeds_inside or vor._qhull is not None or vor._stale):
            # Qhull's vertices: once they exist (an earlier pass met tie points / the host asked for them) they are the
            # cells; and cells with a seed outside the box are not nearest-seed cells (every point takes the crossings test)
            vor = vor.qhull()
        if vor is None or isinstance(vor, (_DevPartition, ClippedVoronoi, PackedPartition)):
            return vor if (vor is None or len(vor)) else None
        if not len(vor):
            return None
        d = _DevPartition(vor, self.device)
        d.seeds_inside = bool(vor.seeds_inside)
        return d

    def assign_reduce(self, lloyd_vor=None, loss_vor=None, w=None, var=None, want_members=False, tie_tol=None,
                      amax_k0=0.0, amax_rel=0.0, out=None):
        """One fused pass.  Returns a dict of DEVICE tensors: cent[Ac,4], amax_val[Ac], amax_idx[Ac], lossp[Ap,2],
        members[G,words] (optional), ties[1] (int32: points whose membership the crossings test decided).  `out`: a
        dict returned by an earlier call with the same cell counts, reused."""
        dev = self.device
        if want_members:         # membership masks are compared bit for bit with the reference's: Qhull's vertices decide ties
            lloyd_vor = lloyd_vor.qhull() if isinstance(lloyd_vor, HybridVoronoi) else lloyd_vor
            loss_vor = loss_vor.qhull() if isinstance(loss_vor, HybridVoronoi) else loss_vor
        C = self.upload(lloyd_vor)
        P = self.upload(loss_vor)
        Ac = C.A if C else 0
        Ap = P.A if P else 0
        if tie_tol is None:
            tie_tol = TIE_TOL
            for v in (C, P):
                if v is not None and not v.seeds_inside:
                    tie_tol = math.inf      # polygons are not plain nearest-seed cells: crossings test everywhere
        f64 = dict(dtype=torch.float64, device=dev)
        reuse = out is not None and not want_members and \
            (out["cent"].shape[0] if out.get("cent") is not None else 0) == Ac and \
            (out["lossp"].shape[0] if out.get("lossp") is not None else 0) == Ap
        if reuse:
            cent, amax_val, amax_idx, lossp = out["cent"], out["amax_val"], out["amax_idx"], out["lossp"]
        else:
            # one packed buffer [cent 4 Ac | amax_val Ac | amax_idx Ac (int64 bits) | lossp 2 Ap | tie count (int32)]:
            # results_to_host() brings everything home with ONE device->host copy
            pack = torch.empty(6 * Ac + 2 * Ap + 1, **f64)
            out = {"pack": pack, "pack_shape": (Ac, Ap), "ties": pack[6 * Ac + 2 * Ap:].view(torch.int32)[:1]}
            cent = pack[:4 * Ac].view(Ac, 4) if Ac else None
            amax_val = pack[4 * Ac:5 * Ac] if Ac else None
            amax_idx = pack[5 * Ac:6 * Ac].view(torch.int64) if Ac else None
            lossp = pack[6 * Ac:6 * Ac + 2 * Ap].view(Ap, 2) if Ap else None
        words = (max(Ac, Ap) + 63) // 64
        words = 1 if words <= 1 else (2 if words == 2 else 4)
        members = torch.zeros((self.G, words), dtype=torch.int64, device=dev) if (want_members and Ac) else None
        work = self._workspace(Ac, Ap)
        ties = out["ties"]
        ny = self.axes.ny if self.axes is not None else 0
        if self.use_sweep and ny and members is None and math.isfinite(tie_tol) and self.G % ny == 0 \
                and self.base_index % ny == 0:
            rc = nat.lib().cov_assign_reduce_grid(          # tensor-product grid (or a whole-column shard): column sweep
                nat.ptr(self.xy), nat.ptr(w), nat.ptr(var), nat.ptr(self.f), self.G, ny, self.base_index,
                nat.ptr(C.seeds) if C else None, Ac, nat.ptr(C.poly) if C else None, nat.ptr(C.off) if C else None,
                C.nvert if C else 0,
                nat.ptr(P.seeds) if P else None, Ap, nat.ptr(P.poly) if P else None, nat.ptr(P.off) if P else None,
                P.nvert if P else 0,
                ctypes.c_double(tie_tol), ctypes.c_double(amax_k0), ctypes.c_double(amax_rel), nat.ptr(cent),
                nat.ptr(amax_val), nat.ptr(amax_idx), nat.ptr(lossp), nat.ptr(ties), nat.ptr(work), work.numel() * 8,
                nat.stream_ptr())
            nat.check(rc, "cov_assign_reduce_grid")
            out.update(cent=cent, amax_val=amax_val, amax_idx=amax_idx, lossp=lossp, members=None)
            return out
        rc = nat.lib().cov_assign_reduce(
            nat.ptr(self.xy), nat.ptr(w), nat.ptr(var), nat.ptr(self.f), self.G, self.base_index,
            nat.ptr(C.seeds) if C else None, Ac, nat.ptr(C.poly) if C else None, nat.ptr(C.off) if C else None,
            C.nvert if C else 0,
            nat.ptr(P.seeds) if P else None, Ap, nat.ptr(P.poly) if P else None, nat.ptr(P.off) if P else None,
            P.nvert if P else 0,
            ctypes.c_double(tie_tol), ctypes.c_double(amax_k0), ctypes.c_double(amax_rel), nat.ptr(cent), nat.ptr(amax_val), nat.ptr(amax_idx), nat.ptr(lossp),
            nat.ptr(members), nat.ptr(ties), nat.ptr(work), work.numel() * 8, nat.stream_ptr())
        nat.check(rc, "cov_assign_reduce")
        out.update(cent=cent, amax_val=amax_val, amax_idx=amax_idx, lossp=lossp, members=members)
        return out

    def reduce_to_host(self, lloyd_vor=None, loss_vor=None, **kw):
        """assign_reduce + results_to_host with the Qhull fallback of HybridVoronoi partitions: if the pass met tie points
        (membership decided by polygon vertices), it is repeated with Qhull's polygons -- exactly the reference's cells."""
        host = self.results_to_host(self.assign_reduce(lloyd_vor, loss_vor, **kw))
        hybrid = [v for v in (lloyd_vor, loss_vor) if isinstance(v, HybridVoronoi) and v._qhull is None]
        if host["ties"] and hybrid:
            q = [v.qhull() if isinstance(v, HybridVoronoi) else v for v in (lloyd_vor, loss_vor)]
            host = self.results_to_host(self.assign_reduce(q[0], q[1], **kw))
        return host

    @staticmethod
    def results_to_host(res):
        """Host copy of an assign_reduce result as a dict of numpy arrays (cent, amax_val, amax_idx, lossp): ONE
        device->host copy of the packed buffer into page-locked memory, one synchronisation."""
        Ac, Ap = res["pack_shape"]
        pack = res["pack"]
        h = torch.empty(pack.shape, dtype=pack.dtype, pin_memory=True)
        h.copy_(pack, non_blocking=True)
        torch.cuda.current_stream(pack.device).synchronize()
        a = h.numpy()
        return {"ties": int(a[6 * Ac + 2 * Ap:].view(np.int32)[0]),
                "cent": a[:4 * Ac].reshape(Ac, 4) if Ac else None,
                "amax_val": a[4 * Ac:5 * Ac] if Ac else None,
                "amax_idx": a[5 * Ac:6 * Ac].view(np.int64) if Ac else None,
                "lossp": a[6 * Ac:6 * Ac + 2 * Ap].reshape(Ap, 2) if Ap else None}

    def finish(self, res, lloyd_vor, loss_vor, bbox, info=None, with_ties=False):
        """Device finishing of an assign_reduce result for DEVICE-resident partitions (ClippedVoronoi / HybridVoronoi):
        returns (loss, centroids[Ac,2], max_var[Ac], argmax_idx[Ac]) -- plus the pass's tie count when `with_ties` -- with
        ONE device->host copy (cov_finish), which also carries the clip-capacity flags and (`info`: device int32, e.g. the
        Cholesky status) the caller's error state."""
        Ac = len(lloyd_vor) if lloyd_vor is not None else 0
        Ap = len(loss_vor) if loss_vor is not None else 0
        n = 5 + 4 * max(Ac, 1)
        if self._fin is None or self._fin[0].numel() != n:
            self._fin = (torch.empty(n, dtype=torch.float64, device=self.device),
                         torch.empty(n, dtype=torch.float64, pin_memory=True))
        out, host = self._fin
        nat.check(nat.lib().cov_finish(nat.ptr(res["cent"]), nat.ptr(lloyd_vor.dev_areas) if Ac else None, Ac,
                                       nat.ptr(res["lossp"]), nat.ptr(loss_vor.dev_areas) if Ap else None, Ap,
                                       nat.ptr(res["amax_val"]), nat.ptr(res["amax_idx"]), bbox[0], bbox[1], bbox[2], bbox[3],
                                       nat.ptr(info), nat.ptr(lloyd_vor.flag) if Ac else None,
                                       nat.ptr(loss_vor.flag) if Ap else None, nat.ptr(res.get("ties")), nat.ptr(out),
                                       nat.stream_ptr()), "cov_finish")
        host.copy_(out, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        h = host.numpy()
        if h[1 + 4 * Ac] < 0:       # info = -1: the tiled Cholesky gave up waiting for a tile (internal error, not a pivot)
            raise RuntimeError("libmfgp_b200: the tiled Cholesky kernel gave up waiting for a tile (internal error)")
        if h[1 + 4 * Ac] != 0:
            raise np.linalg.LinAlgError(f"Matrix is not positive definite (pivot {int(h[1 + 4 * Ac]) - 1})")
        if h[2 + 4 * Ac] != 0 or h[3 + 4 * Ac] != 0:
            raise RuntimeError("cov_voronoi_clip: polygon capacity exceeded")
        r = (float(h[0]), h[1:1 + 2 * Ac].reshape(Ac, 2).copy(), h[1 + 2 * Ac:1 + 3 * Ac].copy(),
             h[1 + 3 * Ac:1 + 4 * Ac].astype(np.int64))
        return r + (int(h[4 + 4 * Ac]),) if with_ties else r

    def cell_moments(self, vor, box, orders, tie_tol=None):
        """Moment tensors mom[A, 3, ry, kpad] of the partition `vor` over this whole tensor-product grid (cov_cell_moments) on
        the Chebyshev basis of `box` = (xlo, xhi, ylo, yhi) with `orders` = (rx, ry), and the device int32 tie count.
        Returns (mom, ties, partition used), the partition as CoverageGrid.upload gives it."""
        if self.axes is None or self.base_index:
            raise ValueError("sample_centroids: the grid is not a whole x-major tensor-product grid [[x, y] for x in ux for y in uy]")
        P = self.upload(vor)
        if P is None:
            raise ValueError("sample_centroids: the partition has no cell")
        if tie_tol is None:
            tie_tol = TIE_TOL if P.seeds_inside else math.inf
        rx, ry = int(orders[0]), int(orders[1])
        lib = nat.lib()
        nx, ny, A = self.axes.nx, self.axes.ny, P.A
        wb = int(lib.cov_cell_moments_workspace_bytes(nx, ny, A, rx, ry))
        f64 = dict(dtype=torch.float64, device=self.device)
        mom = torch.empty((A, 3, ry, -(-rx // 4) * 4), **f64)
        ties = torch.empty(2, dtype=torch.int32, device=self.device)[:1]
        work = torch.empty(wb // 8 + 2, **f64)
        nat.check(lib.cov_cell_moments(nat.ptr(self.xy), nx, ny, nat.ptr(P.seeds), A, nat.ptr(P.poly), nat.ptr(P.off),
                                       ctypes.c_double(tie_tol), *(ctypes.c_double(v) for v in box), rx, ry, nat.ptr(mom),
                                       nat.ptr(ties), nat.ptr(work), wb, nat.stream_ptr()), "cov_cell_moments")
        return mom, ties, P

    def sample_centroids(self, model, vor, normals, bbox=None):
        """Per-cell Lloyd partials and centroids of joint posterior draws over this whole tensor-product grid, without
        evaluating the draws: the draws are DeviceGP.posterior_sample_grid's at the same `normals` (a float64 [d, S] device
        tensor, d = model.grid_sample_dim(grid)), their coefficients are contracted with the partition's moment tensors
        (cov_cell_moments, cov_cell_moments_centroids).  `model`: an MFGP / SFGP; `vor`: the partition (any type
        assign_reduce takes); `bbox`: the clamp box of the centroids, default the grid's extent.
        Returns device tensors cent[S, A, 4] = {sum F_s, sum F_s x, sum F_s y, n} (assign_reduce's `cent` with w = F_s) and
        centroids[S, A, 2] (compute_centroids' arithmetic; NaN for an empty cell).  Like reduce_to_host, a HybridVoronoi
        partition whose pass meets hard ties is passed again on Qhull's polygons.  Raises the sampler's errors: ValueError
        for a grid that is not a whole tensor-product grid or orders above 64, MemoryError before allocating, LinAlgError for
        a non-SPD fit."""
        eng = model._dev
        axes = model._grid_axes(self)
        if not eng.fitted:
            model._refit(check=True)
        eng.check_factor(force=True)
        plan = eng._grid_sample_plan(axes)
        A = len(vor)
        rx, ry = plan["rx"], plan["ry"]
        kpad = -(-rx // 4) * 4
        S = int(normals.shape[1]) if normals.dim() == 2 else 0
        extra = int(nat.lib().cov_cell_moments_workspace_bytes(axes.nx, axes.ny, max(A, 1), rx, ry)) + \
            8 * (3 * A * ry * kpad + 6 * S * A)
        C, plan = eng.posterior_sample_grid_coef(axes, normals, extra_bytes=extra)
        mom, ties, _ = self.cell_moments(vor, plan["box"], (rx, ry))
        if isinstance(vor, HybridVoronoi) and vor._qhull is None and int(ties.item()):
            vor.qhull()          # tie points: their membership is decided by Qhull's vertices, as in the reference
            mom, ties, _ = self.cell_moments(vor, plan["box"], (rx, ry))
        areas = torch.from_numpy(np.ascontiguousarray(vor.areas(), dtype=np.float64)).to(self.device)
        if bbox is None:
            bbox = (axes.xlo, axes.xhi, axes.ylo, axes.yhi)
        f64 = dict(dtype=torch.float64, device=self.device)
        cent = torch.empty((S, A, 4), **f64)
        cen = torch.empty((S, A, 2), **f64)
        nat.check(nat.lib().cov_cell_moments_centroids(nat.ptr(mom), A, rx, ry, nat.ptr(C), S,
                                                       ctypes.c_double(eng.params["mean_H"]), nat.ptr(areas),
                                                       *(ctypes.c_double(v) for v in bbox), nat.ptr(cent), nat.ptr(cen),
                                                       None, 0, nat.stream_ptr()), "cov_cell_moments_centroids")
        return cent, cen

    def argmax(self, v_dev, k0=0.0, rel=0.0):
        """First-index argmax of a device vector (np.argmax semantics): returns (value, index) device tensors."""
        val = torch.empty(1, dtype=torch.float64, device=self.device)
        idx = torch.empty(1, dtype=torch.int64, device=self.device)
        work = self._workspace(1, 0)
        nat.check(nat.lib().cov_argmax(nat.ptr(v_dev), int(v_dev.numel()), self.base_index, ctypes.c_double(k0), ctypes.c_double(rel),
                                       nat.ptr(val),
                                       nat.ptr(idx), nat.ptr(work), work.numel() * 8, nat.stream_ptr()), "cov_argmax")
        return val, idx


# ---- host finishing of the per-cell partial sums (O(A) scalar work, same arithmetic as the reference) ----------------

def loss_from_partials(lossp, areas):
    """simulator.py:215-219: sum_i mean(point_loss_i) * area_i, accumulated in cell order (the per-cell terms are formed
    elementwise, the running sum is sequential: the same IEEE operations in the same order as the reference's loop)."""
    with np.errstate(invalid="ignore", divide="ignore"):
        terms = (lossp[:, 0] / lossp[:, 1]) * np.asarray(areas, dtype=np.float64)[:lossp.shape[0]]
    loss = 0.0
    for t in terms.tolist():
        loss += t
    return np.float64(loss) if lossp.shape[0] else 0


def centroids_from_partials(cent, areas, xmin, xmax, ymin, ymax):
    """simulator.py:256-271: c = (mean(w p) area) / (mean(w) area), clamped to the grid's extent.  Elementwise over the
    cells: per cell exactly the reference's operations (mean, times area, divide, the two one-sided clamps per coordinate)."""
    A = cent.shape[0]
    ar = np.asarray(areas, dtype=np.float64)[:A]
    with np.errstate(invalid="ignore", divide="ignore"):
        n = cent[:, 3]
        f_integral = (cent[:, 0] / n) * ar
        cx = ((cent[:, 1] / n) * ar) / f_integral
        cy = ((cent[:, 2] / n) * ar) / f_integral
        cx = np.where(cx < xmin, xmin, cx)           # a NaN centroid (empty cell) fails both tests and stays NaN
        cx = np.where(cx > xmax, xmax, cx)
        cy = np.where(cy < ymin, ymin, cy)
        cy = np.where(cy > ymax, ymax, cy)
    return np.column_stack((cx, cy))
