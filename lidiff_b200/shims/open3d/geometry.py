import numpy as np

from .utility import Vector3dVector


class KDTreeSearchParamKNN:
    def __init__(self, knn=30):
        self.knn = int(knn)


class KDTreeSearchParamHybrid:
    def __init__(self, radius, max_nn):
        self.radius, self.max_nn = float(radius), int(max_nn)


class Geometry:
    """base class (lidiff/utils/metrics.py tests isinstance(geom, o3d.geometry.Geometry))"""


class GeometryType:
    class _T:
        def __init__(self, v):
            self.value = v
    Unspecified, PointCloud, VoxelGrid = _T(0), _T(1), _T(2)


def _knn(query, ref, k):
    """exact k nearest neighbours of `query` (m,3) among `ref` (n,3), torch tensors on one device -> (dist (m,k), idx (m,k)).
    Bucketed search: queries are sorted into cells of the k-th-neighbour scale; a chunk of consecutive queries searches only the
    reference points inside its bounding box grown by the current margin and is redone with a larger margin if some k-th distance
    exceeds it (so every true neighbour lies inside the searched box).  O(m * local density) instead of O(m * n)."""
    import torch
    m, n = query.shape[0], ref.shape[0]
    k = min(k, n)
    lo, hi = torch.minimum(query.min(0).values, ref.min(0).values), torch.maximum(query.max(0).values, ref.max(0).values)
    vol = float(torch.clamp(hi - lo, min=1e-3).prod())
    cell = max((vol * max(k, 8) / max(n, 1)) ** (1.0 / 3.0), 1e-3)           # a cell holds ~k reference points at the mean density
    ijk = torch.floor((query - lo) / cell).long()
    dims = ijk.max(0).values + 1
    order = torch.argsort((ijk[:, 2] * dims[1] + ijk[:, 1]) * dims[0] + ijk[:, 0])
    qs = query[order]
    dist = torch.empty((m, k), dtype=query.dtype, device=query.device)
    idx = torch.empty((m, k), dtype=torch.long, device=query.device)
    all_ids = torch.arange(n, device=query.device)
    chunk = 4096
    for a in range(0, m, chunk):
        q = qs[a:a + chunk]
        qlo, qhi = q.min(0).values, q.max(0).values
        margin = 2.0 * cell
        while True:
            sel = ((ref >= qlo - margin) & (ref <= qhi + margin)).all(1)
            cand = ref[sel]
            whole = cand.shape[0] == n
            if cand.shape[0] >= k:
                d, j = torch.cdist(q, cand).topk(k, dim=1, largest=False)
                if whole or float(d[:, -1].max()) <= margin:
                    break
            margin *= 2.0
        dist[order[a:a + chunk]] = d
        idx[order[a:a + chunk]] = all_ids[sel][j]
    return dist, idx


class VoxelGrid(Geometry):
    """`VoxelGrid.create_from_point_cloud(pcd, voxel_size)` + `check_if_included(points)` (lidiff/utils/collations.py:44-50,
    eval_path.py:95-100): open3d puts the grid origin at the cloud's minimum bound minus half a voxel and marks the voxels that
    contain at least one point; a query is included when its voxel floor((p - origin) / voxel_size) is marked."""

    def __init__(self):
        self.voxel_size, self.origin, self._keys = 0.0, np.zeros(3), np.zeros((0, 3), np.int64)

    @staticmethod
    def create_from_point_cloud(input, voxel_size):
        g = VoxelGrid()
        pts = np.asarray(input.points, dtype=np.float64)
        g.voxel_size = float(voxel_size)
        g.origin = pts.min(0) - 0.5 * g.voxel_size if len(pts) else np.zeros(3)
        g._keys = np.unique(np.floor((pts - g.origin) / g.voxel_size).astype(np.int64), axis=0) if len(pts) else g._keys
        return g

    def get_geometry_type(self):
        return GeometryType.VoxelGrid

    def get_voxels(self):
        return [tuple(k) for k in self._keys]

    def check_if_included(self, queries):
        q = np.floor((np.asarray(queries, dtype=np.float64) - self.origin) / self.voxel_size).astype(np.int64)
        if len(self._keys) == 0:
            return [False] * len(q)
        span = np.maximum(self._keys.max(0), q.max(0)) - np.minimum(self._keys.min(0), q.min(0)) + 1
        base = np.minimum(self._keys.min(0), q.min(0))
        enc = lambda v: ((v[:, 0] - base[0]) * span[1] + (v[:, 1] - base[1])) * span[2] + (v[:, 2] - base[2])
        return np.isin(enc(q), enc(self._keys)).tolist()


class PointCloud(Geometry):
    def __init__(self, points=None):
        self._points = Vector3dVector(points if points is not None else ())
        self._normals = Vector3dVector(())
        self._colors = Vector3dVector(())

    points = property(lambda s: s._points, lambda s, v: setattr(s, "_points", Vector3dVector(v)))
    normals = property(lambda s: s._normals, lambda s, v: setattr(s, "_normals", Vector3dVector(v)))
    colors = property(lambda s: s._colors, lambda s, v: setattr(s, "_colors", Vector3dVector(v)))

    def has_points(self):
        return len(self._points) > 0

    def has_normals(self):
        return len(self._normals) == len(self._points) > 0

    def __repr__(self):
        return f"PointCloud with {len(self._points)} points."

    def farthest_point_down_sample(self, num_samples):
        """open3d 0.17 semantics: start at index 0, repeatedly add the point farthest from the selected set (first index on
        ties); like open3d's SelectByIndex the result lists the selected points in ORIGINAL index order.  GPU only
        (lb2_farthest_point_sample); no CPU fallback."""
        import torch
        from lidiff_b200.preprocess import farthest_point_sample
        if not torch.cuda.is_available():
            raise RuntimeError("open3d shim: farthest_point_down_sample needs the lidiff_b200 CUDA library and a GPU")
        n = int(num_samples)
        if n <= 0 or n > len(self._points):
            raise RuntimeError("Illegal number of samples")
        sel = farthest_point_sample(torch.as_tensor(np.asarray(self._points), device="cuda"), n)
        out = PointCloud(np.asarray(self._points)[sel.cpu().numpy()])
        if self.has_normals():
            out.normals = np.asarray(self._normals)[sel.cpu().numpy()]
        return out

    def compute_point_cloud_distance(self, target):
        """for every point of this cloud the Euclidean distance to its nearest point of `target` (open3d: KDTreeFlann 1-NN in
        double precision) — what lidiff/utils/metrics.py builds RMSE / Chamfer distance / precision-recall on.  On a GPU this is
        lidiff_b200.metrics.nn_distance (exact fp64 bounding-box hierarchy search)."""
        import torch
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        q64 = torch.as_tensor(np.asarray(self._points), dtype=torch.float64, device=dev)
        r64 = torch.as_tensor(np.asarray(target._points), dtype=torch.float64, device=dev)
        if q64.shape[0] == 0 or r64.shape[0] == 0:
            return np.zeros(q64.shape[0])
        if dev == "cuda":
            from lidiff_b200.metrics import nn_distance
            return nn_distance(q64, r64).cpu().numpy()
        _, idx = _knn(q64.float(), r64.float(), 1)
        # the neighbour found in fp32 can differ from the fp64 one only between candidates equidistant to 1e-7: re-evaluate in fp64
        return (q64 - r64[idx[:, 0]]).norm(dim=1).cpu().numpy()

    def get_geometry_type(self):
        return GeometryType.PointCloud

    def get_min_bound(self):
        return np.asarray(self._points).min(0)

    def get_max_bound(self):
        return np.asarray(self._points).max(0)

    def estimate_normals(self, search_param=None, fast_normal_computation=True):
        """PCA normal of the k nearest neighbours (k = 30 as open3d's default KNN search), sign left unoriented.  Post-processing
        only, not on the timed path; exact bucketed k-NN search (`_knn`)."""
        import torch
        k = getattr(search_param, "knn", None) or getattr(search_param, "max_nn", None) or 30
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        p = torch.as_tensor(np.asarray(self._points), dtype=torch.float32, device=dev)
        n = p.shape[0]
        k = min(k, n)
        out = torch.zeros((n, 3), dtype=torch.float32, device=dev)
        if n >= 3:
            _, idx = _knn(p, p, k)
            for a in range(0, n, 65536):
                nb = p[idx[a:a + 65536]]                                              # (c, k, 3)
                c = nb - nb.mean(1, keepdim=True)
                cov = c.transpose(1, 2) @ c
                out[a:a + 65536] = torch.linalg.eigh(cov.double())[1][:, :, 0].float()   # eigenvector of the smallest eigenvalue
        self._normals = Vector3dVector(out.cpu().numpy())
        return True
