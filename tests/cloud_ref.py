"""Plain FP64 brute-force references for the cloud search operators, and the adversarial clouds they are tested on.

Every distance is computed exactly as the kernels and the oracle define it: d2 = (dx*dx + dy*dy) + dz*dz with dx = q - p,
each operation a separately rounded FP64 ufunc (no FMA).  Sums of square roots are sequential, left to right
(np.add.accumulate), so the references are expected to match the kernels bit for bit, not within a tolerance.
"""
import numpy as np

CHUNK_ELEMS = 1 << 23          # distances per chunk (64 MB of FP64): memory stays bounded at n ~ 30k


def _as_pts(a):
    return np.ascontiguousarray(np.asarray(a, np.float64).reshape(-1, 3))


def brute_d2(q, p):
    """Yields (start, d2) with d2[i, j] = squared distance of query start+i to target j, for chunks of queries."""
    q, p = _as_pts(q), _as_pts(p)
    step = max(1, CHUNK_ELEMS // max(1, len(p)))
    px, py, pz = p[:, 0], p[:, 1], p[:, 2]
    for s in range(0, len(q), step):
        qc = q[s:s + step]
        d2 = np.subtract(qc[:, 0, None], px[None, :])
        np.multiply(d2, d2, out=d2)
        t = np.subtract(qc[:, 1, None], py[None, :])
        np.multiply(t, t, out=t)
        np.add(d2, t, out=d2)
        np.subtract(qc[:, 2, None], pz[None, :], out=t)
        np.multiply(t, t, out=t)
        np.add(d2, t, out=d2)
        yield s, d2


def knn_sorted_d2(p, kmax, q=None):
    """[len(q), min(kmax, n)]: the kmax smallest squared distances of each query (default: the cloud itself, the query
    point included) to the cloud, ascending."""
    p = _as_pts(p)
    q = p if q is None else _as_pts(q)
    k = min(int(kmax), len(p))
    out = np.empty((len(q), k))
    for s, d2 in brute_d2(q, p):
        part = d2 if k == len(p) else np.partition(d2, k - 1, axis=1)[:, :k]
        out[s:s + len(d2)] = np.sort(part, axis=1)
    return out


def mean_dist_from_sorted(sorted_d2, k):
    """d-bar of each row: the sequential sum of the square roots of its k smallest squared distances, over k."""
    k = min(int(k), sorted_d2.shape[1])
    return np.add.accumulate(np.sqrt(sorted_d2[:, :k]), axis=1)[:, -1] / k


def knn_mean_dist(p, k):
    """Per-point mean distance to its k = min(k, n) nearest neighbours (itself included): statistical outlier removal's d-bar."""
    return mean_dist_from_sorted(knn_sorted_d2(p, k), k)


def sor_threshold(dbar, std_ratio):
    """Open3D's rule: the mean is the sum of the d-bar > 0 terms over n, sigma is Bessel's over the same terms."""
    dbar = np.asarray(dbar, np.float64)
    n = len(dbar)
    pos = dbar > 0.0
    total = np.add.accumulate(np.where(pos, dbar, 0.0))[-1]
    mean = float(total) / n
    dev = dbar - mean
    sq = float(np.add.accumulate(np.where(pos, dev * dev, 0.0))[-1])
    sd = float(np.sqrt(sq / (n - 1))) if n > 1 else 0.0
    return mean + std_ratio * sd


def sor_select(dbar, std_ratio):
    """Indices kept by statistical outlier removal: 0 < d-bar < mean + std_ratio * sigma, ascending."""
    dbar = np.asarray(dbar, np.float64)
    if len(dbar) == 0:
        return np.zeros(0, np.int64)
    thr = sor_threshold(dbar, std_ratio)
    return np.nonzero((dbar > 0.0) & (dbar < thr))[0].astype(np.int64)


def nn_distance(q, p):
    """Distance of each query to its nearest target: sqrt(min d2)."""
    q = _as_pts(q)
    out = np.empty(len(q))
    for s, d2 in brute_d2(q, p):
        out[s:s + len(d2)] = np.sqrt(d2.min(axis=1))
    return out


def nn_distance_large(q, p):
    """nn_distance for clouds too large to brute-force: a k-d tree proposes every target within (1 + 1e-9) times its own
    nearest distance (its rounding is far below that margin), and the exact d2 picks the nearest among them."""
    from scipy.spatial import cKDTree
    q, p = _as_pts(q), _as_pts(p)
    tree = cKDTree(p)
    cands = tree.query_ball_point(q, tree.query(q)[0] * (1.0 + 1e-9))
    lens = np.array([len(c) for c in cands])
    j = np.concatenate([np.asarray(c, np.int64) for c in cands])
    i = np.repeat(np.arange(len(q)), lens)
    dx, dy, dz = q[i, 0] - p[j, 0], q[i, 1] - p[j, 1], q[i, 2] - p[j, 2]
    d2 = (dx * dx + dy * dy) + dz * dz
    return np.sqrt(np.minimum.reduceat(d2, np.concatenate([[0], np.cumsum(lens)[:-1]])))


def nn_within(q, p, r):
    """(index, d2) of each query's nearest target with d2 < r*r strictly, ties to the lowest index; (-1, -1.0) if none."""
    q = _as_pts(q)
    idx = np.full(len(q), -1, np.int32)
    dd = np.full(len(q), -1.0)
    if len(_as_pts(p)) == 0:
        return idx, dd
    r2 = float(r) * float(r)
    for s, d2 in brute_d2(q, p):
        j = np.argmin(d2, axis=1)                         # first minimum: the lowest index among ties
        m = d2[np.arange(len(d2)), j]
        hit = m < r2
        idx[s:s + len(d2)][hit] = j[hit]
        dd[s:s + len(d2)][hit] = m[hit]
    return idx, dd


def voxel_down_sample(p, c, voxel):
    """PointCloud.voxel_down_sample: voxel key floor((p - (min - voxel/2)) / voxel) per axis; each voxel's points and colours
    summed sequentially in point-index order, over the count; voxels in lexicographic key order.
    Returns (points, colours or None, int32 keys, int32 counts)."""
    p = _as_pts(p)
    if len(p) == 0:
        return np.zeros((0, 3)), None, np.zeros((0, 3), np.int32), np.zeros(0, np.int32)
    vmin = p.min(axis=0) - voxel * 0.5
    keys = np.floor((p - vmin) / voxel).astype(np.int64)
    uk, inv, cnt = np.unique(keys, axis=0, return_inverse=True, return_counts=True)   # lexicographic rows
    inv = inv.reshape(-1)

    def means(a):
        s = np.zeros((len(uk), 3))
        np.add.at(s, inv, a)                              # unbuffered, applied in index order: sequential sums
        return s / cnt[:, None].astype(np.float64)

    return means(p), (None if c is None else means(_as_pts(c))), uk.astype(np.int32), cnt.astype(np.int32)


# ---------------------------------------------------------------------------------------------------------------------
# adversarial clouds (deterministic)
# ---------------------------------------------------------------------------------------------------------------------
OFFSET = np.array([1e5, -3e4, 250.0])
H = 2.0 ** -6                  # lattice spacing; a power of two keeps every lattice coordinate and cell boundary exact


def surface(n, seed=0):
    """n points on a curved 1.5 m x 1 m sheet."""
    rng = np.random.default_rng(seed)
    x, y = rng.random(n) * 1.5, rng.random(n)
    z = 0.1 * np.sin(3.0 * x) * np.cos(2.0 * y) + 0.3 * x * y
    return np.stack([x, y, z], 1)


def surface_with_outliers(n=20000, seed=0):
    """A sheet and six isolated points 10-50 m away (mostly along x, so that the bounding box stays thin and the coarse
    grid is long enough for a top level)."""
    far = np.array([[12.0, 0.5, 0.1], [25.0, 0.2, 0.0], [50.0, 0.8, 0.1], [-10.0, 0.3, 0.05], [0.7, 15.0, 0.0],
                    [31.0, 14.0, 0.2]])
    p = surface(n, seed)
    ins = np.linspace(0, n, len(far) + 2)[1:-1].astype(int)
    return np.insert(p, ins, far, axis=0)


def lattice(m=17, n=8192, seed=1):
    """An m^3 lattice of spacing H from the origin plus repeats of random lattice points up to n points.  With m = 17
    and n = 8192 the search grid's cell is cbrt((16 H)^3 / (n / 2)) = H exactly, so every point lies on cell faces and
    distances tie everywhere."""
    g = np.arange(m) * H
    p = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    rng = np.random.default_rng(seed)
    extra = p[rng.integers(0, len(p), n - len(p))]
    return np.concatenate([p, extra])[rng.permutation(n)]


def with_duplicates(n=3000, copies=140, seed=2):
    """A sheet in which one of its points appears `copies` more times at scattered indices (d-bar = 0 for them)."""
    p = surface(n, seed)
    rng = np.random.default_rng(seed)
    ins = np.sort(rng.integers(0, n, copies))
    return np.insert(p, ins, np.repeat(p[n // 3][None], copies, 0), axis=0)


def collinear(n=3000, seed=3):
    rng = np.random.default_rng(seed)
    t = rng.random(n) * 2.0 - 0.5
    return np.array([0.3, -1.2, 2.0]) + t[:, None] * np.array([0.6, 0.3, -0.2])


def line_on_faces(m=1025):
    """Points j * H on the x axis: extent 1024 H, so the grid's cell is enlarged to exactly H; every point is on a face."""
    p = np.zeros((m, 3))
    p[:, 0] = np.arange(m) * H
    return p


def coplanar(seed=4):
    """z exactly 0: a 65 x 65 grid spaced 16 H (extent 1024 H, so the cell is exactly H) plus 1000 random points."""
    g = np.arange(65) * 16 * H
    p = np.stack(np.meshgrid(g, g, [0.0], indexing="ij"), -1).reshape(-1, 3)
    rng = np.random.default_rng(seed)
    r = np.zeros((1000, 3))
    r[:, :2] = rng.random((1000, 2)) * 1024 * H
    return np.concatenate([p, r])


def identical(n):
    return np.tile(np.array([[0.25, -1.5, 3.0]]), (n, 1))


def two_clusters(n=2000, seed=5):
    """Two tight clusters 100 m apart along x and one point halfway between them: the coarse grid is long enough for a
    top level, and the middle is empty."""
    rng = np.random.default_rng(seed)
    d = np.array([100.0, 0.0, 0.0])
    a = rng.normal(scale=0.01, size=(n, 3))
    b = rng.normal(scale=0.01, size=(n, 3)) + d
    return np.concatenate([a, d[None] * 0.5, b])


def mirrored(p):
    return -(p + OFFSET)
