"""
Subdivision / filtering criteria for the native path.

The reference's `subdivide` / `filter` take lists of opaque Python callables
`criterion(points: (n,3) ndarray) -> bool` (grid/grid_base.py:126-147): a node splits if ANY
subdivision criterion is true (octree/octree.py:26); a leaf keeps its points only if ALL filtering
criteria are true (octree/octree.py:111).  A GPU cannot call Python per node, so the host folds the
list into a function of the point COUNT, which is what every criterion in the reference's tests
and docs is (`lambda points: len(points) > 100`):

  * `MaxPoints(n)` / `MinPoints(n)` are declarative callables (usable with the reference too);
  * any other callable is probed with (n,3) arrays of several sizes - constant-filled ones and two random clouds of
    different spread; if its answers depend on the size only, the resulting truth table is used.
    Criteria that look at coordinates are never folded (NotCountOnly): `subdivide` / `filter` then evaluate them on the
    host node by node, like the reference, and impose the resulting scheme / keep-masks on the device (_host.py).

Size thresholds.  The reference hands a criterion nothing but the points, so "stop splitting below a node size" cannot
be written as a pure function of its argument; the declarative criteria therefore carry optional NODE-SIZE guards:
`MaxPoints(n, max_depth=d, min_edge=e)` is true iff the node holds more than n points AND is less than d levels below
its grid cell AND its edge is longer than e; `MaxDepth(d)` / `MinEdge(e)` are the guards alone (uniform refinement).
Several criteria still combine with any() (octree/octree.py:26).  The native path folds the guards into a per-LEVEL
decision (`level_limit`), evaluated by `decide_kernel`.  Called as a plain callable - by the reference or by the CPU
oracle - a guarded criterion reads the edge of the node under test from the caller's frame (`self` of
`OctreeNode.subdivide`, octree/octree.py:20-32), which makes the very same object usable with the unmodified
reference: that is how tests/golden/make_golden.py pins the semantics.

Geometric criteria.  `MaxExtent(e)` ("split while the node spans more than e"), `MaxThickness(t)` ("split while the node
is not planar") and `Planar(t)` ("keep planar leaves") look at the coordinates, through two float64 statistics of the
points they are handed: the EXTENT (largest per-axis max - min) and the THICKNESS (RMS distance of the points from their
least-squares plane, sqrt of the smallest eigenvalue of the population covariance).  They are declarative: `subdivide` /
`filter` evaluate them on the GPU (the per-node statistics are one segmented reduction over the points the level loop
holds per leaf, csrc/geometry.cuh) without probing, while the same objects remain plain callables for the reference and
the CPU oracle.  They take the same node-size guards as `MaxPoints` (evaluated by the guard logic of `CountCriterion`).
Extent decisions agree with numpy bit for bit; thickness decisions agree unless a node's thickness lies within the bound
documented in csrc/geometry.cuh of the threshold.  A list that also holds an opaque coordinate-dependent callable is
evaluated on the host as before.
"""
from __future__ import annotations

import sys
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

__all__ = ["MaxPoints", "MinPoints", "MaxDepth", "MinEdge", "CountCriterion", "fold_count_criteria", "as_threshold",
           "fold_levels", "NO_LEVEL_LIMIT", "NotCountOnly", "GeometricCriterion", "MaxExtent", "MaxThickness", "Planar",
           "extent", "thickness"]


class NotCountOnly(NotImplementedError):
    """A criterion could not be folded into a function of the point count (it looks at coordinates, or it failed on the
    probe arrays).  `Grid.subdivide` / `filter` then evaluate it on the host, node by node, like the reference does, and
    hand the resulting scheme / keep-masks to the device (ForestHost._subdivide_on_host); callers that need a
    device-evaluable rule (node-size guards) let it propagate as the NotImplementedError it is."""

NO_LEVEL_LIMIT = 1 << 20  # "may split at every level"

_LARGE_PROBES = [1 << k for k in range(11, 31, 2)] + [(1 << 31) - 1]


def _edge_of_node_under_test() -> float:
    """Edge length of the octree node whose points the caller is testing: the reference evaluates
    `criterion(self._points)` inside `OctreeNode.subdivide` (octree/octree.py:26), the CPU oracle evaluates
    `c(node.pts)` inside `_Tree.subdivide`; both keep the node in a local of a nearby frame."""
    f = sys._getframe(2)
    for _ in range(8):
        if f is None:
            break
        for name in ("self", "node"):
            obj = f.f_locals.get(name)
            if obj is None:
                continue
            for attr in ("edge_length", "edge"):
                try:
                    e = getattr(obj, attr, None)
                except Exception:  # noqa: BLE001
                    e = None
                if isinstance(e, (int, float, np.integer, np.floating)):
                    return float(e)
        f = f.f_back
    raise NotImplementedError(
        "a criterion with a node-size guard (max_depth / min_edge) was called outside OctreeNode.subdivide: the node "
        "under test could not be found")


def halvings(root_edge: float, edge: float) -> int:
    """Depth of a node of edge `edge` below a cell of edge `root_edge` (edges are exact halvings, octree.py:181)."""
    e, k = np.float64(root_edge), 0
    while e > edge and k < 1100:
        e = e / np.float64(2)
        k += 1
    return k


class CountCriterion:
    """`len(points) <op> n` as a callable object with inspectable parameters, optionally guarded by the node size:
    `max_depth` (true only for nodes fewer than `max_depth` levels below their grid cell; needs `voxel_edge_length`
    when used outside this package) and `min_edge` (true only for nodes whose edge is longer than `min_edge`)."""

    _OPS = {
        ">": lambda a, b: a > b,
        ">=": lambda a, b: a >= b,
        "<": lambda a, b: a < b,
        "<=": lambda a, b: a <= b,
        "==": lambda a, b: a == b,
        "!=": lambda a, b: a != b,
    }

    def __init__(self, op: str, n: int, max_depth: Optional[int] = None, min_edge: Optional[float] = None,
                 voxel_edge_length: Optional[float] = None):
        if op not in self._OPS:
            raise ValueError(f"unknown comparison {op!r}")
        if max_depth is not None and int(max_depth) < 0:
            raise ValueError("max_depth must be >= 0")
        if min_edge is not None and not float(min_edge) > 0:
            raise ValueError("min_edge must be positive")
        self.op, self.n = op, int(n)
        self.max_depth = None if max_depth is None else int(max_depth)
        self.min_edge = None if min_edge is None else float(min_edge)
        self.voxel_edge_length = voxel_edge_length

    @property
    def size_guarded(self) -> bool:
        return self.max_depth is not None or self.min_edge is not None

    def level_limit(self, root_edge: float) -> int:
        """Nodes at level >= this (cell root = level 0) never satisfy the criterion."""
        lim = NO_LEVEL_LIMIT
        if self.max_depth is not None:
            lim = min(lim, self.max_depth)
        if self.min_edge is not None:
            lim = min(lim, halvings(root_edge, self.min_edge))
        return lim

    def on_count(self, count: int) -> bool:
        return bool(self._OPS[self.op](count, self.n))

    def on_node(self, count: int, edge: float, root_edge: Optional[float] = None) -> bool:
        if not self.on_count(count):
            return False
        if self.min_edge is not None and not edge > self.min_edge:
            return False
        if self.max_depth is not None:
            root = self.voxel_edge_length if root_edge is None else root_edge
            if root is None:
                raise ValueError("a max_depth guard needs voxel_edge_length=<grid cell edge> when the criterion is used "
                                 "outside octreelib_b200")
            if not halvings(root, edge) < self.max_depth:
                return False
        return True

    def __call__(self, points) -> bool:
        if not self.size_guarded:
            return self.on_count(len(points))
        if not self.on_count(len(points)):
            return False
        return self.on_node(len(points), _edge_of_node_under_test())

    def __repr__(self):
        guard = "".join(f", {k}={v}" for k, v in (("max_depth", self.max_depth), ("min_edge", self.min_edge)) if v is not None)
        return f"CountCriterion(len(points) {self.op} {self.n}{guard})"


class MaxPoints(CountCriterion):
    """Subdivide while a node holds more than `n` points: `lambda points: len(points) > n`; with `max_depth` /
    `min_edge` only down to that depth / node size (point-count AND size threshold)."""

    def __init__(self, n: int, max_depth: Optional[int] = None, min_edge: Optional[float] = None,
                 voxel_edge_length: Optional[float] = None):
        super().__init__(">", n, max_depth, min_edge, voxel_edge_length)


class MinPoints(CountCriterion):
    """Keep a leaf only if it holds at least `n` points: `lambda points: len(points) >= n`."""

    def __init__(self, n: int):
        super().__init__(">=", n)


class MaxDepth(CountCriterion):
    """True for every node fewer than `depth` levels below its grid cell, whatever it holds (as a subdivision
    criterion: uniform refinement to that depth, empty nodes included - like any criterion that is true on an empty
    cloud in the reference)."""

    def __init__(self, depth: int, voxel_edge_length: Optional[float] = None):
        super().__init__(">=", 0, max_depth=depth, voxel_edge_length=voxel_edge_length)


class MinEdge(CountCriterion):
    """True for every node whose edge is longer than `edge` (uniform refinement down to that node size)."""

    def __init__(self, edge: float):
        super().__init__(">=", 0, min_edge=edge)


def extent(points) -> float:
    """Largest per-axis extent (max - min) of an (n, 3) cloud, in float64; 0.0 for an empty cloud."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    if len(p) == 0:
        return 0.0
    return float((p.max(axis=0) - p.min(axis=0)).max())


def thickness(points) -> float:
    """RMS distance of the points from their least-squares plane: sqrt(max(smallest eigenvalue of the population
    covariance, 0)), two-pass in float64; 0.0 for fewer than 3 points."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    n = len(p)
    if n < 3:
        return 0.0
    d = p - p.mean(axis=0)
    cov = (d.T @ d) / n
    return float(np.sqrt(max(float(np.linalg.eigvalsh(cov)[0]), 0.0)))


class GeometricCriterion:
    """`<stat>(points) <op> value` for clouds of at least `min_points` points, stat = 'extent' or 'thickness', op = '>'
    or '<=', as a callable object with inspectable parameters.  The optional node-size guards `max_depth` / `min_edge`
    mean what they mean for `MaxPoints`: they are evaluated by a `CountCriterion` guard (level_limit / on_node)."""

    STATS = {"extent": (0, extent), "thickness": (1, thickness)}  # name -> (native code, host definition)
    OPS = {">": 0, "<=": 1}

    def __init__(self, stat: str, op: str, value: float, min_points: int = 1, max_depth: Optional[int] = None,
                 min_edge: Optional[float] = None, voxel_edge_length: Optional[float] = None):
        if stat not in self.STATS:
            raise ValueError(f"unknown statistic {stat!r}")
        if op not in self.OPS:
            raise ValueError(f"unknown comparison {op!r}")
        value = float(value)
        if not (np.isfinite(value) and value >= 0):
            raise ValueError(f"{stat} threshold must be finite and >= 0, got {value}")
        if int(min_points) < 1:
            raise ValueError("min_points must be >= 1")
        self.stat, self.op, self.value, self.min_points = stat, op, value, int(min_points)
        self._guard = CountCriterion(">=", self.min_points, max_depth, min_edge, voxel_edge_length)

    @property
    def max_depth(self) -> Optional[int]:
        return self._guard.max_depth

    @property
    def min_edge(self) -> Optional[float]:
        return self._guard.min_edge

    @property
    def size_guarded(self) -> bool:
        return self._guard.size_guarded

    def level_limit(self, root_edge: float) -> int:
        """Nodes at level >= this (cell root = level 0) never satisfy the criterion."""
        return self._guard.level_limit(root_edge)

    def term(self) -> tuple:
        """(statistic code, comparison code, min_points, value): one ol_geom_term of the native rule."""
        return (self.STATS[self.stat][0], self.OPS[self.op], self.min_points, self.value)

    def on_points(self, points) -> bool:
        """The criterion without its node-size guards."""
        p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
        if len(p) < self.min_points:
            return False
        v = self.STATS[self.stat][1](p)
        return v > self.value if self.op == ">" else v <= self.value

    def __call__(self, points) -> bool:
        if not self.on_points(points):
            return False
        if not self.size_guarded:
            return True
        return self._guard.on_node(len(points), _edge_of_node_under_test())

    def __repr__(self):
        guard = "".join(f", {k}={v}" for k, v in (("max_depth", self.max_depth), ("min_edge", self.min_edge)) if v is not None)
        return f"GeometricCriterion({self.stat}(points) {self.op} {self.value}, min_points={self.min_points}{guard})"


class MaxExtent(GeometricCriterion):
    """Subdivide while a node's points span more than `e` along some axis (max - min); with `max_depth` / `min_edge`
    only down to that depth / node size."""

    def __init__(self, e: float, max_depth: Optional[int] = None, min_edge: Optional[float] = None,
                 voxel_edge_length: Optional[float] = None):
        super().__init__("extent", ">", e, 1, max_depth, min_edge, voxel_edge_length)


class MaxThickness(GeometricCriterion):
    """Subdivide while a node of at least `min_points` points is not planar: its points lie farther than `t` (RMS) from
    their least-squares plane; with `max_depth` / `min_edge` only down to that depth / node size."""

    def __init__(self, t: float, min_points: int = 4, max_depth: Optional[int] = None, min_edge: Optional[float] = None,
                 voxel_edge_length: Optional[float] = None):
        super().__init__("thickness", ">", t, min_points, max_depth, min_edge, voxel_edge_length)


class Planar(GeometricCriterion):
    """Keep a leaf only if it holds at least `min_points` points lying within `t` (RMS) of their least-squares plane."""

    def __init__(self, t: float, min_points: int = 3):
        super().__init__("thickness", "<=", t, min_points)


def _probe(n: int, fill: float) -> np.ndarray:
    """An (n, 3) float64 array that costs 8 bytes: zero strides over one value (read-only)."""
    a = np.lib.stride_tricks.as_strided(np.array([fill], dtype=np.float64), shape=(n, 3), strides=(0, 0), writeable=False)
    return a


# Non-degenerate probe clouds (views of two fixed random arrays with different spreads and offsets): a criterion that
# looks at extents, variances, planarity ... is translation invariant and answers the same on every CONSTANT-filled
# array, so constant probes alone would fold it into a count table silently.
_SPREAD_CAP = 1 << 16
_spread_cache: dict = {}


def _spread_probe(n: int, which: int) -> np.ndarray:
    if which not in _spread_cache:
        rng = np.random.default_rng(0x0C7EE + which)
        scale, offset = ((0.05, 0.0), (700.0, -1234.5))[which]
        a = rng.standard_normal((_SPREAD_CAP, 3)) * scale + offset
        a.setflags(write=False)
        _spread_cache[which] = a
    return _spread_cache[which][:n]


def _memo_key(criterion: Callable):
    """Key under which the folded form of a plain Python function may be reused, or None.  A function whose code refers
    to nothing but its argument, builtins, constants, hashable defaults and hashable closure values (the documented
    `lambda points: len(points) > N`, also when N is captured from the enclosing scope) answers the same on the same
    probe every time, however often the lambda expression is re-evaluated - so `Grid.subdivide` does not have to probe
    it again on every call (4 100 calls of the criterion, 15-40 ms of host time)."""
    code = getattr(criterion, "__code__", None)
    glob = getattr(criterion, "__globals__", None)
    if code is None or glob is None or getattr(criterion, "__self__", None) is not None:
        return None
    import builtins

    for name in code.co_names:
        if name in glob or not hasattr(builtins, name):
            return None  # module-level state (or attribute access on something we cannot see): not memoised
    cells = []
    for cell in criterion.__closure__ or ():
        try:
            v = cell.cell_contents
        except ValueError:
            return None
        if not isinstance(v, (int, float, bool, str, bytes, type(None))):
            return None
        cells.append((type(v), v))
    defaults = criterion.__defaults__ or ()
    kwdefaults = tuple(sorted((criterion.__kwdefaults__ or {}).items()))
    if not all(isinstance(v, (int, float, bool, str, bytes, type(None))) for v in defaults + tuple(v for _, v in kwdefaults)):
        return None
    return (code, tuple(cells), tuple((type(v), v) for v in defaults), kwdefaults)


_fold_memo: dict = {}
_FOLD_MEMO_MAX = 256


def _eval(criterion: Callable, n: int) -> bool:
    if isinstance(criterion, CountCriterion):
        return criterion.on_count(n)
    try:
        answers = [bool(criterion(_probe(n, 0.0))), bool(criterion(_probe(n, 123456.789)))]
        if n <= _SPREAD_CAP:
            answers += [bool(criterion(_spread_probe(n, 0))), bool(criterion(_spread_probe(n, 1)))]
    except Exception as exc:  # noqa: BLE001
        raise NotCountOnly(
            "octreelib_b200 evaluates subdivision / filtering criteria on the GPU as functions of the point count; "
            f"criterion {criterion!r} failed on a probe array of {n} points ({exc!r}). Use criteria such as "
            "`lambda points: len(points) > N` or octreelib_b200.criteria.MaxPoints / MinPoints.") from exc
    if len(set(answers)) != 1:
        raise NotCountOnly(
            f"criterion {criterion!r} depends on the point coordinates, not only on the point count; "
            "coordinate-dependent criteria cannot be evaluated on the GPU")
    return answers[0]


def fold_count_criteria(criteria: Sequence[Callable], mode: str, upto: int) -> Tuple[np.ndarray, bool]:
    """Truth table t[n], n = 0..upto, of `any(c(points))` (mode 'any') or `all(c(points))` (mode 'all')
    for clouds of n points, plus the value for 'very large' clouds (None if the criteria do not settle
    on one).  Raises NotImplementedError for coordinate-dependent criteria."""
    criteria = list(criteria)
    comb = any if mode == "any" else all
    large = [n for n in _LARGE_PROBES if n > upto]
    # per criterion: truth table over 0..upto and the answers on the large probes (vectorised for the declarative
    # criteria, memoised for self-contained Python functions, probed otherwise)
    tables, larges = [], []
    for c in criteria:
        if isinstance(c, CountCriterion):
            op = CountCriterion._OPS[c.op]
            tables.append(np.asarray(op(np.arange(upto + 1, dtype=np.int64), c.n), dtype=bool))
            larges.append([bool(op(n, c.n)) for n in large])
            continue
        key = _memo_key(c)
        hit = _fold_memo.get((key, upto)) if key is not None else None
        if hit is None:
            t = np.fromiter((_eval(c, n) for n in range(upto + 1)), dtype=bool, count=upto + 1)
            hit = (t, [_eval(c, n) for n in large])
            if key is not None:
                if len(_fold_memo) >= _FOLD_MEMO_MAX:
                    _fold_memo.clear()
                _fold_memo[(key, upto)] = hit
        tables.append(hit[0])
        larges.append(hit[1])
    if not criteria:
        table = np.full(upto + 1, 0 if mode == "any" else 1, dtype=np.uint8)
        return table, mode != "any"
    stack = np.stack(tables)
    table = (stack.any(axis=0) if mode == "any" else stack.all(axis=0)).astype(np.uint8)
    beyond_vals = {bool(comb([lv[i] for lv in larges])) for i in range(len(large))}
    if len(beyond_vals) > 1:
        return table, None  # no single answer for "more points than the table covers"
    beyond = beyond_vals.pop() if beyond_vals else bool(table[-1])
    return table, beyond


def as_threshold(table: np.ndarray, beyond: bool, criteria: Sequence[Callable] = None, mode: str = "any"):
    """If the folded criteria are the step `count > n`, return n; if they are never true return a huge n; else None.

    `table` covers the counts 0..len(table)-1 and `beyond` is the settled answer for very large clouds.  A step that
    lies ABOVE the table (all-False table, `beyond` True, e.g. `len(points) > 1500` with a 1025-entry table) is located
    by bisection over the criteria themselves; without `criteria` such a table is not a recognisable step (None), so
    the caller falls back to an explicit count table."""
    t = table.astype(bool)
    if beyond is None and (criteria is None or t.any()):
        return None  # the large-count probes disagree and the step (if it is one) cannot be located
    if not t.any() and beyond is False:
        return (1 << 62)
    if t.any():
        first = int(np.argmax(t))
        if t[first:].all() and beyond and not t[:first].any():
            return first - 1
        return None
    # all False inside the table, True for (some) very large clouds: the step is somewhere above len(t) - 1
    if criteria is None:
        return None
    criteria = list(criteria)
    comb = any if mode == "any" else all

    def f(n: int) -> bool:
        return bool(comb([_eval(c, n) for c in criteria]))

    lo = len(t) - 1                       # f(lo) is False
    hi = next((n for n in _LARGE_PROBES if n > lo and f(n)), None)
    if hi is None:
        return None
    while hi - lo > 1:                    # invariant: f(lo) False, f(hi) True
        mid = (lo + hi) // 2
        if f(mid):
            hi = mid
        else:
            lo = mid
    # a step function has no other transition: spot-check both sides (geometric + neighbouring counts)
    below = {max(len(t) - 1, lo - d) for d in (0, 1, 2, 7, 64, 1000)} | {len(t) - 1 + (lo - len(t) + 1) * k // 8 for k in range(9)}
    above = {hi + d for d in (0, 1, 2, 7, 64, 1000)} | {n for n in _LARGE_PROBES if n > hi}
    if any(f(n) for n in below) or not all(f(n) for n in above):
        return None
    return lo


def fold_levels(criteria: Sequence[Callable], root_edge: float, upto: int):
    """Per-level form of `any(criteria)` for subdivision with node-size guards and geometric criteria.

    Returns a list of (first_level, table, beyond, count criteria, geometric terms): the count decision table and the
    native terms (GeometricCriterion.term) that apply from `first_level` on (until the next entry's first level); the
    last entry applies to every deeper level.  A node splits iff the table OR one of the terms says so.  Without guarded
    criteria the list has one entry that starts at level 0."""
    criteria = list(criteria)
    guarded = (CountCriterion, GeometricCriterion)
    limits = [c.level_limit(root_edge) if isinstance(c, guarded) else NO_LEVEL_LIMIT for c in criteria]
    cuts = sorted({0} | {l for l in limits if l < NO_LEVEL_LIMIT})
    out = []
    for first in cuts:
        active = [c for c, l in zip(criteria, limits) if l > first]
        plain = [CountCriterion(c.op, c.n) if isinstance(c, CountCriterion) else c for c in active
                 if not isinstance(c, GeometricCriterion)]
        terms = [c.term() for c in active if isinstance(c, GeometricCriterion)]
        if plain:
            table, beyond = fold_count_criteria(plain, "any", upto)
        else:
            table, beyond = np.zeros(upto + 1, dtype=np.uint8), False
        out.append((first, table, beyond, plain, terms))
    return out
