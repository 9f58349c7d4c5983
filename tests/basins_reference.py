"""Serial CPU reference of drainage-basin labelling (overflow_b200.basins states the rules).

`basins` walks each unlabelled cell's path to a labelled cell or a root and writes the label back along the path
from an explicit stack: every cell is pushed once, O(N) in all.  `basins_by_jumping` restates the same labels by
pointer doubling over whole arrays, an independent route used to cross-check the walk.
"""
import numpy as np

DY = np.array([0, -1, -1, -1, 0, 1, 1, 1], dtype=np.int64)
DX = np.array([1, 1, 0, -1, -1, -1, 0, 1], dtype=np.int64)


def _codes(fdr):
    fdr = np.asarray(fdr)
    if fdr.ndim != 2:
        raise ValueError("flow direction raster must be 2-D")
    if fdr.size and (fdr.min() < 0 or fdr.max() > 255):
        raise ValueError("codes must be in 0..255")
    return np.ascontiguousarray(fdr, dtype=np.int64)


def successors(fdr):
    """Flat index of each cell's downstream cell under the accumulation's edge rule, -1 where there is none."""
    fdr = _codes(fdr)
    rows, cols = fdr.shape
    r, c = np.indices((rows, cols))
    code = fdr
    d = np.where(code <= 7, code, 0)
    nr, nc = r + DY[d], c + DX[d]
    inside = (code <= 7) & (nr >= 0) & (nr < rows) & (nc >= 0) & (nc < cols)
    nidx = np.where(inside, nr * cols + nc, 0)
    ok = inside & (fdr.reshape(-1)[nidx] != 9)
    return np.where(ok, nidx, -1).reshape(-1)


def _roots(fdr, pour_points):
    """(successor array with pour points cut, root label per cell or -1 where the cell is not a root)."""
    fdr = _codes(fdr)
    rows, cols = fdr.shape
    n = rows * cols
    succ = successors(fdr)
    nodata = fdr.reshape(-1) == 9
    own = np.arange(1, n + 1, dtype=np.int64)
    root = np.where(succ < 0, own if pour_points is None else 0, -1)
    if pour_points is not None:
        pp = np.asarray(pour_points, dtype=np.int64).reshape(-1, 2)
        idx = pp[:, 0] * cols + pp[:, 1]
        idx = idx[~nodata[idx]]
        succ[idx] = -1
        root[idx] = idx + 1
    root[nodata] = 0
    succ[nodata] = -1
    return succ, root


def basins(fdr, pour_points=None):
    """int64 labels by a serial path walk; raises ValueError on a cycle."""
    fdr = _codes(fdr)
    rows, cols = fdr.shape
    succ, root = _roots(fdr, pour_points)
    succ, root = succ.tolist(), root.tolist()
    label = [-1] * (rows * cols)
    on_stack = bytearray(rows * cols)
    for start in range(rows * cols):
        if label[start] >= 0:
            continue
        stack = []
        c = start
        while label[c] < 0 and root[c] < 0:
            if on_stack[c]:
                raise ValueError("flow direction raster contains a cycle")
            on_stack[c] = 1
            stack.append(c)
            c = succ[c]
        lab = label[c] if label[c] >= 0 else root[c]
        label[c] = lab
        for u in stack:
            label[u] = lab
    return np.array(label, dtype=np.int64).reshape(rows, cols)


def basins_by_jumping(fdr, pour_points=None):
    """The same labels by pointer doubling (numpy); raises ValueError on a cycle."""
    fdr = _codes(fdr)
    rows, cols = fdr.shape
    succ, root = _roots(fdr, pour_points)
    n = rows * cols
    ptr = np.where(succ < 0, np.arange(n), succ)
    for _ in range(max(1, n).bit_length() + 1):
        nxt = ptr[ptr]
        if np.array_equal(nxt, ptr):
            break
        ptr = nxt
    if n and (root[ptr] < 0).any():
        raise ValueError("flow direction raster contains a cycle")
    return root[ptr].reshape(rows, cols) if n else np.zeros((rows, cols), dtype=np.int64)


def random_acyclic_codes(rows, cols, seed, special=0.1):
    """Codes that point strictly downhill on a random permutation of heights (so no cycle), with off-raster steps,
    code-8 cells and, on a fraction `special` of the cells, NODATA or codes 10..255."""
    rng = np.random.default_rng(seed)
    height = rng.permutation(rows * cols).reshape(rows, cols)
    fdr = np.full((rows, cols), 8, dtype=np.uint8)
    for r in range(rows):
        for c in range(cols):
            if rng.random() < 0.05:
                continue  # a code-8 outlet
            cand = [d for d in range(8)
                    if not (0 <= r + DY[d] < rows and 0 <= c + DX[d] < cols) or height[r + DY[d], c + DX[d]] < height[r, c]]
            if cand:
                fdr[r, c] = cand[rng.integers(len(cand))]
    mask = rng.random((rows, cols)) < special
    fdr[mask] = rng.choice(np.array([9, 9, 9, 10, 77, 200, 255], dtype=np.uint8), size=int(mask.sum()))
    return fdr
