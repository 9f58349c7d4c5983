"""CPU checks of drainage-basin labelling: the serial reference against an independent restatement, and the
argument checks of overflow_b200.basins, which refuse bad input before any device call."""
import numpy as np
import pytest

import basins_reference as ref
from overflow_b200 import _native
from overflow_b200.basins import label_basins, pour_point_indices


def test_reference_hand_example():
    # row 0 drains east off the raster; row 1 drains north into row 0, except (1, 2), which steps north-east off the
    # raster; row 2: a pit, NODATA, a cell draining into NODATA
    fdr = np.array([[0, 0, 0], [2, 2, 1], [8, 9, 4]], dtype=np.uint8)
    want = np.array([[3, 3, 3], [3, 3, 6], [7, 0, 9]])
    assert np.array_equal(ref.basins(fdr), want)
    # pour point at (0, 1): (0, 0), (0, 1) and (1, 1) drain through it; everything else reaches no pour point
    want = np.array([[2, 2, 0], [2, 2, 0], [0, 0, 0]])
    assert np.array_equal(ref.basins(fdr, [[0, 1]]), want)


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (41, 1), (23, 29), (64, 65)])
@pytest.mark.parametrize("seed", [0, 1])
def test_reference_walk_equals_pointer_jumping(shape, seed):
    fdr = ref.random_acyclic_codes(*shape, seed=seed)
    labels = ref.basins(fdr)
    assert np.array_equal(labels, ref.basins_by_jumping(fdr))
    outlets = (ref.successors(fdr) < 0) & (fdr.reshape(-1) != 9)
    flat = labels.reshape(-1)
    assert np.array_equal(flat[outlets], np.flatnonzero(outlets) + 1)  # every outlet carries its own label
    assert (flat[fdr.reshape(-1) == 9] == 0).all()


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_reference_pour_points(seed):
    rows, cols = 31, 43
    fdr = ref.random_acyclic_codes(rows, cols, seed=seed)
    rng = np.random.default_rng(100 + seed)
    pp = np.stack([rng.integers(0, rows, 12), rng.integers(0, cols, 12)], axis=1)
    # nested: the successor of a pour point; a NODATA cell; a duplicate; an outlet
    succ = ref.successors(fdr)
    i = int(pp[0, 0] * cols + pp[0, 1])
    if succ[i] >= 0:
        pp = np.vstack([pp, [divmod(int(succ[i]), cols)]])
    nodata = np.argwhere(fdr == 9)
    outlet = np.argwhere(((succ < 0) & (fdr.reshape(-1) != 9)).reshape(rows, cols))
    pp = np.vstack([pp, nodata[:1], pp[:2], outlet[:1]])
    labels = ref.basins(fdr, pp)
    assert np.array_equal(labels, ref.basins_by_jumping(fdr, pp))
    live = [tuple(p) for p in pp if fdr[p[0], p[1]] != 9]
    for r, c in live:
        assert labels[r, c] == r * cols + c + 1
    for r, c in nodata[:1]:
        assert labels[r, c] == 0
    assert set(np.unique(labels)) <= {0} | {r * cols + c + 1 for r, c in live}


def test_reference_reports_cycle():
    fdr = np.full((4, 6), 8, dtype=np.uint8)
    fdr[1, 2], fdr[1, 3] = 0, 4  # east / west pair
    with pytest.raises(ValueError, match="cycle"):
        ref.basins(fdr)
    with pytest.raises(ValueError, match="cycle"):
        ref.basins_by_jumping(fdr)


def test_label_basins_refuses_bad_codes():
    with pytest.raises(TypeError):
        label_basins(np.zeros((3, 3), dtype=np.float32))
    with pytest.raises(ValueError):
        label_basins(np.full((3, 3), 256, dtype=np.int32))


@pytest.mark.parametrize("pp", [
    [[0, 3]], [[3, 0]], [[-1, 0]], [[0, -1]],   # outside a 3 x 3 raster
    [[0, 1, 2]], [1, 2], [[[0, 1]]],            # not (k, 2)
    [[0.0, 1.0]],                               # not integers
])
def test_label_basins_refuses_bad_pour_points(pp):
    with pytest.raises(ValueError):
        label_basins(np.zeros((3, 3), dtype=np.uint8), pour_points=np.asarray(pp))


def test_pour_point_indices():
    assert pour_point_indices(None, (3, 4)) is None
    assert np.array_equal(pour_point_indices([[1, 2], [2, 3], [1, 2]], (3, 4)), [6, 11, 6])
    assert len(pour_point_indices(np.zeros((0, 2), dtype=np.int64), (3, 4))) == 0


def test_basins_command_is_registered():
    import overflow_cli

    cmd = overflow_cli.main.commands["basins"]
    assert cmd is overflow_cli.basins_cli
    opts = {o for p in cmd.params for o in p.opts}
    assert {"--input_file", "--output_file", "--chunk_size", "--pour_points"} <= opts


def test_label_basins_without_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(_native.OverflowB200Error):
        label_basins(np.zeros((5, 5), dtype=np.uint8))
