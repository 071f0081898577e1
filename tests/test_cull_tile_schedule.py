"""CPU check of the unit schedule of the culled symmetric MLAPM evaluation (piml_b200/csrc/mlapm.cu, CullItem,
CullKeep, mlapm_cull_masks_kernel, mlapm_sym_tiles_kernel): with every column tile live, the (128-row tile, 32-column
tile) units cover every unordered pair of agents exactly once, and the pairs inside a row tile once in each
direction.  A unit covers whole tiles, so pairs of agents reduce to pairs of column tiles."""
import numpy as np
import pytest

BLOCK, RT, CT = 512, 128, 32
RPB, CPB = BLOCK // RT, BLOCK // CT
TPR = CPB // RPB                                                  # column tiles per row tile


def units(T):
    """(row tile, global column tile, diag) of every unit the kernel evaluates when every column tile is live."""
    D = T // 2
    out = []
    for c in range(RPB * T * (D + 1)):                            # item c = R * (D + 1) + d
        R, d = divmod(c, D + 1)
        I = R // RPB
        if T % 2 == 0 and d == D and 2 * I >= T:                  # CullKeep: the pairs at d = T/2 belong to I < T/2
            continue
        J = (I + d) % T
        first = (R % RPB) * TPR if d == 0 else 0                  # CullItem::first_tile
        for ct in range(first, CPB):
            diag = d == 0 and ct // TPR == R % RPB
            out.append((R, J * CPB + ct, diag))
    return out


@pytest.mark.parametrize("T", list(range(1, 42)) + [195, 196])
def test_every_agent_pair_exactly_once(T):
    u = np.array(units(T), dtype=np.int64)
    ntiles = T * CPB
    R, col, diag = u[:, 0], u[:, 1], u[:, 2].astype(bool)
    # unordered pairs of column tiles in different row tiles: one symmetric unit (R, b) with a in R, b elsewhere
    sym = np.zeros((ntiles, ntiles), np.int32)
    rows_tiles = R[~diag, None] * TPR + np.arange(TPR)[None, :]   # the row tile's own column tiles
    a = rows_tiles.ravel()
    b = np.repeat(col[~diag], TPR)
    assert (a // TPR != b // TPR).all(), "a symmetric unit inside its own row tile"
    np.add.at(sym, (np.minimum(a, b), np.maximum(a, b)), 1)
    ra = np.arange(ntiles) // TPR
    other = ra[:, None] != ra[None, :]
    upper = np.triu(np.ones((ntiles, ntiles), bool), 1)
    assert (sym[other & upper] == 1).all()
    assert (sym[~(other & upper)] == 0).all()
    # pairs inside a row tile: the row direction of units (R, own column tile), each of the R's 4 tiles exactly once
    own = np.zeros((T * RPB, TPR), np.int32)
    assert (col[diag] // TPR == R[diag]).all()
    np.add.at(own, (R[diag], col[diag] % TPR), 1)
    assert (own == 1).all()
    # each row tile meets each unordered block pair once
    assert len({(r, c // CPB) for r, c, _ in u.tolist()}) == RPB * T * (T + 1) // 2
