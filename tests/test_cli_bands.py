"""The command line's row-band feature_adj (torchrun, WORLD_SIZE > 1) without a GPU: every rank forms exactly the rows of
its tile-row shard and of its result band, each equal to the same rows of the full matrix."""
import numpy as np
import pytest
import torch


@pytest.mark.parametrize("dataset", ["cora", "polblogs"])
@pytest.mark.parametrize("nofeature", [False, True])
@pytest.mark.parametrize("n,world", [(300, 3), (90, 3), (1000, 8)])
def test_feature_adj_bands_are_rows_of_the_full_matrix(dataset, nofeature, n, world):
    from mcgra_b200.engine import TILE, output_band, shard_tile_rows
    from mcgra_b200.main import dot_product_decode, feature_adj_bands
    Z = torch.from_numpy(np.random.RandomState(n).random_sample((n, 12)).astype(np.float32))
    full = torch.eye(n) if nofeature else dot_product_decode(Z, dataset)
    T = (n + TILE - 1) // TILE
    covered = torch.zeros(n, dtype=torch.int64)
    for rank in range(world):
        tr0, tr1 = shard_tile_rows(T, world)[rank]
        need = {(tr0 * TILE, min(n, tr1 * TILE)), output_band(n, rank, world)}
        need = {b for b in need if b[1] > b[0]}
        hb = feature_adj_bands(Z, dataset, rank, world, nofeature)
        assert set(hb.bands) == need                        # nothing beyond the two bands the rank touches
        held = sum(r1 - r0 for r0, r1 in hb.bands)
        assert held <= min(n, tr1 * TILE) - min(n, tr0 * TILE) + max(0, output_band(n, rank, world)[1]
                                                                         - output_band(n, rank, world)[0])
        for (r0, r1), t in hb.bands.items():
            assert tuple(t.shape) == (r1 - r0, n)
            torch.testing.assert_close(t, full[r0:r1], rtol=0, atol=1e-6)
        r0, r1 = tr0 * TILE, min(n, tr1 * TILE)
        covered[r0:max(r0, r1)] += 1
        torch.testing.assert_close(hb.rows(r0, r1, "cpu"), full[r0:r1], rtol=0, atol=1e-6)
    assert bool((covered == 1).all())                       # the tile-row shards cover every row once


def test_dot_product_decode_full_is_unchanged():
    """dot_product_decode without `rows` computes what main.dot_product_decode always did."""
    from mcgra_b200.main import dot_product_decode
    Z = torch.from_numpy(np.random.RandomState(0).standard_normal((70, 9)).astype(np.float32))
    eye = torch.eye(70)
    assert torch.equal(dot_product_decode(Z, "cora"), torch.sigmoid(torch.relu(Z @ Z.t() - eye)))
    Zn = torch.nn.functional.normalize(Z, p=2, dim=1)
    assert torch.equal(dot_product_decode(Z, "polblogs"), torch.relu(Zn @ Zn.t() - eye))
