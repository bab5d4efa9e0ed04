"""bench.py --dump-outputs (bench.write_outputs): all ranks together stay within the budget; outputs that fit are written
whole, larger ones as a fixed, seeded sample of elements stored next to their flat indices."""
import numpy as np
import pytest

import bench


def _outputs(views, hw, P):
    g = np.random.default_rng(7)
    return {"color": g.random((views, 3, hw, hw), dtype=np.float32),
            "radii": g.integers(0, 40, (views, P)).astype(np.int32)}


def _written(path, world, rank, name):
    return np.load(path / f"{name}{f'_rank{rank}' if world > 1 else ''}.npy")


def test_outputs_that_fit_are_written_whole(tmp_path):
    out = _outputs(2, 16, 1000)
    bench.write_outputs(tmp_path, out, budget=10**6)
    assert sorted(p.name for p in tmp_path.iterdir()) == ["color.npy", "radii.npy"]
    for k, a in out.items():
        got = np.load(tmp_path / f"{k}.npy")
        assert got.dtype == np.float32
        np.testing.assert_array_equal(got, a)


@pytest.mark.parametrize("world", [1, 3, 8])
def test_larger_outputs_are_a_seeded_sample_within_the_budget_of_all_ranks(tmp_path, world):
    budget = 200_000
    out = _outputs(4, 64, 20_000)                      # 517 KB per rank in float32
    total = sum(bench.write_outputs(tmp_path / "a", out, world, r, budget=budget) for r in range(world))
    assert total == sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= budget
    for r in range(world):
        bench.write_outputs(tmp_path / "b", out, world, r, budget=budget)
        for k, a in out.items():
            vals, idx = _written(tmp_path / "a", world, r, k), _written(tmp_path / "a", world, r, k + "_index")
            assert vals.dtype == np.float32 and idx.dtype == np.float64 and 0 < len(vals) == len(idx) < a.size
            np.testing.assert_array_equal(vals, a.reshape(-1)[idx.astype(np.int64)])
            # the same elements in every run
            np.testing.assert_array_equal(idx, _written(tmp_path / "b", world, r, k + "_index"))


def test_c2_outputs_of_three_ranks_fit_the_real_budget(tmp_path):
    views, hw, P = bench.VIEWS, bench.HW, bench.P_GAUSS   # 22 MB per rank: whole at N = 1, sampled at N = 3
    out = {"color": np.zeros((views, 3, hw, hw), np.float32), "radii": np.zeros((views, P), np.int32)}
    assert bench.write_outputs(tmp_path / "one", out) > sum(a.nbytes for a in out.values())
    assert sum(bench.write_outputs(tmp_path / "three", out, 3, r) for r in range(3)) <= bench.DUMP_BUDGET
