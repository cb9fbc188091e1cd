"""bench.py --dump-outputs: float64 files below 64 MB in all, the same rows on every run."""
import numpy as np

import bench


def test_dump_outputs_are_bounded_exact_and_repeatable(tmp_path):
    rng = np.random.default_rng(3)
    arrays = {"counts": rng.integers(0, 1 << 31, (30_000, 2)).astype(np.uint32),
              "hit_off": np.arange(12_000_000, dtype=np.uint32),
              "genotype_pl": rng.integers(0, 1 << 52, (2_000_000, 3))}
    kept = [bench.dump_outputs(str(tmp_path / d), arrays) for d in ("a", "b")]
    assert kept[0] == kept[1]
    assert kept[0]["counts"] == (30_000, 30_000)
    assert kept[0]["hit_off"][0] < 12_000_000 and kept[0]["genotype_pl"][0] < 2_000_000
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) < 64_000_000
    got = {}
    for name in arrays:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, b)
        got[name] = a
    assert np.array_equal(got["counts"], arrays["counts"])          # small enough: whole and exact
    assert (np.diff(got["hit_off"]) > 0).all()                      # a sample keeps the order of the rows
    assert np.isin(got["genotype_pl"][:, 0], arrays["genotype_pl"][:, 0]).all()
