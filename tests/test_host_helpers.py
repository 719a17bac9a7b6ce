"""Host-side helpers that restate reference encodings outside the CUDA library (no GPU needed): bucket definitions built in Python for the
histogram entry points, and the numpy models of the device generators that bench.py / the tests rebuild oracle inputs from."""
import numpy as np
import pytest


def test_bucket_definitions_match_the_reference_serialisation(oracle):
    # HistogramBuckets.serialize: GeometricBuckets Histogram.scala:609-617, CustomBuckets :878-884 (NibblePack.packDoubles of the tops)
    from filodb_b200 import capi
    from oracle import hist as H
    for first, mult, n, minus_one in ((2.0, 3.0, 20, False), (1.0, 2.0, 8, False), (0.5, 1.5, 64, False)):
        d, fmt = capi.geometric_bucket_def(first, mult, n)
        assert fmt == 3 and (d == H.Buckets.geometric(first, mult, n).serialize()).all()
    rng = np.random.default_rng(3)
    for les in ([2.0 * 3 ** i for i in range(19)] + [float("inf")], [0.5 * 2 ** i for i in range(12)] + [float("inf")], [1.0, 2.5, 7.25],
                list(np.cumsum(rng.random(33)) * 1e3), [5.0]):
        d, fmt = capi.custom_bucket_def(les)
        ref = H.Buckets.custom(les).serialize()
        assert fmt == 5 and d.size == ref.size and (d == ref).all(), les


def test_numpy_generator_models_agree():
    # bench.gen_hist_series_np (vectorised) == tests/synth_ref.gen_hist_series (row by row): both model hist_row in synth_kernels.cu
    import bench
    from tests import synth_ref as sr
    for seed, gid, rows, nb, reset in ((42, 0, 480, 20, 97), (42, 97, 480, 20, 97), (5, 194, 230, 13, 97), (7, 12345, 64, 8, 0)):
        assert (bench.gen_hist_series_np(seed, gid, rows, nb, reset) == sr.gen_hist_series(seed, gid, rows, nb, reset)).all()
    g = bench.synth_group_ids(42, 1000, 64, 7)
    assert list(g) == [sr.group_id(42, 1000 + i, 7) for i in range(64)]


def test_bench_dump_outputs_are_fixed_and_bounded(tmp_path, oracle):
    # bench.py --dump-outputs: a result too large for the limit is sampled by rows, the same rows every time; the files are float64 and two
    # runs with the same arguments write the same bits
    import subprocess
    import sys
    import bench
    row_bytes = 481 * 8
    rows = bench.dump_row_sample(10_000_000, row_bytes)
    assert (rows == bench.dump_row_sample(10_000_000, row_bytes)).all() and (np.diff(rows) > 0).all() and rows[-1] < 10_000_000
    assert rows.size * (row_bytes + 8) + 2 * bench.NPY_HEADER_BYTES <= bench.DUMP_LIMIT_BYTES
    assert bench.dump_row_sample(1000, row_bytes) is None
    got = []
    for run in ("a", "b"):
        subprocess.run([sys.executable, bench.__file__, "--impl", "reference", "--workload", "c2", "--series", "300", "--cpu-series", "300",
                        "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path / run)], check=True, capture_output=True)
        assert sorted(p.name for p in (tmp_path / run).iterdir()) == ["values.npy"]
        got.append(np.load(tmp_path / run / "values.npy"))
    assert got[0].dtype == np.float64 and got[0].shape == (300, 481) and np.isfinite(got[0]).any()
    assert (got[0].view(np.uint64) == got[1].view(np.uint64)).all()
