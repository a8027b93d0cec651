"""bench.py pieces that run without a GPU: the `parity` leg (the step's result frames vs the oracle on the bit-identical NumPy
twin) and the N > 1 summary matrix on the frames of a MIXED workload - exercised through the NumPy engine stand-in."""
import tempfile

import numpy as np

import cpu_engine


def test_parity_leg_and_summary_matrix_on_a_mixed_frame():
    import bench
    import anovos.drift_stability.drift_detector as dd
    from anovos_b200 import parallel, synth
    from anovos_b200.frame import ColumnFrame
    rows, cols, cat_every = 20_000, 8, 4
    with cpu_engine.installed():
        src = ColumnFrame.from_arrow(synth.host_table(rows, cols, cat_every=cat_every))
        tgt = ColumnFrame.from_arrow(synth.host_table(rows, cols, seed=43, shifted=True, cat_every=cat_every))
        frames = bench.stats_step(src)
        drift = dd.statistics(None, tgt, src, method_type="all", use_sampling=False, source_path=tempfile.mkdtemp()).toPandas()
        par = bench.parity_check(rows, cols, 0, cat_every, src, frames, drift)
    assert par["mismatches"] == 0 and par["cells_checked"] > 100, par
    assert set(par["columns"]) == {"c0000", "c0001", "c0002", "c0003", "c0004"}       # four numeric families + one string column
    assert par["drift"]["max_rel_err"] < 1e-9
    # the per-rank summary matrix of the N > 1 exchange: frames of different row counts align on `attribute`
    m, names = parallel.frames_to_matrix(frames)
    assert m.shape == (cols, len(names)) and "stddev" in names and "fill_count" in names
    string_rows = [i for i, c in enumerate(frames[0]["attribute"]) if c in ("c0003", "c0007")]
    assert np.isnan(m[string_rows][:, names.index("stddev")]).all()


def _decoded(files, key):
    """The values the caller received: the `.nonfinite` codes put null / NaN, +inf and -inf back."""
    a = files[key + ".npy"].copy()
    code = files.get(key + ".nonfinite.npy", np.zeros_like(a))
    assert np.all(a[code != 0] == 0)
    a[code == 1], a[code == 2], a[code == 3] = np.nan, np.inf, -np.inf
    return a


def test_dump_outputs_writes_every_field_of_the_result_tables(tmp_path):
    import zlib
    import pandas as pd
    import bench
    from anovos_b200 import synth
    from anovos_b200.frame import ColumnFrame
    rows, cols = 20_000, 8
    with cpu_engine.installed():
        frames = bench.stats_step(ColumnFrame.from_arrow(synth.host_table(rows, cols, cat_every=4)))
    named = list(zip(bench.STATS_FUNCTIONS, frames))
    named.append(("special", pd.DataFrame({"attribute": ["w", "x", "y", "z"], "v": [1.5, np.inf, -np.inf, np.nan],
                                           "t": pd.array(["2.5", None, "text", "-inf"], dtype="string")})))
    bench.dump_outputs(str(tmp_path / "a"), named)
    files = {p.name: np.load(p) for p in (tmp_path / "a").iterdir()}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in files.values())
    assert files["measures_of_centralTendency.mean.nonfinite.npy"].any()        # string columns have no mean
    for fn, df in named:
        assert np.array_equal(files[fn + ".attribute.crc32.npy"], [zlib.crc32(a.encode()) for a in df["attribute"]])
        for field in df.columns:
            if field not in ("attribute", "mode", "t"):
                assert np.array_equal(_decoded(files, "%s.%s" % (fn, field)), df[field].to_numpy(np.float64, na_value=np.nan),
                                      equal_nan=True)
    central = named[1][1]
    mode_num = _decoded(files, "measures_of_centralTendency.mode")
    mode_crc = files["measures_of_centralTendency.mode.crc32.npy"]
    for i, (a, v) in enumerate(zip(central["attribute"], central["mode"])):
        assert mode_crc[i] == zlib.crc32(str(v).encode())
        assert np.isnan(mode_num[i]) if a in ("c0003", "c0007") else mode_num[i] == float(v)   # string columns: the mode is text
    assert np.array_equal(_decoded(files, "special.t"), [2.5, np.nan, np.nan, -np.inf], equal_nan=True)
    assert np.array_equal(_decoded(files, "special.t.crc32"), [zlib.crc32(b"2.5"), np.nan, zlib.crc32(b"text"), zlib.crc32(b"-inf")],
                          equal_nan=True)
    # over the size limit: the same fixed sample of rows on every call, named by the attribute CRCs
    limit = sum(a.nbytes for a in files.values()) // 2
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), named, limit_bytes=limit)
    sampled = {p.name: np.load(p) for p in (tmp_path / "b").iterdir()}
    assert sampled.keys() == files.keys() and 0 < sum(a.nbytes for a in sampled.values()) <= limit
    assert all(np.isfinite(a).all() and np.array_equal(a, np.load(tmp_path / "c" / n)) for n, a in sampled.items())
    kept = sampled["measures_of_counts.attribute.crc32.npy"]
    full = list(files["measures_of_counts.attribute.crc32.npy"])
    idx = [full.index(c) for c in kept]
    assert idx == sorted(idx) and np.array_equal(sampled["measures_of_counts.fill_count.npy"],
                                                 files["measures_of_counts.fill_count.npy"][idx])
