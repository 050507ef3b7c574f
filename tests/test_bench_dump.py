"""CPU: bench.py --dump-outputs -- the seeded row windows, the copy of the window rows out of each batch, and the float .npy
files they become (every column kind, nulls, the byte budget), checked against the batches they came from."""
import numpy as np
import pyarrow as pa

import bench
from conftest import GOLDEN


def _table(name, tags):
    from oracle.bam_oracle import OracleBam
    return pa.Table.from_batches([OracleBam(str(GOLDEN / name), tag_fields=tags).scan()])


def _dump(t, windows, out, budget=bench.DUMP_BYTES, batch_rows=1000):
    kept = []
    for lo in range(0, t.num_rows, batch_rows):
        bench.keep_window_rows(t.slice(lo, batch_rows).to_batches()[0], lo, windows, kept)
    return bench.dump_outputs(out, kept, windows, "", budget)


def _load(out, t, column):
    typ = t.schema.field(column).type
    if pa.types.is_string(typ) or pa.types.is_list(typ):
        lens = np.load(out / f"{column}.lengths.npy")
        vals = np.load(out / f"{column}.{'bytes' if pa.types.is_string(typ) else 'values'}.npy")
        assert lens.dtype == np.float64 and vals.dtype == (np.float32 if pa.types.is_string(typ) else np.float64)
        rows, p = [], 0
        for n in lens:
            if np.isnan(n):
                rows.append(None)
                continue
            v = vals[p:p + int(n)]
            rows.append(v.astype(np.uint8).tobytes().decode() if pa.types.is_string(typ) else [int(x) for x in v])
            p += int(n)
        assert p == len(vals)
        return rows
    v = np.load(out / f"{column}.npy")
    assert v.dtype == np.float64
    return [None if np.isnan(x) else int(x) for x in v]


def test_windows_are_seeded_strata():
    w = bench.dump_windows(100_000_000)
    assert w == bench.dump_windows(100_000_000) and len(w) == bench.DUMP_WINDOWS
    assert all(hi - lo == bench.DUMP_WINDOW_ROWS for lo, hi in w)
    stratum = 100_000_000 // bench.DUMP_WINDOWS
    assert all(k * stratum <= lo and hi <= (k + 1) * stratum for k, (lo, hi) in enumerate(w))
    assert bench.dump_windows(5000) == [(0, 5000)]


def test_dump_holds_the_window_rows_of_every_column(tmp_path):
    for name, tags in (("multi_chrom_large.bam", ["NM", "MD", "RG"]), ("nanopore_custom_tags.bam", ["pa", "ns", "MD", "tp"])):
        t = _table(name, tags)
        windows = [(0, 3), (990, 1010), (t.num_rows - 5, t.num_rows)] if t.num_rows > 1010 else [(2, 7), (15, t.num_rows)]
        out = tmp_path / name
        info = _dump(t, windows, out, batch_rows=7)
        rows = np.concatenate([np.arange(lo, hi) for lo, hi in windows])
        assert info["rows"] == len(rows) and np.array_equal(np.load(out / "row_index.npy"), rows)
        want = t.take(pa.array(rows))
        assert info["bytes"] == sum(f.stat().st_size for f in out.iterdir())
        for column in t.column_names:
            assert _load(out, t, column) == want[column].to_pylist(), (name, column)


def test_dump_fits_the_budget_with_equal_window_prefixes(tmp_path):
    t = _table("multi_chrom_large.bam", ["NM", "MD"])
    windows = [(100, 600), (2000, 2500), (3500, 4000)]
    info = _dump(t, windows, tmp_path, budget=200_000)
    assert 0 < info["bytes"] <= 200_000 and sum(f.stat().st_size for f in tmp_path.iterdir()) == info["bytes"]
    idx = np.load(tmp_path / "row_index.npy")
    per = info["rows"] // 3
    assert 0 < per < 500 and np.array_equal(idx, np.concatenate([np.arange(lo, lo + per) for lo, _ in windows]))
    assert _load(tmp_path, t, "sequence") == t.take(pa.array(idx.astype(np.int64)))["sequence"].to_pylist()
