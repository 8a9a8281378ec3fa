"""bench.py --dump-outputs: one .npy per result field, rows in (ref_id, query_id) order, a size cap met by a sample of
pairs that does not depend on the order or the number of rows a build returns."""
import importlib.util
import os

import numpy as np

from skani_b200.host import RESULT_DTYPE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def results(n, seed):
    rng = np.random.default_rng(seed)
    pairs = rng.choice(500 * 500, n, replace=False)
    res = np.zeros(n, RESULT_DTYPE)
    res["ref_id"], res["query_id"] = pairs // 500, pairs % 500
    for f in ("ani", "af_query", "af_ref", "std"):
        res[f] = rng.random(n).astype(np.float32)
    res["total_bases_covered"] = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    return res


def test_dump_fields_types_order(tmp_path):
    bench = load_bench()
    res = results(300, 1)
    info = bench.dump_outputs(res[::-1], str(tmp_path))
    assert info["rows"] == 300 and not info["sampled"]
    assert sorted(os.listdir(tmp_path)) == sorted(n + ".npy" for n in RESULT_DTYPE.names)
    want = res[np.lexsort((res["query_id"], res["ref_id"]))]
    for n in RESULT_DTYPE.names:
        a = np.load(tmp_path / (n + ".npy"))
        assert a.dtype == (np.float32 if RESULT_DTYPE[n] == np.float32 else np.float64), n
        assert np.array_equal(a, want[n].astype(a.dtype)), n
    assert np.array_equal(np.load(tmp_path / "total_bases_covered.npy"), want["total_bases_covered"].astype(np.float64))


def test_dump_sample_is_stable(tmp_path, monkeypatch):
    bench = load_bench()
    row_bytes = 12 * 4 + 6 * 8
    monkeypatch.setattr(bench, "DUMP_LIMIT", (1 << 20) + 100 * row_bytes)
    res = results(1000, 2)
    a = bench.dump_outputs(res, str(tmp_path / "a"))
    b = bench.dump_outputs(res[np.random.default_rng(3).permutation(1000)], str(tmp_path / "b"))
    assert a["rows"] == b["rows"] == 100 and a["sampled"]
    for n in ("ref_id", "query_id", "ani"):
        assert np.array_equal(np.load(tmp_path / "a" / (n + ".npy")), np.load(tmp_path / "b" / (n + ".npy"))), n
    ids = np.load(tmp_path / "a" / "ref_id.npy") * 500 + np.load(tmp_path / "a" / "query_id.npy")
    assert np.all(np.diff(ids) > 0)
