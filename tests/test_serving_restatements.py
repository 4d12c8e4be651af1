"""The GPU serving tests (tests/test_gpu_serving.py) compare the device parsers with small RESTATEMENTS of the container's own
parsing routes.  Here the restatements themselves -- and the host routes serving.py falls back to -- are checked against what
the container's real functions (encoder.csv_to_dmatrix, encoder.libsvm_to_dmatrix, serve_utils._get_sparse_matrix_from_libsvm
+ xgb.DMatrix) built on the very same bodies: tests/golden/container/serving.npz, recorded by
tests/golden/make_container_goldens.py.  CPU test engine."""
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "container", "serving.npz")
TAB_INSIDE_TOKEN = "1 1:2\t3:4 5:6"          # a token with a tab inside: the container's float() refuses it
NO_ENTRIES = "1\n0\n"                        # labels only: the container's empty DMatrix


def libsvm_bodies():
    import test_gpu_serving as T
    bodies = [T._libsvm_body(np.random.default_rng(31 + ob), 400, 40, ob) for ob in (True, False)]
    return bodies + ["1 1:0.5 1:0.25 2:3", "1 1:0.5 2:3\n0", "1 +1:0.5 2:3", "1 1:0.12345678901234567890123 2:3", "1 1:nan 2:3",
                     "1 1:0.5 1:0.25 2:3\n0\n1 4:1", "0 3:1e-3\t7:2 \n\n1 1:5", "1 0:1 5:2\n0 2:3"]


def csv_bodies():
    rng = np.random.default_rng(7)
    X = rng.standard_normal((300, 9)) * np.exp(rng.uniform(-20, 20, size=(300, 9)))
    lines = []
    for r in range(300):
        vals = [("%.6g", "%.17g", "%.3e")[r % 3] % v for v in X[r]]
        if r % 11 == 0:
            vals[r % 9] = ""
        if r % 13 == 0:
            vals[(r + 2) % 9] = ["nan", "inf", "-inf", "+1.5", "-0", "1e-45", "1e39"][(r // 13) % 7]
        lines.append(",".join(vals))
    bodies = [("\n".join(lines), ",")]
    for delim in (";", "\t", " "):
        bodies.append(("\n".join(delim.join("%g" % v for v in row) for row in rng.standard_normal((20, 4))), delim))
    return bodies


@pytest.fixture()
def engine(monkeypatch):
    import sagemaker_xgboost_container_b200 as xgb
    from sagemaker_xgboost_container_b200 import backend
    from oracle.engine import OracleBackend
    monkeypatch.setattr(backend, "_BACKEND", OracleBackend(error_cls=xgb.XGBoostError))
    return xgb


@pytest.fixture(scope="module")
def golden():
    g = np.load(GOLDEN)
    mats = {k: g[k] for k in g.files if k not in ("errors", "dense_is_sparse_with_zeros")}
    for k in g["dense_is_sparse_with_zeros"]:          # recorded where the container's dense route gave exactly this
        mats[str(k)] = np.nan_to_num(mats[str(k).replace("dense", "sparse")], nan=0.0, posinf=np.inf, neginf=-np.inf)
    return mats, json.loads(str(g["errors"]))


def _matrix(d):
    return d.handle.X                                   # oracle engine: the float32 matrix the DMatrix holds (NaN = missing)


def _same(a, b):
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.nan_to_num(a), np.nan_to_num(b))


def _check(key, golden, *routes):
    mats, errors = golden
    if key in errors:
        for route in routes:
            with pytest.raises(Exception) as e:
                route()
            assert type(e.value).__name__ == errors[key], key
    else:
        for route in routes:
            assert _same(np.asarray(route(), np.float32), mats[key]), key


def test_libsvm_restatements_equal_the_reference_functions(engine, golden):
    import test_gpu_serving as T
    from sagemaker_xgboost_container_b200 import serving
    bodies = libsvm_bodies()
    assert sum(k.startswith("libsvm_") for k in list(golden[0]) + list(golden[1])) == 2 * len(bodies) + 2
    for i, body in enumerate(bodies):
        # sparse route of the algorithm-mode handler (serve_utils.py:94-118 + xgb.DMatrix(csr)): absent entries are missing
        _check("libsvm_sparse/%d" % i, golden, lambda: T._ref_sparse_route(body), lambda: _matrix(serving.sparse_libsvm_to_dmatrix(body)))
        # dense route of the script-mode handler (encoder.py:54-86): absent entries are 0.0
        _check("libsvm_dense/%d" % i, golden, lambda: T._ref_dense_route(body), lambda: _matrix(serving.libsvm_to_dmatrix(body)))
    assert golden[0]["libsvm_dense/no_entries"].shape[0] == serving.libsvm_to_dmatrix(NO_ENTRIES).num_row() == 0
    assert golden[1]["libsvm_sparse/tab_inside_token"] == "ValueError"
    with pytest.raises(ValueError):
        serving.sparse_libsvm_to_dmatrix(TAB_INSIDE_TOKEN)


def test_csv_restatement_equals_the_reference_function(engine, golden):
    import test_gpu_serving as T
    from sagemaker_xgboost_container_b200 import serving
    for i, (body, delim) in enumerate(csv_bodies()):
        with np.errstate(over="ignore"):
            routes = [lambda: _matrix(serving.csv_to_dmatrix(body, dtype=float))]          # CPU engine: the mirror's host route
            if delim == ",":
                routes.append(lambda: T._reference_route(body))
            _check("csv/%d" % i, golden, *routes)
