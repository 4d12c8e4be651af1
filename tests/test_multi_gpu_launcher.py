"""`use_dask_gpu_training=true` on the native one-process-per-GPU path (multi_gpu.py; SURVEY.md section 8(f) row 3, reference
algorithm_mode/train.py:183-214 + distributed_gpu/distributed_gpu_training.py:93-222).

CPU: world_size-2 runs of the launcher on the oracle-backed test engine (tracker rendezvous, row shards read per rank,
master-only model / checkpoints, failures surfaced) -- the sharded job must write the model the single-process job writes.
GPU (needs 2 GPUs): the same through the CUDA engine, model bit-identical to the 1-GPU model."""
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "helpers"))
import oracle_worker_init  # noqa: E402

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "abalone")


def _libsvm_to_csv(src, dst):
    with open(dst, "w") as out:
        for line in open(src):
            p = line.split()
            vals = {int(k): v for k, v in (kv.split(":") for kv in p[1:])}
            out.write(",".join([p[0]] + [vals.get(i, "0") for i in range(1, 9)]) + "\n")


def _channels(tmp_path):
    tr, va = tmp_path / "train", tmp_path / "validation"
    tr.mkdir(); va.mkdir()
    _libsvm_to_csv(os.path.join(G, "abalone.train_0"), tr / "abalone.train_0.csv")
    _libsvm_to_csv(os.path.join(G, "abalone.train_1"), tr / "abalone.train_1.csv")
    _libsvm_to_csv(os.path.join(G, "abalone.validation"), va / "abalone.validation.csv")
    return tr, va


def test_shards_cover_the_channel_exactly_once(tmp_path):
    from sagemaker_xgboost_container_b200 import multi_gpu
    tr, _ = _channels(tmp_path)
    files = multi_gpu._channel_files(str(tr), "csv")
    whole = b"\n".join(open(f, "rb").read().strip(b"\n") for f in files)
    for world in (1, 2, 3, 8):
        parts = [multi_gpu._csv_shard_text(files, r, world) for r in range(world)]
        assert all(n == 2922 for _, n in parts)
        assert b"\n".join(t for t, _ in parts) == whole
        sizes = [t.count(b"\n") + 1 for t, _ in parts]
        assert max(sizes) - min(sizes) <= 1
    assert multi_gpu._csv_shard_text(files, 0, 4000)[0] == b""           # more workers than lines: an empty shard, reported by load_shard
    import pyarrow as pa
    import pyarrow.parquet as pq
    pqd = tmp_path / "pq"
    pqd.mkdir()
    arr = np.genfromtxt(whole.decode().splitlines(), delimiter=",", dtype=np.float32)
    for i, (a, b) in enumerate([(0, 1000), (1000, 2922)]):
        pq.write_table(pa.table({"c%d" % j: arr[a:b, j] for j in range(arr.shape[1])}), pqd / ("part-%d.parquet" % i), row_group_size=300)
    # (the DMatrix itself needs an engine: only the row bookkeeping is checked here)
    metas = [pq.ParquetFile(f) for f in multi_gpu._channel_files(str(pqd), "parquet")]
    assert sum(m.metadata.num_rows for m in metas) == 2922


def test_validation_mirrors_the_reference_checks():
    from sagemaker_xgboost_container_b200 import multi_gpu as mg
    rep = {"train": {"S3DistributionType": "FullyReplicated"}}
    assert mg.validate_gpu_train_configuration("hist", 1, 8, "File", "csv", rep) == []
    assert mg.validate_gpu_train_configuration("gpu_hist", 2, 8, "File", "parquet", rep) == []
    assert mg.validate_gpu_train_configuration("approx", 1, 8, "File", "csv", rep) == [mg.NON_GPU_ERROR_MSG]
    assert mg.validate_gpu_train_configuration("hist", 1, 0, "Pipe", "libsvm", rep) == [mg.NON_GPU_ERROR_MSG, mg.PIPE_MODE_ERROR_MSG, mg.INPUT_FORMAT_ERROR_MSG]
    sharded = {"train": {"S3DistributionType": "ShardedByS3Key"}}
    assert mg.validate_gpu_train_configuration("hist", 1, 8, "File", "csv", sharded) == []
    assert mg.validate_gpu_train_configuration("hist", 2, 8, "File", "csv", sharded) == [mg.NOT_REPLICATED_ERROR_MSG]


def test_sagemaker_train_with_use_dask_gpu_training_runs_the_native_launcher(tmp_path, capfd):
    """The container's entry point with the HP set hands its launcher the arguments recorded in
    tests/golden/container/entrypoint.json (train.py:203, the one-line binding of INTEGRATION.md); replayed on multi_gpu with
    two worker processes, the model equals the one the container's ordinary single-process route trained.  The container's
    callback helpers, which the launcher uses when the container is installed, are stood in for by
    oracle_worker_init.use_oracle_engine_with_container_callbacks: checkpoints come from the master only."""
    from sagemaker_xgboost_container_b200 import multi_gpu
    from oracle import ubjson
    from util import assert_same_structure
    rec = json.load(open(os.path.join(os.path.dirname(G), "container", "entrypoint.json")))
    kw = json.loads(json.dumps(rec["dask_route_launcher_call"]["kwargs"]).replace("{tmp}", str(tmp_path)))
    assert kw["num_gpus"] == 2 and kw["content_type"] == "csv"
    _channels(tmp_path)
    os.makedirs(kw["checkpoint_dir"])
    multi_gpu.run_training_with_dask(**kw, worker_init=oracle_worker_init.use_oracle_engine_with_container_callbacks)
    out = capfd.readouterr().out
    lines = [l for l in out.splitlines() if l.startswith("[") and "train-rmse:" in l]
    assert len(lines) == 8 and "validation-rmse:" in lines[-1]          # the master's monitor only: one line per round, not two
    assert sorted(os.listdir(kw["model_dir"])) == ["xgboost-model"]
    # both ranks asked for callbacks, one of them as the master; checkpoints were written, by that rank only
    files = os.listdir(kw["checkpoint_dir"])
    notes = sorted(f.rsplit("-", 1)[1] for f in files if f.startswith("get_callbacks-"))
    assert notes == ["False", "True"]
    assert len([f for f in files if f.startswith("xgboost-checkpoint")]) >= 1
    got = ubjson.model_from_xgb_json(ubjson.load(os.path.join(kw["model_dir"], "xgboost-model")))
    g = np.load(os.path.join(os.path.dirname(G), "container", "entrypoint_models.npz"))
    ref = {k.split("/")[-1]: g[k] for k in g.files if k.startswith("dask_route_single_process/0/")}
    assert_same_structure(got, ref)
    np.testing.assert_array_equal(got["split_cond"], ref["split_cond"])


def test_unbound_reference_dask_route_still_trains_through_xgboost_dask(tmp_path, monkeypatch, capfd):
    """Without the multi_gpu binding the container's own run_training_with_dask (distributed_gpu_training.py:93-222) reaches
    `xgboost.dask.DaskDMatrix` / `xgboost.dask.train` of this package.  Its calls, recorded in
    tests/golden/container/entrypoint.json (Dask cluster stubbed), replayed on xgb.dask: the same inputs, the warning that
    names the native launcher, every round printed twice (the container adds an EvaluationMonitor and leaves dask.train's
    verbose_eval at its default True), and the model the recorded call trained."""
    import hashlib
    import sagemaker_xgboost_container_b200 as xgb
    from sagemaker_xgboost_container_b200 import backend
    from oracle.engine import OracleBackend
    from oracle import ubjson
    from util import assert_same_structure, max_leaf_diff
    monkeypatch.setattr(backend, "_BACKEND", OracleBackend(error_cls=xgb.XGBoostError))
    xgb.install_as_xgboost()
    import xgboost.dask as dxgb
    assert dxgb is xgb.dask and sys.modules["xgboost"].dask is xgb.dask
    rec = json.load(open(os.path.join(os.path.dirname(G), "container", "entrypoint.json")))["dask_route_unbound"]
    tr, va = _channels(tmp_path)
    # dask_data_utils.read_data: the channel's CSV files in name order, label in column 0
    arrays = [np.concatenate([np.loadtxt(f, delimiter=",", ndmin=2) for f in sorted(str(p) for p in d.iterdir())]) for d in (tr, va)]
    mats = []
    for a, m in zip(arrays, rec["matrices"]):
        X, y = a[:, 1:], a[:, 0]
        assert list(X.shape) == m["shape"] and not m["kwargs"]
        assert hashlib.sha256(np.ascontiguousarray(X, np.float32).tobytes() + np.ascontiguousarray(y, np.float32).tobytes()).hexdigest() == m["sha256"]
        mats.append(dxgb.DaskDMatrix(None, X, y))
    call = rec["train"]
    assert call["callbacks"] == ["sagemaker_xgboost_container_b200.EvaluationMonitor"] and call["verbose_eval"] == "default"
    params = dict(call["params"])
    if call["has_custom_metric"]:                # the container's metric function stands for the eval_metric it was built from
        params["eval_metric"] = rec["hyperparameters"]["eval_metric"]
    with pytest.warns(UserWarning) as caught:
        out = dxgb.train(None, params, mats[call["dtrain"]], num_boost_round=call["num_boost_round"],
                         evals=[(mats[i], n) for i, n in call["evals"]], callbacks=[xgb.callback.EvaluationMonitor()])
    assert [str(w.message) for w in caught if issubclass(w.category, UserWarning)] == rec["warnings"]
    assert "multi_gpu.run_training_with_dask" in rec["warnings"][0]
    lines = [l for l in capfd.readouterr().out.splitlines() if l.startswith("[")]
    assert lines == rec["eval_lines"] and len(lines) == 10
    got = ubjson.model_from_xgb_json(ubjson.loads(bytes(out["booster"].save_raw("ubj"))))
    g = np.load(os.path.join(os.path.dirname(G), "container", "entrypoint_models.npz"))
    ref = {k.split("/")[-1]: g[k] for k in g.files if k.startswith("dask_route_unbound/0/")}
    assert_same_structure(got, ref)
    assert max_leaf_diff(got, ref) <= 1e-5
    assert out["booster"].num_boosted_rounds() == 5 and out["booster"].num_features() == 8


def _boom():
    raise RuntimeError("engine refused to start")


def test_worker_failures_reach_the_caller(tmp_path):
    from sagemaker_xgboost_container_b200 import multi_gpu
    tr, _ = _channels(tmp_path)
    with pytest.raises(Exception, match="engine refused to start"):
        multi_gpu.run_training_with_dask({"num_round": 2}, str(tr), None, str(tmp_path / "m"), "csv", ["algo-1"], "algo-1", None, 2, worker_init=_boom)


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
def test_two_gpu_launcher_equals_single_gpu(xgb, tmp_path):
    if _ngpu() < 2:
        pytest.skip("needs 2 GPUs")
    from sagemaker_xgboost_container_b200 import multi_gpu
    rng = np.random.default_rng(11)
    n, F = 60000, 12
    X = (np.round(np.clip(rng.standard_normal((n, F)), -4, 4 - 1 / 32) * 32) / 32).astype(np.float32)
    y = (X @ (rng.standard_normal(F) / np.sqrt(F)) + 0.1 * rng.standard_normal(n)).astype(np.float32)
    tr = tmp_path / "train"
    tr.mkdir()
    for i, (a, b) in enumerate([(0, 25000), (25000, n)]):
        np.savetxt(tr / ("part-%d.csv" % i), np.column_stack([y[a:b], X[a:b]]), delimiter=",", fmt="%.9g")
    hp = {"objective": "reg:squarederror", "tree_method": "hist", "num_round": 6, "max_depth": 5, "eta": 0.3, "eval_metric": ["rmse"]}
    multi_gpu.run_training_with_dask(dict(hp), str(tr), None, str(tmp_path / "m2"), "csv", ["algo-1"], "algo-1", None, 2, worker_init=oracle_worker_init.bind_package)
    multi = xgb.Booster(model_file=str(tmp_path / "m2" / "xgboost-model"))
    d = xgb.DMatrix(str(tr) + "?format=csv&label_column=0&delimiter=,")
    single = xgb.train({k: v for k, v in hp.items() if k != "num_round"}, d, num_boost_round=6, verbose_eval=False)
    be = xgb.get_backend()
    m1, m2 = be.booster_export_model(single.handle), be.booster_export_model(multi.handle)
    for k in ("left", "right", "split_index", "split_cond"):
        np.testing.assert_array_equal(m1[k], m2[k])


def test_two_hosts_with_one_gpu_each_rendezvous_through_the_master_tracker(tmp_path):
    """Several hosts (train.py:236-269 analogue for the GPU route): every host calls run_training_with_dask with the same host
    list; the first host runs the tracker on the fixed port, ranks follow (host, gpu), rank 0 alone writes the model.  Two
    'hosts' on this machine (two names of the loopback interface), CPU test engine."""
    import threading
    from sagemaker_xgboost_container_b200 import multi_gpu
    tr, va = _channels(tmp_path)
    hosts = ["localhost", "127.0.0.1"]
    hp = {"objective": "reg:squarederror", "tree_method": "hist", "num_round": 4, "max_depth": 3, "eta": 0.3}
    dirs = [tmp_path / "model-host0", tmp_path / "model-host1"]
    errors = []

    def host(i):
        try:
            multi_gpu.run_training_with_dask(dict(hp), str(tr), str(va), str(dirs[i]), "csv", hosts, hosts[i], None, 1,
                                             worker_init=oracle_worker_init.use_oracle_engine)
        except BaseException as e:      # noqa: BLE001
            errors.append((i, e))
    threads = [threading.Thread(target=host, args=(i,)) for i in (1, 0)]          # the non-master host may well come up first
    for t in threads:
        t.start()
    for t in threads:
        t.join(300)
    assert not errors, errors
    assert os.path.exists(dirs[0] / "xgboost-model") and not os.path.exists(dirs[1])      # the master (rank 0 lives on host 0) saves, nobody else
    # same model as one process on all rows
    import sagemaker_xgboost_container_b200 as xgb
    from sagemaker_xgboost_container_b200 import backend
    from oracle.engine import OracleBackend
    from oracle import ubjson
    old = backend._BACKEND
    backend._BACKEND = OracleBackend(error_cls=xgb.XGBoostError)
    try:
        arr = np.concatenate([np.loadtxt(f, delimiter=",", dtype=np.float32) for f in sorted(str(p) for p in tr.iterdir())])
        single = xgb.train({k: v for k, v in hp.items() if k != "num_round"}, xgb.DMatrix(arr[:, 1:], label=arr[:, 0]), num_boost_round=4, verbose_eval=False)
        a = ubjson.model_from_xgb_json(ubjson.loads(bytes(single.save_raw("ubj"))))
    finally:
        backend._BACKEND = old
    b = ubjson.model_from_xgb_json(ubjson.load(str(dirs[0] / "xgboost-model")))
    for k in ("left", "split_index", "split_cond"):
        np.testing.assert_array_equal(a[k], b[k])


def test_memory_mapped_shards_equal_the_whole_file_split(tmp_path, monkeypatch):
    """_csv_shard_text never loads the channel: it maps the files and scans them in chunks.  Against the obvious whole-file
    implementation on random channels: several files, CRLF and LF endings, leading / trailing blank lines, empty files, scan
    chunks far smaller than a line run."""
    from sagemaker_xgboost_container_b200 import multi_gpu as mg

    def whole_file(files, rank, world):
        chunks = [b for b in (open(f, "rb").read().replace(b"\r\n", b"\n").strip(b"\n") for f in files) if b]
        buf = np.frombuffer(b"\n".join(chunks), np.uint8)
        ends = np.flatnonzero(buf == 10)
        n = len(ends) + (1 if len(buf) else 0)
        lo, hi = mg.shard_bounds(n, rank, world)
        if hi <= lo:
            return b"", n
        return buf[(0 if lo == 0 else int(ends[lo - 1]) + 1):(len(buf) if hi == n else int(ends[hi - 1]))].tobytes(), n
    monkeypatch.setattr(mg, "_SCAN_CHUNK", 37)
    rng = np.random.default_rng(0)
    for trial in range(120):
        files = []
        for k in range(int(rng.integers(1, 5))):
            eol = b"\r\n" if rng.random() < 0.3 else b"\n"
            body = eol.join(b",".join(b"%d" % int(x) for x in rng.integers(0, 1000, int(rng.integers(1, 6)))) for _ in range(int(rng.integers(0, 12))))
            p = tmp_path / ("t%d_%d.csv" % (trial, k))
            p.write_bytes(b"\n" * int(rng.integers(0, 3)) + body + eol * int(rng.integers(0, 3)))
            files.append(str(p))
        for world in (1, 2, 3, 7):
            for r in range(world):
                assert mg._csv_shard_text(files, r, world) == whole_file(files, r, world)


def test_the_references_own_validation_tests_pass_on_the_native_module():
    """validate_gpu_train_configuration and its four message constants against what the container's distributed_gpu_training returned
    on every combination of tree method, hosts, GPUs, input mode, content type and channel distribution
    (tests/golden/container/launcher_validation.json)."""
    from sagemaker_xgboost_container_b200 import multi_gpu
    rec = json.load(open(os.path.join(os.path.dirname(G), "container", "launcher_validation.json")))
    msgs = [getattr(multi_gpu, name) for name in rec["messages"]]
    assert len(set(msgs)) == 4
    cases = next(v for k, v in rec.items() if k.startswith("cases"))
    assert len(cases) == 384
    for tm, hosts, gpus, mode, fmt, dc, expect in cases:
        assert multi_gpu.validate_gpu_train_configuration(tm, hosts, gpus, mode, fmt, rec["data_configs"][dc]) == [msgs[i] for i in expect], (tm, hosts, gpus, mode, fmt, dc)
