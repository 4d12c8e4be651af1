"""The predictor on its own, every launch route against the oracle walking the same model.

Each case first asks XGB200BoosterPredictPlan which kernel a predict call will run, then compares: leaf indices bit-exact,
raw margins bit-exact from the same per-row base margin (both sides add fp32 leaf values in tree order), transformed outputs
within the tolerances of test_gpu_parity.py.  Models are trained (device slot-padded trees) or built synthetically by replacing
the trees of a trained booster's JSON document, which controls depth, node counts, split features and default directions."""
import json

import numpy as np
import pytest

from util import synth

pytestmark = pytest.mark.gpu

RTOL, ATOL = 2e-6, 1e-6            # transformed outputs (test_gpu_parity.py)


def _be():
    from sagemaker_xgboost_container_b200.backend import get_backend
    return get_backend()


# ---------------------------------------------------------------------------------------------------------------- models
def _trained(xgb, params, X, y, rounds):
    """The booster as the trainer leaves it: each tree sits in a fixed-capacity device slot (2^(depth+1) - 1 nodes rounded up
    to 16).  xgb.train returns a copy made through the model document, whose trees are uploaded at their exact node counts."""
    d = xgb.DMatrix(X, label=y)
    bst = xgb.Booster(params, [d])
    for i in range(rounds):
        bst.update(d, i)
    m = _be().booster_export_model(bst.handle)
    m["objective"] = params["objective"]
    return bst, m


def _random_tree(rng, F_model, depth, split_prob=1.0, force_feature=None):
    """BFS-numbered tree (children adjacent, after their parent) of at most `depth` levels; thresholds on the synth() grid."""
    left, right, feat, cond, dl = [], [], [], [], []
    level = [0]
    left.append(-1); right.append(-1); feat.append(0); cond.append(0.0); dl.append(0)
    for d in range(depth):
        nxt = []
        for nid in level:
            if d > 0 and rng.random() >= split_prob:
                continue
            f = int(rng.integers(0, F_model))
            if force_feature is not None and rng.random() < 0.3:
                f = force_feature
            feat[nid] = f
            cond[nid] = float(np.float32(rng.integers(-48, 48) / 32))
            dl[nid] = int(rng.integers(0, 2))
            l = len(left)
            for _ in range(2):
                left.append(-1); right.append(-1); feat.append(0); cond.append(0.0); dl.append(0)
            left[nid], right[nid] = l, l + 1
            nxt += [l, l + 1]
        level = nxt
    for i in range(len(left)):
        if left[i] == -1:
            cond[i] = float(np.float32(rng.standard_normal() * 0.25))
    return {"left": left, "right": right, "split_index": feat, "split_cond": cond, "default_left": dl}


def _tree_with_leaves(rng, F_model, leaves):
    """A lossguide-shaped tree: expand random leaves until it has `leaves` of them (2 * leaves - 1 nodes)."""
    left, right, feat, cond, dl = [-1], [-1], [0], [0.0], [0]
    open_ = [0]
    while len(open_) < leaves:
        nid = open_.pop(int(rng.integers(0, len(open_))))
        feat[nid] = int(rng.integers(0, F_model)); cond[nid] = float(np.float32(rng.integers(-48, 48) / 32)); dl[nid] = int(rng.integers(0, 2))
        l = len(left)
        for _ in range(2):
            left.append(-1); right.append(-1); feat.append(0); cond.append(0.0); dl.append(0)
        left[nid], right[nid] = l, l + 1
        open_ += [l, l + 1]
    for i in range(len(left)):
        if left[i] == -1:
            cond[i] = float(np.float32(rng.standard_normal() * 0.25))
    return {"left": left, "right": right, "split_index": feat, "split_cond": cond, "default_left": dl}


def _preorder(tree):
    """Renumber depth-first (node, left subtree, right subtree): children still follow their parent, but are not adjacent."""
    order, stack = [], [0]
    while stack:
        i = stack.pop()
        order.append(i)
        if tree["left"][i] != -1:
            stack += [tree["right"][i], tree["left"][i]]
    new = {old: k for k, old in enumerate(order)}
    out = {k: [None] * len(order) for k in tree}
    for old, k in new.items():
        for key in ("split_index", "split_cond", "default_left"):
            out[key][k] = tree[key][old]
        out["left"][k] = new[tree["left"][old]] if tree["left"][old] != -1 else -1
        out["right"][k] = new[tree["right"][old]] if tree["right"][old] != -1 else -1
    return out


_BASE_DOCS = {}


def _base_doc(xgb, objective, K):
    """JSON document of a small trained booster with this objective: the frame the synthetic trees go into."""
    key = (objective, K)
    if key not in _BASE_DOCS:
        X, y = synth(300, 4, 1, "multi" if K > 1 else ("bin" if objective.startswith("binary") else "reg"), K=K)
        params = {"objective": objective, "max_depth": 2}
        if K > 1:
            params["num_class"] = K
        bst = xgb.train(params, xgb.DMatrix(X, label=y), num_boost_round=1, verbose_eval=False)
        _BASE_DOCS[key] = json.loads(bytes(bst.save_raw("json")).decode())
    return json.loads(json.dumps(_BASE_DOCS[key]))


def _synthetic(xgb, trees, F_model, objective="binary:logistic", K=1):
    """(Booster, oracle model) of a document holding exactly `trees` (tree t belongs to class t % K)."""
    from oracle import ubjson
    doc = _base_doc(xgb, objective, K)
    doc["learner"]["learner_model_param"]["num_feature"] = str(F_model)
    gb = doc["learner"]["gradient_booster"]["model"]
    jt = []
    for t, tr in enumerate(trees):
        nn = len(tr["left"])
        parents = [-1] * nn
        for i in range(nn):
            if tr["left"][i] != -1:
                parents[tr["left"][i]] = i; parents[tr["right"][i]] = i
        jt.append({"base_weights": list(tr["split_cond"]), "categories": [], "categories_nodes": [], "categories_segments": [],
                   "categories_sizes": [], "default_left": list(tr["default_left"]), "id": t, "left_children": list(tr["left"]),
                   "loss_changes": [0.0] * nn, "parents": parents, "right_children": list(tr["right"]),
                   "split_conditions": list(tr["split_cond"]), "split_indices": list(tr["split_index"]), "split_type": [0] * nn,
                   "sum_hessian": [1.0] * nn,
                   "tree_param": {"num_deleted": "0", "num_feature": str(F_model), "num_nodes": str(nn), "size_leaf_vector": "1"}})
    gb["trees"] = jt
    gb["tree_info"] = [t % K for t in range(len(trees))]
    gb["iteration_indptr"] = list(range(0, len(trees) + 1, K))
    gb["gbtree_model_param"]["num_trees"] = str(len(trees))
    bst = xgb.Booster(model_file=bytearray(json.dumps(doc).encode()))
    return bst, ubjson.model_from_xgb_json(doc)


# ----------------------------------------------------------------------------------------------------------- checking
def _plan(xgb, bst, X, iteration_range=(0, 0)):
    d = xgb.DMatrix(X)
    return _be().booster_predict_plan(bst.handle, d.handle, iteration_range)


def _assert_route(xgb, bst, X, route, iteration_range=(0, 0), absent=None):
    plan = _plan(xgb, bst, X, iteration_range)
    assert plan["route"] == route, plan["route"]
    assert plan["kernel"] == ("predict_tiled_kernel" if route == "tiled" else "predict_kernel")
    if absent is not None:
        assert plan["absent_features"] == absent
    return plan


def _check(xgb, oracle, bst, model, X, iteration_range=(0, 0), X_ref=None, seed=0):
    """pred_leaf and output_margin bit-exact, transformed output within tolerance, for the request X (the oracle reads X_ref,
    default X: it treats columns past the matrix as missing, like the product must)."""
    X_ref = X if X_ref is None else X_ref
    n = len(X)
    K = int(model["num_class"])
    rounds = len(model["tree_info"]) // K
    ib, ie = iteration_range
    ie = ie or rounds
    tb, te = ib * K, ie * K
    d = xgb.DMatrix(X)
    leaf = bst.predict(d, pred_leaf=True, iteration_range=iteration_range, validate_features=False)
    np.testing.assert_array_equal(leaf.astype(np.int32).reshape(n, te - tb), oracle.predict_leaf(model, X_ref, tb, te))
    bm = np.random.default_rng(seed).standard_normal((n, K)).astype(np.float32)
    db = xgb.DMatrix(X, base_margin=bm.ravel())
    margin = bst.predict(db, output_margin=True, iteration_range=iteration_range, validate_features=False).reshape(n, K)
    ref = oracle.predict_margin(model, X_ref, tb, te, base_margin=bm)
    if not np.array_equal(margin, ref):
        pytest.fail("output_margin is not bit-exact: max |diff| = %.3g over %d of %d values"
                    % (float(np.abs(margin - ref).max()), int((margin != ref).sum()), margin.size))
    pred = bst.predict(d, iteration_range=iteration_range, validate_features=False).reshape(n, -1)
    np.testing.assert_allclose(pred, oracle.transform(model, oracle.predict_margin(model, X_ref, tb, te)).reshape(n, -1), rtol=RTOL, atol=ATOL)


def _check_narrow(xgb, oracle, bst, model, X, route, widths=None):
    """The request lacks the model's last columns (container CSV rule: one fewer; libsvm bodies: any width): those features
    are missing, so the default direction is taken -- X has no NaN, the oracle reads the NaN-padded matrix."""
    Fm = X.shape[1]
    for w in widths or (Fm - 1, max(1, Fm // 2)):
        Xn = np.ascontiguousarray(X[:, :w])
        _assert_route(xgb, bst, Xn, route, absent=True)
        padded = X.copy()
        padded[:, w:] = np.nan
        _check(xgb, oracle, bst, model, Xn, X_ref=padded, seed=w)


def _check_wide(xgb, oracle, bst, model, X, route):
    """Extra columns past the model's width never change the output, whatever they hold."""
    n, Fm = X.shape
    junk = np.random.default_rng(3).standard_normal((n, 9)).astype(np.float32) * 1e30
    junk[:, 0] = np.nan
    junk[:, 1] = np.inf
    Xw = np.ascontiguousarray(np.hstack([X, junk]))
    _assert_route(xgb, bst, Xw, route, absent=False)
    for kw in ({"pred_leaf": True}, {"output_margin": True}, {}):
        np.testing.assert_array_equal(bst.predict(xgb.DMatrix(Xw), validate_features=False, **kw), bst.predict(xgb.DMatrix(X), **kw))
    _check(xgb, oracle, bst, model, Xw, X_ref=X)


# ----------------------------------------------------------------------------------------------------------------- cases
@pytest.mark.parametrize("nan", [False, True], ids=["no_nan", "nan"])
@pytest.mark.parametrize("objective,K", [("binary:logistic", 1), ("multi:softprob", 4)])
def test_tiled_variants(xgb, oracle, objective, K, nan):
    """All four tiled kernels {NaN-aware, not} x {margin, leaf}, with one and with four classes; narrow and wide requests."""
    X, y = synth(20000, 28, 31, "multi" if K > 1 else "bin", K=K, missing_frac=0.1 if nan else 0.0)
    params = {"objective": objective, "max_depth": 6, "eta": 0.3}
    if K > 1:
        params["num_class"] = K
    bst, m = _trained(xgb, params, X, y, 8)
    plan = _assert_route(xgb, bst, X, "tiled", absent=False)
    assert len(plan["chunks"]) == 1 and plan["chunks"][0]["rows"] == 1024
    _check(xgb, oracle, bst, m, X)
    if not nan:
        _check_narrow(xgb, oracle, bst, m, X, "tiled")
        _check_wide(xgb, oracle, bst, m, X, "tiled")


def test_multi_chunk_trained(xgb, oracle):
    """330 trained depth-6 trees (128-node slots): four chunks; ranges that start and end inside a chunk."""
    X, y = synth(6000, 28, 32)
    bst, m = _trained(xgb, {"objective": "reg:squarederror", "max_depth": 6, "eta": 0.05}, X, y, 330)
    plan = _assert_route(xgb, bst, X, "tiled")
    bounds = [c["tree_lo"] for c in plan["chunks"]]
    assert len(bounds) >= 4, bounds
    _check(xgb, oracle, bst, m, X)
    for rng_ in ((bounds[0] + 10, bounds[-1] + 5), (bounds[1] - 1, bounds[2] + 1), (7, 8)):
        _assert_route(xgb, bst, X, "tiled", iteration_range=rng_)
        _check(xgb, oracle, bst, m, X, iteration_range=rng_)
    _check_narrow(xgb, oracle, bst, m, X, "tiled", widths=(27, 5))


def test_multi_chunk_three_classes_boundaries_inside_rounds(xgb, oracle):
    """960 synthetic trees of varied size, K = 3: chunk boundaries fall inside a round; ranges start and end inside chunks."""
    rng = np.random.default_rng(33)
    F = 40
    trees = [_random_tree(rng, F, 6, split_prob=0.85, force_feature=F - 1) for _ in range(960)]
    bst, m = _synthetic(xgb, trees, F, "multi:softprob", 3)
    X, _ = synth(5000, F, 34)
    plan = _assert_route(xgb, bst, X, "tiled")
    lows = [c["tree_lo"] for c in plan["chunks"]]
    assert len(lows) >= 3 and any(lo % 3 for lo in lows), lows
    _check(xgb, oracle, bst, m, X)
    rounds = 320
    for rng_ in ((lows[1] // 3 - 2, lows[2] // 3 + 2), (1, rounds - 1), (lows[-1] // 3, rounds)):
        _check(xgb, oracle, bst, m, X, iteration_range=rng_)
    _check_narrow(xgb, oracle, bst, m, X, "tiled")


@pytest.mark.parametrize("F", [28, 600])
def test_row_counts_around_the_tile(xgb, oracle, F):
    """n = 1, rows_per_tile - 1, + 0, + 1 and a ragged last tile, for 1024-row tiles (F = 28) and 64-row tiles (F = 600)."""
    rng = np.random.default_rng(35 + F)
    trees = [_random_tree(rng, F, 6, split_prob=0.9, force_feature=F - 1) for _ in range(40)]
    bst, m = _synthetic(xgb, trees, F)
    X, _ = synth(8 * 1024 + 77, F, 36)
    plan = _assert_route(xgb, bst, X, "tiled")
    rows = plan["chunks"][0]["rows"]
    assert rows == (1024 if F == 28 else 64), plan
    for n in (1, rows - 1, rows, rows + 1, 5 * rows + 17, len(X)):
        _check(xgb, oracle, bst, m, X[:n], seed=n)
    _check_narrow(xgb, oracle, bst, m, X[: 3 * rows + 5], "tiled")


@pytest.mark.parametrize("F,rounds,depth", [(1000, 100, 6), (1247, 64, 6)])
def test_wide_tables_trained(xgb, oracle, F, rounds, depth):
    """Shapes whose tree chunk left no room for a 32-row tile (zero rows per tile, a division by zero on the host)."""
    X, y = synth(3000, F, 37)
    y = (y + X[:, -1]).astype(np.float32)                     # so the last feature is split on
    bst, m = _trained(xgb, {"objective": "reg:squarederror", "max_depth": depth, "eta": 0.1, "min_child_weight": 0.1}, X, y, rounds)
    plan = _assert_route(xgb, bst, X, "tiled")
    assert all(c["rows"] >= 32 for c in plan["chunks"]) and len(plan["chunks"]) >= 2
    _check(xgb, oracle, bst, m, X)
    _check(xgb, oracle, bst.copy(), m, X)                    # the same trees at their exact node counts
    _check_narrow(xgb, oracle, bst, m, X, "tiled")
    _check_wide(xgb, oracle, bst, m, X[:500], "tiled" if F + 9 <= 1247 else "thread_per_row")   # 9 extra columns


@pytest.mark.parametrize("F,rounds,depth", [(1000, 100, 6), (990, 100, 6), (1247, 64, 6), (1200, 30, 8)])
def test_wide_tables_loaded(xgb, oracle, F, rounds, depth):
    rng = np.random.default_rng(38 + F)
    trees = [_random_tree(rng, F, depth, force_feature=F - 1) for _ in range(rounds)]
    bst, m = _synthetic(xgb, trees, F)
    X, _ = synth(2500, F, 39)
    plan = _assert_route(xgb, bst, X, "tiled")
    assert all(c["rows"] >= 32 for c in plan["chunks"])
    _check(xgb, oracle, bst, m, X)
    _check_narrow(xgb, oracle, bst, m, X, "tiled")


def test_thread_per_row_wide_data(xgb, oracle):
    """F >= 1248: a 32-row tile and a node chunk no longer fit together."""
    rng = np.random.default_rng(40)
    F = 1300
    trees = [_random_tree(rng, F, 6, force_feature=F - 1) for _ in range(20)]
    bst, m = _synthetic(xgb, trees, F)
    X, _ = synth(3000, F, 41)
    _assert_route(xgb, bst, X, "thread_per_row")
    _check(xgb, oracle, bst, m, X)
    _check_narrow(xgb, oracle, bst, m, X, "thread_per_row", widths=(F - 1, 1000))     # 1000 wide, the model still is not
    _check_wide(xgb, oracle, bst, m, X[:500], "thread_per_row")


def test_thread_per_row_tree_over_the_node_budget_trained(xgb, oracle):
    """max_depth 13: 16384-node slots, over the 12288 nodes a chunk holds."""
    X, y = synth(30000, 20, 42)
    y = (y + X[:, -1]).astype(np.float32)
    bst, m = _trained(xgb, {"objective": "reg:squarederror", "max_depth": 13, "min_child_weight": 0.1}, X, y, 2)
    _assert_route(xgb, bst, X, "thread_per_row")
    _check(xgb, oracle, bst, m, X)
    _check_narrow(xgb, oracle, bst, m, X, "thread_per_row")
    _check_wide(xgb, oracle, bst, m, X[:2000], "thread_per_row")
    _check(xgb, oracle, bst.copy(), m, X)


def test_thread_per_row_lossguide_sized_tree_loaded(xgb, oracle):
    """A 6200-leaf tree (12399 nodes) among small ones; 6000 leaves (11999 nodes) still fit a chunk."""
    rng = np.random.default_rng(43)
    F = 30
    small = [_random_tree(rng, F, 4, force_feature=F - 1) for _ in range(5)]
    bst, m = _synthetic(xgb, small + [_tree_with_leaves(rng, F, 6200)] + small, F)
    X, _ = synth(20000, F, 44)
    _assert_route(xgb, bst, X, "thread_per_row")
    _check(xgb, oracle, bst, m, X)
    _check_narrow(xgb, oracle, bst, m, X, "thread_per_row")
    bst2, m2 = _synthetic(xgb, small + [_tree_with_leaves(rng, F, 6000)] + small, F)
    _assert_route(xgb, bst2, X, "tiled")
    _check(xgb, oracle, bst2, m2, X)
    _check_narrow(xgb, oracle, bst2, m2, X, "tiled")


def test_thread_per_row_children_not_adjacent(xgb, oracle):
    """A foreign model numbered depth-first: children after their parent but not side by side."""
    rng = np.random.default_rng(45)
    F = 28
    trees = [_preorder(_random_tree(rng, F, 6, split_prob=0.9, force_feature=F - 1)) for _ in range(30)]
    assert any(t["right"][0] != t["left"][0] + 1 for t in trees)
    bst, m = _synthetic(xgb, trees, F, "multi:softprob", 3)
    X, _ = synth(20000, F, 46)
    _assert_route(xgb, bst, X, "thread_per_row")
    _check(xgb, oracle, bst, m, X)
    _check_narrow(xgb, oracle, bst, m, X, "thread_per_row")
    _check_wide(xgb, oracle, bst, m, X[:2000], "thread_per_row")


def test_model_wider_than_32767_features(xgb, oracle):
    """Splits on feature 40000 do not fit the tiled kernel's 15-bit feature field: thread-per-row, narrow or full width."""
    rng = np.random.default_rng(47)
    Fm = 40001
    trees = []
    for _ in range(12):
        t = _random_tree(rng, 60, 5)
        for i in range(len(t["left"])):
            if t["left"][i] != -1 and rng.random() < 0.4:
                t["split_index"][i] = int(rng.choice([40000, 32767, 32768, 39999]))
        trees.append(t)
    bst, m = _synthetic(xgb, trees, Fm)
    Xn, _ = synth(3000, 60, 48)
    _assert_route(xgb, bst, Xn, "thread_per_row", absent=True)
    padded = np.full((len(Xn), Fm), np.nan, np.float32)
    padded[:, :60] = Xn
    _check(xgb, oracle, bst, m, Xn, X_ref=padded)
    Xf, _ = synth(64, Fm, 49)
    _assert_route(xgb, bst, Xf, "thread_per_row", absent=False)
    _check(xgb, oracle, bst, m, Xf)


def test_serving_libsvm_body_narrower_than_the_model(xgb, oracle):
    """A libsvm request body whose rows list only the first features: parsed on the device into a narrow matrix, predicted
    through serving.predict; equals the oracle on the body padded with NaN to the model's width."""
    from sagemaker_xgboost_container_b200 import serving
    F = 28
    X, y = synth(20000, F, 50)
    y = (y + X[:, -1]).astype(np.float32)
    bst, m = _trained(xgb, {"objective": "reg:squarederror", "max_depth": 6}, X, y, 10)
    w = 14
    body = "\n".join("0 " + " ".join("%d:%r" % (j + 1, float(v)) for j, v in enumerate(row[:w])) for row in X[:3000])
    d = serving.sparse_libsvm_to_dmatrix(body)
    assert (d.num_row(), d.num_col()) == (3000, w)
    assert _be().booster_predict_plan(bst.handle, d.handle)["absent_features"]
    got = serving.predict(bst, "xgb_format", d, "text/libsvm")
    padded = np.full((3000, F), np.nan, np.float32)
    padded[:, :w] = X[:3000, :w]
    np.testing.assert_array_equal(got, oracle.predict_margin(m, padded)[:, 0])      # reg:squarederror: identity transform
    # an eval set of that width goes through the trainer's prediction cache, the same launcher
    de = xgb.DMatrix(np.ascontiguousarray(X[:3000, :w]), base_margin=np.zeros(3000, np.float32))
    np.testing.assert_array_equal(_be().booster_cached_margin(bst.handle, de.handle, 1)[:, 0],
                                  oracle.predict_margin(m, padded, base_margin=np.zeros((3000, 1), np.float32))[:, 0])
