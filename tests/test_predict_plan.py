"""The predictor's launch plan (XGB200PredictPlan, host code: no GPU needed) over data widths, model widths and tree sizes.

The tiled kernel stages a chunk of trees (8 B per node, plus one int offset per tree) and a tile of rows (`pitch` floats each)
in one block's dynamic shared memory, walks children as `left`, `left + 1` through a 16-bit child index and a 15-bit feature
field, and gives each thread one row of the tile.  Whatever the plan hands it must respect all of that; anything else must
take the thread-per-row kernel."""
import numpy as np
import pytest

SMEM = 220 * 1024                 # dynamic shared memory of the tiled predictor
NODE_CAP = 96 * 1024              # at most this many bytes of packed nodes per chunk
WIDTHS = list(range(1, 1301)) + [32767, 32768, 40000]
TREE_COUNTS = [1, 63, 64, 95, 96, 97, 1000]


@pytest.fixture(scope="module")
def be():
    import __graft_entry__
    from sagemaker_xgboost_container_b200.backend import LIB_PATH, CudaBackend
    import os
    if not os.path.exists(LIB_PATH):
        __graft_entry__.build()
    return CudaBackend()


def trained_slots(depth):
    """Device slot of a depthwise tree this engine trains: 2^(depth+1) - 1 nodes rounded up to 16."""
    return ((1 << (depth + 1)) - 1 + 15) & ~15


def lossguide_slots(max_leaves):
    return (2 * max_leaves - 1 + 15) & ~15


def offsets_bytes(ntrees):
    return ((ntrees + 1) * 4 + 15) & ~15


def check(plan, F, F_model, counts, tree_begin=0, adjacent=True):
    """Every invariant the kernels rely on; returns the plan's route."""
    counts = [int(c) for c in counts]
    width = max(F, F_model)
    pitch = width | 1
    assert plan["smem_limit"] == SMEM
    assert plan["absent_features"] == (F < F_model)
    if plan["route"] == "thread_per_row":
        assert plan["kernel"] == "predict_kernel" and plan["chunks"] == []
        # the tiled kernel was refused for a reason: a feature index it cannot pack, sibling order, or a tree that cannot
        # share the block with a 32-row tile
        fits_alone = all(c <= 65534 and 8 * c <= NODE_CAP and offsets_bytes(1) + 8 * c + 32 * pitch * 4 <= SMEM for c in counts)
        assert not (adjacent and width <= 32767 and pitch * 4 * 32 + 64 * 1024 <= SMEM and fits_alone), \
            "thread-per-row route although every tree fits a tile next to 32 rows"
        return "thread_per_row"
    assert plan["route"] == "tiled" and plan["kernel"] == "predict_tiled_kernel"
    assert adjacent, "the tiled kernel assumes right == left + 1"
    assert width <= 32767, "the tiled kernel packs the feature index into 15 bits"
    assert plan["pitch"] == pitch, "rows must be staged at the wider of the data and the model"
    assert plan["node_budget"] <= NODE_CAP
    chunks = plan["chunks"]
    assert chunks and chunks[0]["tree_lo"] == tree_begin and chunks[-1]["tree_hi"] == tree_begin + len(counts)
    for a, b in zip(chunks, chunks[1:]):
        assert a["tree_hi"] == b["tree_lo"], "chunks must partition the trees in order"
    for i, c in enumerate(chunks):
        lo, hi = c["tree_lo"] - tree_begin, c["tree_hi"] - tree_begin
        assert hi > lo
        nodes = counts[lo:hi]
        assert max(nodes) <= 65534, "the packed node keeps a 16-bit child index"
        node_bytes = 8 * sum(nodes)
        assert node_bytes <= plan["node_budget"]
        head = offsets_bytes(hi - lo) + node_bytes
        assert c["head"] == head
        rows, threads = c["rows"], c["threads"]
        assert threads in (256, 512, 1024)
        assert 32 <= rows <= threads and rows % 32 == 0, (i, c)
        assert c["smem"] == head + rows * pitch * 4
        assert c["smem"] <= SMEM, (i, c)
        if i + 1 < len(chunks):         # greedy: the next tree did not fit this chunk
            nxt = counts[hi]
            assert (node_bytes + 8 * nxt > NODE_CAP or
                    offsets_bytes(hi - lo + 1) + node_bytes + 8 * nxt + 32 * pitch * 4 > SMEM), "chunk %d ends early" % i
    return "tiled"


def plan_of(be, F, F_model, counts, tree_begin=0, adjacent=True):
    plan = be.predict_plan(F, F_model, counts, tree_begin, adjacent)
    return plan, check(plan, F, F_model, counts, tree_begin, adjacent)


# the shapes of the zero-row tile plan: (F, model) -> the route after the fix is tiled, 32-row tiles at most
TABLE = {
    "f1000_100_rounds_depth6": (1000, [trained_slots(6)] * 100),
    "f990_100_rounds_depth6": (990, [trained_slots(6)] * 100),
    "f1247_64_rounds_depth6": (1247, [trained_slots(6)] * 64),
    "f1200_30_rounds_depth8": (1200, [trained_slots(8)] * 30),
    "f980_100_rounds_depth6": (980, [trained_slots(6)] * 100),
}


@pytest.mark.parametrize("name", sorted(TABLE))
def test_table_shapes_get_a_tile_of_at_least_32_rows(be, name):
    F, counts = TABLE[name]
    plan, route = plan_of(be, F, F, counts)
    assert route == "tiled"
    if name == "f980_100_rounds_depth6":       # this one always fitted: its plan is unchanged
        assert (plan["chunks"][0]["tree_hi"], plan["chunks"][0]["head"], plan["chunks"][0]["rows"]) == (96, 98704, 32)


def test_baseline_config5_plan_is_one_chunk_of_1024_rows(be):
    """1M x 28 rows, 50 depth-6 rounds (bench.py predict section): one launch, full 1024-row tiles."""
    plan, route = plan_of(be, 28, 28, [trained_slots(6)] * 50)
    assert route == "tiled" and len(plan["chunks"]) == 1
    c = plan["chunks"][0]
    assert (c["rows"], c["threads"], plan["pitch"], plan["node_budget"]) == (1024, 1024, 29, NODE_CAP)


@pytest.mark.parametrize("F_model_of", [lambda F: F, lambda F: F + 1, lambda F: 2 * F + 3], ids=["same", "plus1", "double"])
def test_every_width(be, F_model_of):
    rng = np.random.default_rng(7)
    mixed = rng.choice([trained_slots(d) for d in range(1, 11)], size=97)
    for F in WIDTHS:
        Fm = F_model_of(F)
        for counts in ([trained_slots(6)] * 100, [trained_slots(8)] * 30, mixed):
            plan, route = plan_of(be, F, Fm, counts)
            if max(F, Fm) <= 1247 and max(counts) <= trained_slots(8):
                assert route == "tiled", (F, Fm)
            if max(F, Fm) > 32767:
                assert route == "thread_per_row"


@pytest.mark.parametrize("ntrees", TREE_COUNTS)
@pytest.mark.parametrize("depth", range(1, 15))
def test_trained_slot_sizes(be, depth, ntrees):
    counts = [trained_slots(depth)] * ntrees
    for F in (1, 28, 127, 500, 980, 990, 1000, 1200, 1247, 1248, 1300, 32767, 32768, 40000):
        for Fm in (F, F + 7):
            plan, route = plan_of(be, F, Fm, counts, tree_begin=3)
            if depth >= 13:            # 16384+ node slots: over the 96 KiB chunk budget
                assert route == "thread_per_row"


@pytest.mark.parametrize("max_leaves,tiled_at_small_F", [(2, True), (255, True), (6000, True), (6144, True), (6145, False), (6200, False)])
def test_lossguide_slot_sizes(be, max_leaves, tiled_at_small_F):
    """max_leaves 6000 -> 12000 node slots, just inside the budget (12288 nodes); 6200 -> 12400, just over it."""
    slots = lossguide_slots(max_leaves)
    for ntrees in TREE_COUNTS:
        for F in (1, 28, 100, 500, 1000, 1247):
            plan, route = plan_of(be, F, F, [slots] * ntrees)
            if F <= 28:
                assert (route == "tiled") == tiled_at_small_F, (max_leaves, ntrees, F)


def test_foreign_exact_sizes_and_random_mixes(be):
    """Loaded models keep their exact node counts (2 * leaves - 1): any odd number, mixed with trained slots."""
    rng = np.random.default_rng(11)
    for trial in range(60):
        ntrees = int(rng.choice(TREE_COUNTS))
        kind = trial % 3
        if kind == 0:
            counts = 2 * rng.integers(1, 512, size=ntrees) - 1
        elif kind == 1:
            counts = 2 * rng.integers(1, 7000, size=ntrees) - 1
        else:
            counts = np.where(rng.random(ntrees) < 0.5, 2 * rng.integers(1, 200, size=ntrees) - 1,
                              rng.choice([trained_slots(d) for d in range(1, 15)], size=ntrees))
        for F in (1, 50, 700, 1100, 1247, 1248):
            plan_of(be, F, F + int(rng.integers(0, 3)), counts, tree_begin=int(rng.integers(0, 5)))


def test_trees_the_tiled_kernel_cannot_hold(be):
    plan, route = plan_of(be, 28, 28, [trained_slots(6)] * 10 + [70000] + [trained_slots(6)] * 10)
    assert route == "thread_per_row"                                   # over the 16-bit child index
    plan, route = plan_of(be, 28, 28, [lossguide_slots(6200)])
    assert route == "thread_per_row"                                   # over the node budget on its own
    plan, route = plan_of(be, 28, 28, [lossguide_slots(6000)] * 3)
    assert route == "tiled" and [c["tree_hi"] - c["tree_lo"] for c in plan["chunks"]] == [1, 1, 1]


@pytest.mark.parametrize("F", [1, 28, 1000, 32767])
def test_models_wider_than_the_15_bit_feature_field(be, F):
    """A model with features >= 32768 never takes the tiled route, however narrow the request."""
    plan, route = plan_of(be, F, 40001, [trained_slots(3)] * 5)
    assert route == "thread_per_row" and plan["absent_features"]
    plan, route = plan_of(be, F, 32768, [trained_slots(3)] * 5)
    assert route == "thread_per_row"


@pytest.mark.parametrize("F", [1, 28, 1000])
def test_children_not_adjacent_takes_the_thread_per_row_route(be, F):
    plan, route = plan_of(be, F, F, [trained_slots(6)] * 20, adjacent=False)
    assert route == "thread_per_row"


def test_narrow_requests_stage_at_the_model_width(be):
    plan, route = plan_of(be, 13, 28, [trained_slots(6)] * 50)
    assert route == "tiled" and plan["pitch"] == 29 and plan["absent_features"]
    plan, route = plan_of(be, 40, 28, [trained_slots(6)] * 50)       # wider matrices keep their own width
    assert route == "tiled" and plan["pitch"] == 41 and not plan["absent_features"]
    plan, route = plan_of(be, 1000, 1247, [trained_slots(6)] * 64)   # the tile is sized for the model's width
    assert route == "tiled" and plan["pitch"] == 1247
