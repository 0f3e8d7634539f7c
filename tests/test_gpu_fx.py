"""GPU parity of the lean kernel's FX variant (double sums as fixed-point limbs updated with native 32-bit shared atomics,
csrc/agg_direct.cuh + csrc/fx.h) against the row-engine oracle, through the C ABI: value distributions that exercise the main / fine /
exact classes, special values, group counts on both sides of the shared table's capacity, the fused join probe, and agreement with the CAS variant."""
import numpy as np
import pytest

from baikaldb_b200 import datagen, plan as P, queries
from baikaldb_b200.column import make_column, rows_as_set
from baikaldb_b200.exec_node import execute
from baikaldb_b200.plan import PrimitiveType as T
from tests.util import run_both

pytestmark = pytest.mark.gpu
FX = {"lean_fx": 1}
NAME = "k_agg_group_lean_fx"


def sum_plan(n_sums=2, key_type=T.INT32, with_filter=True, int_sum=False):
    """SELECT k, COUNT(*), SUM(a) [, AVG(b)] [, SUM(c) int64] FROM t [WHERE f < 50] GROUP BY k"""
    aggs = [P.agg_expr("count_star", 1, 1), P.agg_expr("sum", 1, 2, None, P.slot_ref(0, 3, T.DOUBLE))]
    types = [T.INT64, T.DOUBLE]
    slots = [(1, key_type), (2, T.INT32), (3, T.DOUBLE)]
    if n_sums >= 2:
        aggs.append(P.agg_expr("avg", 1, 3, 4, P.slot_ref(0, 4, T.DOUBLE))); types.append(T.DOUBLE); slots.append((4, T.DOUBLE))
    if int_sum:
        aggs.append(P.agg_expr("sum", 1, 5, None, P.slot_ref(0, 5, T.INT64))); types.append(T.INT64); slots.append((5, T.INT64))
    child = P.where(P.scan(0), P.lt(P.slot_ref(0, 2, T.INT32), P.int_lit(50))) if with_filter else P.scan(0)
    root = P.agg(child, 1, [P.slot_ref(0, 1, key_type)], aggs)
    return P.Plan(root, {0: slots, 1: P.agg_tuple_slots(aggs, types)})


def table(rng, n, groups, a, b=None, key_type=T.INT32, c=None):
    cols = [make_column(0, 1, key_type, rng.integers(0, groups, n)), make_column(0, 2, T.INT32, rng.integers(0, 100, n)), make_column(0, 3, T.DOUBLE, a)]
    if b is not None:
        cols.append(make_column(0, 4, T.DOUBLE, b))
    if c is not None:
        cols.append(make_column(0, 5, T.INT64, c))
    return cols


DISTS = {
    "uniform": lambda r, n: r.random(n),
    "normal_1e3": lambda r, n: r.normal(size=n) * 1e3,
    "lognormal_2": lambda r, n: np.exp(r.normal(size=n) * 2.0),
    "lognormal_6": lambda r, n: np.exp(r.normal(size=n) * 6.0) * np.where(r.random(n) < 0.5, -1.0, 1.0),
    "sorted": lambda r, n: np.arange(n, dtype=np.float64) * 1e-3,
    "outliers": lambda r, n: np.where(np.arange(n) % 1000 == 0, 1e12, r.random(n) * 1e-6),
    "integers": lambda r, n: r.integers(-1000, 1001, n).astype(np.float64),
    "zeros_90pct": lambda r, n: np.where(r.random(n) < 0.9, 0.0, r.random(n)),
    "tiny_1e-300": lambda r, n: r.random(n) * 1e-300,
    "huge_1e300": lambda r, n: (r.random(n) - 0.5) * 1e300,
    "denormals": lambda r, n: 5e-324 * r.integers(0, 1000, n),
    "all_zero": lambda r, n: np.zeros(n),
    "minus_zero": lambda r, n: np.full(n, -0.0),
}


@pytest.mark.parametrize("dist", sorted(DISTS))
@pytest.mark.parametrize("n,groups", [(70_001, 37), (400_000, 1000)])
def test_fx_value_distributions(dist, n, groups):
    rng = np.random.default_rng(len(dist) * 1000 + groups)
    cols = table(rng, n, groups, DISTS[dist](rng, n), DISTS["normal_1e3"](rng, n))
    _, stats, _ = run_both(sum_plan(), cols, keys=["0_1"], options=FX, abs_tol=1e-300)
    assert stats.main_kernel_name.decode() == NAME


@pytest.mark.parametrize("n", [1, 3, 4, 5, 127, 128, 129, 1000, 65537, 300_003])
def test_fx_c2_ragged_sizes(n):
    cols = datagen.c2_table(0, n, n_groups=50)
    _, stats, _ = run_both(queries.c2_filter_groupby(), cols, keys=["0_1"], options=FX)
    assert stats.main_kernel_name.decode() == NAME


def test_fx_nan_and_inf_values_take_the_exact_path():
    rng = np.random.default_rng(5)
    n, groups = 120_000, 12
    a = rng.random(n)
    key = rng.integers(0, groups, n)
    a[(key == 1) & (rng.random(n) < 0.01)] = np.nan             # group 1: NaN
    a[(key == 2) & (rng.random(n) < 0.01)] = np.inf             # group 2: +Inf
    a[(key == 3) & (rng.random(n) < 0.01)] = -np.inf            # group 3: -Inf
    m4 = key == 4
    a[m4] = np.where(rng.random(m4.sum()) < 0.5, np.inf, -np.inf)   # group 4: Inf - Inf = NaN
    cols = [make_column(0, 1, T.INT32, key), make_column(0, 2, T.INT32, rng.integers(0, 40, n)), make_column(0, 3, T.DOUBLE, a), make_column(0, 4, T.DOUBLE, rng.normal(size=n))]
    got, stats, _ = run_both(sum_plan(), cols, keys=["0_1"], options=FX)
    assert stats.main_kernel_name.decode() == NAME
    rows = rows_as_set(list(got), ["0_1"])
    names = [c.name for c in got]
    s = names.index("1_2")
    assert np.isnan(rows[(1,)][s]) and rows[(2,)][s] == np.inf and rows[(3,)][s] == -np.inf and np.isnan(rows[(4,)][s])


@pytest.mark.parametrize("groups", [1, 2, 1000, 3000, 40_000])
def test_fx_group_counts_on_both_sides_of_the_shared_table(groups):
    """1 group: every row of a CTA lands in one slot (the head room M is sized for that); 3000 / 40k groups: the shared table overflows or
    is skipped, rows go to the global table beside the fixed-point slots"""
    rng = np.random.default_rng(groups)
    n = 500_000
    cols = table(rng, n, groups, rng.normal(size=n) * 7.0, rng.random(n), c=rng.integers(-(1 << 40), 1 << 40, n))
    plan = sum_plan(int_sum=True)
    for run in range(2):   # the second run sizes its table from the cardinality the first one learned
        _, stats, _ = run_both(plan, cols, keys=["0_1"], options=FX)
    assert stats.main_kernel_name.decode() in (NAME, "k_agg_group_direct", "k_agg_interp")


@pytest.mark.parametrize("shape", ["one_sum", "no_filter", "int64_key", "three_sums"])
def test_fx_shapes(shape):
    rng = np.random.default_rng(hash(shape) % 1000)
    n = 200_000
    if shape == "one_sum":
        cols, plan = table(rng, n, 300, rng.normal(size=n)), sum_plan(n_sums=1)
    elif shape == "no_filter":
        cols, plan = table(rng, n, 300, rng.normal(size=n), rng.random(n)), sum_plan(with_filter=False)
    elif shape == "int64_key":
        cols = table(rng, n, 300, rng.normal(size=n), rng.random(n), key_type=T.INT64)
        cols[0] = make_column(0, 1, T.INT64, (cols[0].values.astype(np.int64) - 150) * (1 << 33))
        plan = sum_plan(key_type=T.INT64)
    else:
        cols, plan = table(rng, n, 300, rng.normal(size=n), rng.random(n) * 1e-5, c=rng.integers(-(1 << 62), 1 << 62, n)), sum_plan(int_sum=True)
    _, stats, _ = run_both(plan, cols, keys=["0_1"], options=FX)
    assert stats.main_kernel_name.decode() == NAME


def test_fx_agrees_with_the_cas_variant():
    """both variants of the lean kernel over the same table: counts identical, double sums within 1e-9 (each FX value is rounded to at
    least 30 significant bits at this size; the CAS variant reorders IEEE adds), two FX runs within 1e-12 of each other (a CTA's limbs
    do not depend on the order of its atomics; the CTAs' partial sums still meet in floating point in the global table)"""
    cols = datagen.c2_table(0, 2_000_000, n_groups=200)
    plan = queries.c2_filter_groupby()
    a, sa = execute(plan, cols, device=0, options=FX)
    b, _ = execute(plan, cols, device=0, options=FX)
    c, sc = execute(plan, cols, device=0, options={"lean_fx": 0})
    assert sa.main_kernel_name.decode() == NAME and sc.main_kernel_name.decode() == "k_agg_group_lean"
    ra, rb, rc = rows_as_set(list(a), ["0_1"]), rows_as_set(list(b), ["0_1"]), rows_as_set(list(c), ["0_1"])
    assert set(ra) == set(rb) == set(rc)
    for k in ra:
        for x, y, z in zip(ra[k], rb[k], rc[k]):
            if isinstance(x, float):
                assert abs(x - y) <= 1e-12 * max(abs(y), 1.0), (k, x, y)
                assert abs(x - z) <= 1e-9 * max(abs(z), 1.0), (k, x, z)
            elif not isinstance(x, bytes):
                assert x == y == z


def test_fx_fused_join_probe():
    rng = np.random.default_rng(9)
    nd, nf = 50_000, 600_000
    dim = [make_column(1, 1, T.INT32, rng.permutation(nd)), make_column(1, 2, T.INT32, rng.integers(0, 500, nd))]
    fact = [make_column(0, 1, T.INT32, rng.integers(0, nd + 1000, nf)), make_column(0, 2, T.DOUBLE, rng.normal(size=nf) * 100)]
    _, stats, _ = run_both(queries.c3_join_groupby(), fact + dim, keys=["1_2"], options=FX, batches=[dim, fact])
    assert stats.main_kernel_name.decode() == NAME


def test_fx_plan_goes_back_to_cas_when_its_values_do_not_fit_one_scale():
    """a reused plan (bkgpu_reset) whose double column puts most rows on FX's exact path — outliers 1e18 times the bulk dominate the
    sample — launches the CAS kernel from its second request on (the exact-path counter comes back with the counter block)"""
    from baikaldb_b200.exec_node import ColumnSource, GpuExecNode, RowBatch, RuntimeState
    rng = np.random.default_rng(3)
    n = 300_000
    cols = table(rng, n, 20, DISTS["outliers"](rng, n), rng.random(n))
    st = RuntimeState(device=0, options=dict(FX))
    node = GpuExecNode(); node.init(sum_plan()); node.add_child(ColumnSource([cols]))
    assert node.open(st) == 0, st.error_msg
    rb = RowBatch()
    eos = False
    while not eos:
        _, eos = node.get_next(st, rb)
    assert node.stats().main_kernel_name.decode() == NAME
    node.reset(); node.push(cols); node.finish()
    assert node.stats().main_kernel_name.decode() == "k_agg_group_lean"
    node.close()
