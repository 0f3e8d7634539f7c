"""STRING columns through order-preserving dictionary codes (baikaldb_b200/dictionary.py): the rewritten fragment — INT32 codes, literal
comparisons as code thresholds — executed by the oracle equals pyarrow's own string kernels on the original strings: filters with every
comparison operator and literals that are / are not in the dictionary, IN, NULLs, GROUP BY a string key with MIN / MAX / COUNT of another
string column, a join on string keys (both sides share one dictionary), ORDER BY a string LIMIT k; unsupported uses are refused."""
import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pytest

from baikaldb_b200 import dictionary as D, plan as P
from baikaldb_b200._lib import explain
from baikaldb_b200.column import make_column
from baikaldb_b200.plan import PrimitiveType as T
from oracle import oracle

WORDS = [b"", b"a", b"ab", b"abc", b"b", b"ba", b"k", b"kk", b"m", b"zebra", b"Zebra", b"\xe4\xb8\xad", b"0", b"10", b"9"]


def _strings(rng, n, null_frac=0.1, words=WORDS):
    idx = rng.integers(0, len(words), n)
    ok = rng.random(n) >= null_frac
    return [words[i] if o else None for i, o in zip(idx, ok)]


def _run(plan, string_cols, other_cols):
    enc = D.encode_strings(plan, string_cols)
    explain(enc.plan.serialize())                           # the library lowers the rewritten fragment (host side)
    res = oracle.execute(enc.plan.serialize(), enc.columns + other_cols)
    return enc, enc.decode(res.columns)


def test_filters_with_literals_group_by_string_min_max_count():
    rng = np.random.default_rng(1)
    n = 20_000
    s1, s2, s3 = _strings(rng, n), _strings(rng, n, 0.2), _strings(rng, n, 0.0)
    v = rng.normal(size=n)
    tbl = pa.table({"s1": pa.array(s1, pa.binary()), "s2": pa.array(s2, pa.binary()), "s3": pa.array(s3, pa.binary()), "v": v})
    S = lambda slot: P.slot_ref(0, slot, T.STRING)
    cases = [("ge_present", P.ge(S(3), P.str_lit("k")), pc.greater_equal(tbl["s3"], b"k")),
             ("gt_absent", P.gt(S(3), P.str_lit("c")), pc.greater(tbl["s3"], b"c")),
             ("lt_absent", P.lt(S(3), P.str_lit("aa")), pc.less(tbl["s3"], b"aa")),
             ("le_present", P.le(S(3), P.str_lit("ab")), pc.less_equal(tbl["s3"], b"ab")),
             ("ne_present", P.ne(S(3), P.str_lit("abc")), pc.not_equal(tbl["s3"], b"abc")),
             ("eq_absent", P.eq(S(3), P.str_lit("nope")), pc.equal(tbl["s3"], b"nope")),
             ("lit_left", P.lt(P.str_lit("b"), S(3)), pc.greater(tbl["s3"], b"b")),
             ("in", P.in_(S(3), P.str_lit("zebra"), P.str_lit("k"), P.str_lit("missing")), pc.is_in(tbl["s3"], value_set=pa.array([b"zebra", b"k", b"missing"], pa.binary()))),
             ("nullable_ne_absent", P.ne(S(2), P.str_lit("nope")), pc.not_equal(tbl["s2"], b"nope"))]
    for name, pred, mask in cases:
        aggs = [P.agg_expr("count_star", 1, 1), P.agg_expr("sum", 1, 2, None, P.slot_ref(0, 4, T.DOUBLE)), P.agg_expr("min", 1, 3, None, S(2)),
                P.agg_expr("max", 1, 4, None, S(2)), P.agg_expr("count", 1, 5, None, S(2))]
        plan = P.Plan(P.agg(P.where(P.scan(0), pred), 1, [S(1)], aggs),
                      {0: [(1, T.STRING), (2, T.STRING), (3, T.STRING), (4, T.DOUBLE)], 1: [(1, T.INT64), (2, T.DOUBLE), (3, T.STRING), (4, T.STRING), (5, T.INT64)]})
        scols = [D.StringColumn(0, 1, s1), D.StringColumn(0, 2, s2), D.StringColumn(0, 3, s3)]
        enc, got = _run(plan, scols, [make_column(0, 4, T.DOUBLE, v)])
        by = {c.name: (c.values if isinstance(c, D.StringColumn) else c.to_list()) for c in got}
        want = tbl.filter(pc.fill_null(mask, False)).group_by("s1", use_threads=False).aggregate([([], "count_all"), ("v", "sum"), ("s2", "min"), ("s2", "max"), ("s2", "count")]).to_pydict()
        w = {k: (c, sv, mn, mx, cn) for k, c, sv, mn, mx, cn in zip(want["s1"], want["count_all"], want["v_sum"], want["s2_min"], want["s2_max"], want["s2_count"])}
        g = {k: (c, sv, mn, mx, cn) for k, c, sv, mn, mx, cn in zip(by["0_1"], by["1_1"], by["1_2"], by["1_3"], by["1_4"], by["1_5"])}
        assert set(g) == set(w), (name, set(g) ^ set(w))
        for k in g:
            assert g[k][0] == w[k][0] and g[k][2:] == w[k][2:], (name, k, g[k], w[k])
            assert abs(g[k][1] - w[k][1]) <= 1e-9 * max(1.0, abs(w[k][1])), (name, k)


def test_join_on_string_keys_shares_one_dictionary():
    rng = np.random.default_rng(2)
    names = [f"dim{i:04d}".encode() for i in range(400)] + [b"only_in_dim"]
    dk = list(names); rng.shuffle(dk)
    dattr = rng.integers(0, 12, len(dk))
    fk = [names[i] if o else None for i, o in zip(rng.integers(0, 400, 30_000), rng.random(30_000) > 0.05)] + [b"only_in_fact"] * 7
    fv = rng.normal(size=len(fk))
    aggs = [P.agg_expr("count_star", 2, 1), P.agg_expr("sum", 2, 2, None, P.slot_ref(0, 2, T.DOUBLE))]
    j = P.join(P.scan(1), P.scan(0), [P.eq(P.slot_ref(1, 1, T.STRING), P.slot_ref(0, 1, T.STRING))])
    plan = P.Plan(P.agg(j, 2, [P.slot_ref(1, 2, T.INT32)], aggs), {0: [(1, T.STRING), (2, T.DOUBLE)], 1: [(1, T.STRING), (2, T.INT32)], 2: P.agg_tuple_slots(aggs, [T.INT64, T.DOUBLE])})
    enc = D.encode_strings(plan, [D.StringColumn(0, 1, fk), D.StringColumn(1, 1, dk)])
    assert enc.dictionaries[(0, 1)] is enc.dictionaries[(1, 1)]                     # one comparison domain
    explain(enc.plan.serialize())
    res = oracle.execute(enc.plan.serialize(), [enc.columns[0], make_column(0, 2, T.DOUBLE, fv), enc.columns[1], make_column(1, 2, T.INT32, dattr)])
    got = {k: (c, s) for k, c, s in zip(res.columns[0].to_list(), res.columns[1].to_list(), res.columns[2].to_list())}
    fact = pa.table({"k": pa.array(fk, pa.binary()), "v": fv}); dim = pa.table({"k": pa.array(dk, pa.binary()), "attr": dattr})
    want = fact.join(dim, "k", join_type="inner").group_by("attr", use_threads=False).aggregate([([], "count_all"), ("v", "sum")]).to_pydict()
    w = {k: (c, s) for k, c, s in zip(want["attr"], want["count_all"], want["v_sum"])}
    assert set(got) == set(w)
    for k in got:
        assert got[k][0] == w[k][0] and abs(got[k][1] - w[k][1]) <= 1e-9 * max(1.0, abs(w[k][1]))


@pytest.mark.parametrize("asc", [True, False])
def test_order_by_string_limit(asc):
    rng = np.random.default_rng(3)
    n = 5000
    s = _strings(rng, n, 0.15, [f"{i:03d}".encode() for i in range(300)])
    rid = np.arange(n, dtype=np.int32)
    plan = P.Plan(P.sort(P.scan(0), [P.slot_ref(0, 1, T.STRING)], [asc], limit=40, tuple_id=0), {0: [(1, T.STRING), (2, T.INT32)]})
    enc, got = _run(plan, [D.StringColumn(0, 1, s)], [make_column(0, 2, T.INT32, rid)])
    keys, rows = got[0].values, got[1].to_list()
    # the planner's default: NULLs first when ascending, last when descending; ties keep arrival order (TopNSorter is stable)
    order = sorted(range(n), key=lambda i: ((0, b"") if s[i] is None else (1, s[i]), i)) if asc else \
        sorted(range(n), key=lambda i: ((1, b"") if s[i] is None else (0, bytes(255 - b for b in s[i]) + b"\xff"), i))
    assert rows == [int(rid[i]) for i in order[:40]] and keys == [s[i] for i in order[:40]]


def test_unsupported_uses_of_strings_are_refused():
    s = D.StringColumn(0, 1, [b"a", b"b", None])
    S = P.slot_ref(0, 1, T.STRING)
    tuples = {0: [(1, T.STRING), (2, T.DOUBLE)], 1: [(1, T.DOUBLE)]}
    with pytest.raises(D.Unsupported):   # SUM over strings
        D.encode_strings(P.Plan(P.agg(P.scan(0), 1, [], [P.agg_expr("sum", 1, 1, None, S)]), tuples), [s])
    with pytest.raises(D.Unsupported):   # a string compared with a number
        D.encode_strings(P.Plan(P.agg(P.where(P.scan(0), P.gt(S, P.int_lit(3))), 1, [], [P.agg_expr("count_star", 1, 1)]), tuples), [s])
    with pytest.raises(D.Unsupported):   # a function of a string
        D.encode_strings(P.Plan(P.agg(P.where(P.scan(0), P.eq(P.common("length", S), P.int_lit(1))), 1, [], [P.agg_expr("count_star", 1, 1)]), tuples), [s])


@pytest.mark.gpu
def test_gpu_runs_the_rewritten_fragment():
    """the GPU sees only INT32 codes: the rewritten GROUP BY / MIN / MAX fragment through the C ABI equals the oracle, and decodes to pyarrow's answer"""
    from tests.util import run_both
    rng = np.random.default_rng(4)
    n = 200_000
    s1, s2 = _strings(rng, n), _strings(rng, n, 0.2)
    v = rng.normal(size=n)
    S = lambda slot: P.slot_ref(0, slot, T.STRING)
    aggs = [P.agg_expr("count_star", 1, 1), P.agg_expr("sum", 1, 2, None, P.slot_ref(0, 4, T.DOUBLE)), P.agg_expr("min", 1, 3, None, S(2)), P.agg_expr("max", 1, 4, None, S(2))]
    plan = P.Plan(P.agg(P.where(P.scan(0), P.ge(S(2), P.str_lit("b"))), 1, [S(1)], aggs),
                  {0: [(1, T.STRING), (2, T.STRING), (4, T.DOUBLE)], 1: [(1, T.INT64), (2, T.DOUBLE), (3, T.STRING), (4, T.STRING)]})
    enc = D.encode_strings(plan, [D.StringColumn(0, 1, s1), D.StringColumn(0, 2, s2)])
    got, _, _ = run_both(enc.plan, enc.columns + [make_column(0, 4, T.DOUBLE, v)], keys=["0_1"])
    dec = {c.name: (c.values if isinstance(c, D.StringColumn) else c.to_list()) for c in enc.decode(got)}
    tbl = pa.table({"s1": pa.array(s1, pa.binary()), "s2": pa.array(s2, pa.binary()), "v": v})
    want = tbl.filter(pc.fill_null(pc.greater_equal(tbl["s2"], b"b"), False)).group_by("s1", use_threads=False).aggregate([([], "count_all"), ("s2", "min"), ("s2", "max")]).to_pydict()
    w = {k: (c, mn, mx) for k, c, mn, mx in zip(want["s1"], want["count_all"], want["s2_min"], want["s2_max"])}
    g = {k: (c, mn, mx) for k, c, mn, mx in zip(dec["0_1"], dec["1_1"], dec["1_3"], dec["1_4"])}
    assert g == w


def test_like_matcher_equals_the_references_known_answers():
    """test/test_predicate.cpp:33-66 (TEST(test_covent_pattern, case_all)): the Binary-charset vectors and the charset-independent ASCII ones of
    LikePredicate::like<Charset>, through the restatement in dictionary.like_match (the GBK vectors need a GBK decoder and are not restated)"""
    binary = [(b"www.bad/aca?bd_vid", b"www.bad/aca?bd_vid", True), (b"abc", b"a_c", True), (b"abc", b"%", True), (b"axxx", b"a%x%x", True),
              (b"test", b"te%st", True), (b"test", b"te%%st", True), (b"test", b"%test%", True), (b"3hello", b"3%hello", True),
              (b"aaaaaaaaaaaaaaaaaaaaaaaaaaa", b"a%a%a%a%a%a%a%a%b", False)]
    for t, p, want in binary:
        assert D.like_match(t, p, "binary") is want, (t, p)
    for t, p, want in [(b"", b"", True), (b"test", b"_%_%_%_", True), (b"test", b"_%_%st", True), (b"axxx", b"a%x%x", True)] + binary:
        assert D.like_match(t, p, "utf8") is want, (t, p)
    # the escape character takes `%` and `_` literally (the reference's GBK vectors "x\\%y" / "x\\_y", here with ASCII and UTF-8 text)
    assert D.like_match("中%文".encode(), "中\\%文".encode(), "utf8") is True and D.like_match("中间文".encode(), "中\\%文".encode(), "utf8") is False
    assert D.like_match("中f文".encode(), "中\\_文".encode(), "utf8") is False and D.like_match("中f文".encode(), "中_文".encode(), "utf8") is True
    assert D.like_match("中aaa文".encode(), "中%文".encode(), "utf8") is True
    # `_` is one CHARACTER in a charset, one BYTE in Binary
    assert D.like_match("中".encode(), b"_", "utf8") is True and D.like_match("中".encode(), b"_", "binary") is False and D.like_match("中".encode(), b"___", "binary") is True
    assert D.like_match(b"\xffa", b"\xffa", "utf8") is None and D.like_one(b"\xffa", b"\xffa", "utf8") is True   # a malformed character: retried as Binary (like_one)
    assert D.like_match(b"\xff\xfe", b"_", "utf8") is False                                                       # ... but `_` steps over a malformed byte


def test_like_becomes_ranges_of_the_dictionary():
    rng = np.random.default_rng(8)
    words = [b"", b"a", b"ab", b"abc", b"abd", b"b", b"ba", b"bab", b"cab", b"k", b"zebra", "中文".encode(), "中间".encode(), b"a%c", b"a_c"]
    n = 8000
    s = _strings(rng, n, 0.1, words)
    tbl = pa.table({"s": pa.array(s, pa.binary())})
    for pat, n_ranges in [("ab%", 1), ("%", 1), ("a_", 1), ("%ab%", 2), ("b%b", 1), ("nomatch%", 0), ("中_", 1), ("a\\%c", 1), ("%a%", None), ("_", None)]:
        plan = P.Plan(P.agg(P.where(P.scan(0), P.like(P.slot_ref(0, 1, T.STRING), P.str_lit(pat))), 1, [P.slot_ref(0, 1, T.STRING)], [P.agg_expr("count_star", 1, 1)]),
                      {0: [(1, T.STRING)], 1: [(1, T.INT64)]})
        enc, got = _run(plan, [D.StringColumn(0, 1, s)], [])
        g = dict(zip(got[0].values, got[1].to_list()))
        mask = pc.match_like(tbl["s"].cast(pa.string()), pat)     # (utf8 type: `_` is one character, as in the reference's UTF8Charset; on binary pyarrow counts bytes)
        w = tbl.filter(pc.fill_null(mask, False)).group_by("s", use_threads=False).aggregate([([], "count_all")]).to_pydict()
        assert g == dict(zip(w["s"], w["count_all"])), pat
        if n_ranges is not None:   # the shape of the rewritten predicate: no range -> `code = -1`, one -> AND, several -> OR of ANDs
            pred = enc.plan.root.children[0].conjuncts[0]
            shape = 0 if pred.node_type == P.ExprNodeType.FUNCTION_CALL else 1 if pred.node_type == P.ExprNodeType.AND_PREDICATE else len(pred.children)
            assert shape == n_ranges, (pat, shape)
    many = [f"{c}x".encode() for c in "abcdefghijklmnopqrstuvwxyz"] + [f"{c}y".encode() for c in "abcdefghijklmnopqrstuvwxyz"]
    with pytest.raises(D.Unsupported):   # 26 separate ranges: refused, the caller keeps its CPU engine for this fragment
        D.encode_strings(P.Plan(P.agg(P.where(P.scan(0), P.like(P.slot_ref(0, 1, T.STRING), P.str_lit("%x"))), 1, [], [P.agg_expr("count_star", 1, 1)]),
                                {0: [(1, T.STRING)], 1: [(1, T.INT64)]}), [D.StringColumn(0, 1, many)])


def test_ipc_in_and_out_with_string_columns():
    """the store <-> db wire with STRING fields (large_binary, the Chunk map): strings in, dictionary-coded fragment (run by the oracle here),
    strings out — equal to pyarrow's own group-by over the same batch"""
    from baikaldb_b200 import arrow_io
    rng = np.random.default_rng(6)
    n = 12_000
    city = pa.array(_strings(rng, n, 0.05, [b"beijing", b"shanghai", b"shenzhen", "杭州".encode(), b"chengdu", b"xi'an"]), pa.large_binary())
    tag = pa.array(_strings(rng, n, 0.3), pa.large_binary())
    amount = rng.random(n) * 100
    rb = pa.RecordBatch.from_arrays([city, tag, pa.array(amount)], names=["0_1", "0_2", "0_3"])
    S = lambda s: P.slot_ref(0, s, T.STRING)
    aggs = [P.agg_expr("count_star", 1, 1), P.agg_expr("sum", 1, 2, None, P.slot_ref(0, 3, T.DOUBLE)), P.agg_expr("max", 1, 3, None, S(2))]
    plan = P.Plan(P.agg(P.where(P.scan(0), P.like(S(1), P.str_lit("s%")), P.ne(S(1), P.str_lit("shenzhen"))), 1, [S(1)], aggs),
                  {0: [(1, T.STRING), (2, T.STRING), (3, T.DOUBLE)], 1: [(1, T.INT64), (2, T.DOUBLE), (3, T.STRING)]})
    s, d = arrow_io.execute_ipc_with_strings(plan, rb.schema.serialize().to_pybytes(), rb.serialize().to_pybytes(),
                                             runner=lambda p, c: oracle.execute(p.serialize(), c).columns)
    out = pa.ipc.read_record_batch(pa.py_buffer(d), pa.ipc.read_schema(pa.py_buffer(s))).to_pydict()
    assert pa.ipc.read_schema(pa.py_buffer(s)).field("0_1").type == pa.large_binary() and pa.ipc.read_schema(pa.py_buffer(s)).field("1_3").type == pa.large_binary()
    tbl = pa.table({"city": city, "tag": tag, "amount": amount})
    m = pc.and_kleene(pc.match_like(tbl["city"].cast(pa.string()), "s%"), pc.not_equal(tbl["city"], b"shenzhen"))
    want = tbl.filter(pc.fill_null(m, False)).group_by("city", use_threads=False).aggregate([([], "count_all"), ("amount", "sum"), ("tag", "max")]).to_pydict()
    g = {k: (c, mx) for k, c, mx in zip(out["0_1"], out["1_1"], out["1_3"])}
    assert g == {k: (c, mx) for k, c, mx in zip(want["city"], want["count_all"], want["tag_max"])} and set(g) == {b"shanghai"}
    sums = dict(zip(out["0_1"], out["1_2"]))
    for k, v in zip(want["city"], want["amount_sum"]):
        assert abs(sums[k] - v) <= 1e-9 * abs(v)


@pytest.mark.parametrize("seed", range(40))
def test_fuzz_string_predicates_against_pyarrow(seed):
    """random predicate trees (AND / OR / NOT over = != < <= > >= with literals in and out of the dictionary, IN, LIKE, IS NULL, and
    column-to-column comparisons) over three nullable STRING columns: rewritten to codes and run by the oracle == pyarrow's Kleene logic"""
    rng = np.random.default_rng(1000 + seed)
    n = 3000
    words = [b"", b"a", b"aa", b"ab", b"abc", b"b", b"bb", b"c", b"ca", b"cab", b"d", b"x", b"xy", b"xyz", b"y"]
    cols = {i: _strings(rng, n, 0.15, words) for i in (1, 2, 3)}
    tbl = pa.table({f"s{i}": pa.array(v, pa.binary()) for i, v in cols.items()})
    lits = words + [b"0", b"ab0", b"bz", b"zz"]
    S = lambda i: P.slot_ref(0, i, T.STRING)

    def leaf():
        i = int(rng.integers(1, 4))
        kind = rng.integers(0, 10)
        f = tbl[f"s{i}"]
        if kind < 5:
            op = ["eq", "ne", "lt", "le", "gt", "ge"][int(rng.integers(0, 6))]
            lit = lits[int(rng.integers(0, len(lits)))]
            pcf = {"eq": pc.equal, "ne": pc.not_equal, "lt": pc.less, "le": pc.less_equal, "gt": pc.greater, "ge": pc.greater_equal}[op]
            if rng.random() < 0.25:   # literal on the left
                mirror = {"eq": "eq", "ne": "ne", "lt": "gt", "le": "ge", "gt": "lt", "ge": "le"}[op]
                return getattr(P, mirror)(P.str_lit(lit.decode()), S(i)), pcf(f, lit)
            return getattr(P, op)(S(i), P.str_lit(lit.decode())), pcf(f, lit)
        if kind == 5:
            j = int(rng.integers(1, 4))
            return P.lt(S(i), S(j)), pc.less(f, tbl[f"s{j}"])
        if kind == 6:
            members = [lits[int(k)] for k in rng.integers(0, len(lits), 3)]
            # (pyarrow's is_in answers FALSE for a NULL input; SQL's IN — InPredicate, include/expr/predicate.h:281-345 — answers NULL, which matters under NOT)
            return P.in_(S(i), *[P.str_lit(m.decode()) for m in members]), pc.if_else(pc.is_null(f), pa.scalar(None, pa.bool_()), pc.is_in(f, value_set=pa.array(members, pa.binary())))
        if kind == 7:
            pat = ["a%", "%b", "_", "%a%", "x_z", "c%b", "%"][int(rng.integers(0, 7))]
            return P.like(S(i), P.str_lit(pat)), pc.match_like(f.cast(pa.string()), pat)
        if kind == 8:
            return P.is_null(S(i)), pc.is_null(f)
        return P.eq(S(i), S(int(rng.integers(1, 4)))), None

    def tree(depth):
        if depth == 0 or rng.random() < 0.3:
            e, m = leaf()
            while m is None:
                e, m = leaf()
            return e, m
        k = rng.integers(0, 3)
        if k == 0:
            e, m = tree(depth - 1)
            return P.not_(e), pc.invert(m)
        (a, ma), (b, mb) = tree(depth - 1), tree(depth - 1)
        return (P.and_(a, b), pc.and_kleene(ma, mb)) if k == 1 else (P.or_(a, b), pc.or_kleene(ma, mb))

    pred, mask = tree(3)
    plan = P.Plan(P.agg(P.where(P.scan(0), pred), 1, [S(1)], [P.agg_expr("count_star", 1, 1), P.agg_expr("max", 1, 2, None, S(2))]),
                  {0: [(1, T.STRING), (2, T.STRING), (3, T.STRING)], 1: [(1, T.INT64), (2, T.STRING)]})
    enc, got = _run(plan, [D.StringColumn(0, i, cols[i]) for i in (1, 2, 3)], [])
    g = {k: (c, m) for k, c, m in zip(got[0].values, got[1].to_list(), got[2].values)} if got and len(got[0].values) else {}
    want = tbl.filter(pc.fill_null(mask, False)).group_by("s1", use_threads=False).aggregate([([], "count_all"), ("s2", "max")]).to_pydict()
    assert g == {k: (c, m) for k, c, m in zip(want["s1"], want["count_all"], want["s2_max"])}
