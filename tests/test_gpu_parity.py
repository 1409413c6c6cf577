"""GPU (-m gpu): the CUDA path through the C ABI vs the CPU oracle on the same seeded inputs — bit-exact on u32 ids, compared as
bags (canonical sort), because the reference's own row order is hash-iteration order (SURVEY.md §7)."""
import os

import numpy as np
import pytest

from kolibrie_b200 import capi as c
from kolibrie_b200 import datagen
from kolibrie_b200.engine import Dictionary
from tests import helpers as H
from tests import oracle_api as O

pytestmark = pytest.mark.gpu

S, P, Ob = 0, 1, 2
ORDERED = os.environ.get("KOLIBRIE_ORDERED", "0") != "0"


def load(ctx, d):
    ctx.store_load(d.s, d.p, d.o)
    ctx.dict_numeric_load(d.num_or0, d.is_num)
    return O.Db(d.s, d.p, d.o, d.num_or0, d.is_num)


_EMP = {}


@pytest.fixture
def emp(ctx):
    """20 000-employee store: generated once, (re)loaded for every test that asks for it (other tests replace the store)"""
    if "d" not in _EMP:
        _EMP["d"] = datagen.employee_dataset(20000)
    d = _EMP["d"]
    return d, load(ctx, d)


def random_store(seed, n, n_terms=50, n_preds=5):
    rng = np.random.default_rng(seed)
    tr = np.stack([rng.integers(0, n_terms, n), rng.integers(100, 100 + n_preds, n), rng.integers(0, n_terms, n)], axis=1).astype(np.uint32)
    return np.unique(tr, axis=0)


def test_integration_fixture_on_device(ctx):
    fx = H.load("integration_fixture.json")
    tr = np.array(fx["triples"], dtype=np.uint32)
    ctx.store_load(tr[:, 0], tr[:, 1], tr[:, 2])
    ex = fx["expect"]
    r = ctx.scan([c.pattern(c.K(0), c.V(P), c.V(Ob)), c.pattern(c.V(S), c.K(3), c.V(Ob)), c.pattern(c.V(S), c.V(P), c.K(10)),
                  c.pattern(c.V(S), c.K(6), c.K(2))])
    assert [x.n_rows for x in r[:3]] == [ex["subject==person1"], ex["predicate==ex:name"], ex["object==Jane Doe"]]
    assert sorted(r[3].column(0).tolist()) == ex["worksFor_company1_subjects"]
    assert sorted(r[0].to_numpy([P, Ob]).tolist()) == [[3, 9], [4, 12], [5, 14], [6, 2]]
    # the two joins whose answers integration_test.rs asserts (:286-299 tech employees, :302-342 ACME employees under 30), on the
    # device, with and without the store index. ids: terms list of the fixture (ex:name 3, ex:age 4, ex:worksFor 6, ex:industry 8, ...)
    t = {name: i for i, name in enumerate(fx["terms"])}
    num = np.zeros(len(t))
    isn = np.zeros(len(t), np.uint8)
    for name in ("30", "25", "2000"):
        num[t[name]], isn[t[name]] = float(name), 1
    ctx.dict_numeric_load(num, isn)
    C_, E_, A_ = 0, 1, 2
    tech = [c.pattern(c.V(C_), c.K(t["ex:industry"]), c.K(t["Technology"])), c.pattern(c.V(E_), c.K(t["ex:worksFor"]), c.V(C_))]
    young = [c.pattern(c.V(C_), c.K(t["ex:name"]), c.K(t["ACME Corp"])), c.pattern(c.V(E_), c.K(t["ex:worksFor"]), c.V(C_)),
             c.pattern(c.V(E_), c.K(t["ex:age"]), c.V(A_))]
    lt30 = [c.fop(c.F_CMP_NUM, slot=A_, cmp=c.CMP_LT, value=30.0)]
    for indexed in (False, True):
        if indexed:
            ctx.build_index()
        assert sorted(ctx.bgp_execute(tech).to_numpy([E_])[:, 0].tolist()) == ex["tech_employees"]
        assert sorted(ctx.bgp_execute(young, lt30).to_numpy([E_])[:, 0].tolist()) == ex["young_acme_employees"]


@pytest.mark.parametrize("n", [0, 1, 31, 2047, 2048, 2049, 70001])
def test_scan_edges_vs_oracle(ctx, n):
    """empty, sub-tile, exact-tile and ragged stores; constants in every position; repeated variable; all patterns in ONE pass"""
    tr = random_store(n, n) if n else np.empty((0, 3), np.uint32)
    ctx.store_load(tr[:, 0], tr[:, 1], tr[:, 2])
    db = O.Db(tr[:, 0], tr[:, 1], tr[:, 2])
    pats = [c.pattern(c.V(S), c.K(101), c.V(Ob)), c.pattern(c.K(7), c.V(P), c.V(Ob)), c.pattern(c.V(S), c.V(P), c.K(3)),
            c.pattern(c.K(7), c.K(101), c.V(Ob)), c.pattern(c.V(S), c.K(102), c.K(3)), c.pattern(c.V(S), c.V(P), c.V(Ob)),
            c.pattern(c.V(S), c.K(103), c.V(S)), c.pattern(c.K(7), c.K(101), c.K(3))]
    rels = ctx.scan(pats)
    for pt, r in zip(pats, rels):
        want = db.scan(pt)
        assert r.slots == want.slots
        got = r.to_numpy()
        if ORDERED:
            assert np.array_equal(got, want.to_numpy()), "ordered compaction must reproduce store order exactly"
        else:
            H.assert_same_bag(got, want.to_numpy(), "scan")


def test_scan_multi_segment_and_evict(ctx):
    tr = random_store(5, 30000)
    parts = np.array_split(tr, 5)
    ctx.store_clear()
    for i, pt in enumerate(parts):
        ctx.store_append(pt[:, 0], pt[:, 1], pt[:, 2], tag=100 + i)
    assert ctx.store_size() == (len(tr), 5)
    pat = c.pattern(c.V(S), c.K(102), c.V(Ob))
    same = (lambda a, b: np.array_equal(a, b)) if ORDERED else (lambda a, b: np.array_equal(H.canon(a), H.canon(b)))
    assert same(ctx.scan([pat])[0].to_numpy(), O.Db(tr[:, 0], tr[:, 1], tr[:, 2]).scan(pat).to_numpy())
    ctx.store_evict(102)  # RSP slide: drop the third segment
    rest = np.concatenate([parts[0], parts[1], parts[3], parts[4]])
    assert same(ctx.scan([pat])[0].to_numpy(), O.Db(rest[:, 0], rest[:, 1], rest[:, 2]).scan(pat).to_numpy())
    with pytest.raises(c.KolibrieError):
        ctx.store_evict(999)
    # kb_store_delete = set difference by value (SparqlDatabase::delete_triple)
    dele = rest[::7]
    ctx.store_delete(dele[:, 0], dele[:, 1], dele[:, 2])
    keep = np.array(sorted(set(map(tuple, rest.tolist())) - set(map(tuple, dele.tolist()))), dtype=np.uint32)
    s, p, o = ctx.store_download()
    H.assert_same_bag(np.stack([s, p, o], axis=1), keep, "store after delete")
    # more segments than one scan launch walks (16), of ragged sizes, one of them empty: a star join over the window
    tr2 = random_store(6, 60000, n_terms=3000)
    cuts = sorted(np.random.default_rng(1).choice(np.arange(1, len(tr2)), 22, replace=False).tolist())
    ctx.store_clear()
    for i, pt in enumerate(np.split(tr2, cuts[:10] + [cuts[10], cuts[10]] + cuts[11:])):
        ctx.store_append(pt[:, 0], pt[:, 1], pt[:, 2], tag=500 + i)
    assert ctx.store_size() == (len(tr2), 24)
    db2 = O.Db(tr2[:, 0], tr2[:, 1], tr2[:, 2])
    assert same(ctx.scan([pat])[0].to_numpy(), db2.scan(pat).to_numpy())
    pats = [c.pattern(c.V(0), c.K(100), c.V(1)), c.pattern(c.V(0), c.K(101), c.V(2))]
    H.assert_same_bag(ctx.star_join(0, pats).to_numpy([0, 1, 2]), db2.bgp(pats).to_numpy([0, 1, 2]), "24-segment window")


def test_filter_programs_vs_oracle(ctx, emp):
    d, db = emp
    sal = d.ids["ds:annual_salary"]
    rel = ctx.scan([c.pattern(c.V(0), c.K(sal), c.V(2))])[0]
    orel = db.scan(c.pattern(c.V(0), c.K(sal), c.V(2)))
    some_salary = int(d.o[5])
    progs = [
        [c.fop(c.F_CMP_NUM, slot=2, cmp=c.CMP_GT, value=100000.0)],
        [c.fop(c.F_CMP_NUM, slot=2, cmp=c.CMP_GE, value=60000.0), c.fop(c.F_CMP_NUM, slot=2, cmp=c.CMP_LT, value=61000.0), c.fop(c.F_AND)],
        [c.fop(c.F_CMP_NUM, slot=2, cmp=c.CMP_LE, value=31000.0), c.fop(c.F_CMP_NUM, slot=2, cmp=c.CMP_GT, value=149000.0), c.fop(c.F_OR), c.fop(c.F_NOT)],
        [c.fop(c.F_EQ_ID, slot=2, id=some_salary)],
        [c.fop(c.F_NE_ID, slot=2, id=some_salary)],
        [c.fop(c.F_EQ_ID, slot=2, id=c.KB_ID_NONE)],          # literal not in the dictionary: = is false ...
        [c.fop(c.F_NE_ID, slot=2, id=c.KB_ID_NONE)],          # ... != is true (types.rs:131-132)
        [c.fop(c.F_CMP_NUM, slot=0, cmp=c.CMP_GE, value=0.0)],  # non-numeric term compares as 0.0 (unwrap_or)
        [c.fop(c.F_CMP_NUM, slot=0, cmp=c.CMP_GT, value=0.0)],
        # arithmetic: (?s * 2 - 100000) / 1000 truthy; division by zero and non-numeric operands make the expression false
        [c.fop(c.F_PUSH_VAR, slot=2), c.fop(c.F_PUSH_CONST, value=2.0), c.fop(c.F_MUL), c.fop(c.F_PUSH_CONST, value=100000.0), c.fop(c.F_SUB),
         c.fop(c.F_PUSH_CONST, value=1000.0), c.fop(c.F_DIV), c.fop(c.F_TRUTHY)],
        [c.fop(c.F_PUSH_VAR, slot=2), c.fop(c.F_PUSH_CONST, value=0.0), c.fop(c.F_DIV), c.fop(c.F_TRUTHY)],
        [c.fop(c.F_PUSH_VAR, slot=0), c.fop(c.F_PUSH_CONST, value=1.0), c.fop(c.F_ADD), c.fop(c.F_TRUTHY)],
        [c.fop(c.F_IS_TRIPLE, slot=0), c.fop(c.F_NOT)],
    ]
    for prog in progs:
        got = ctx.filter(rel, prog).to_numpy()
        want = db.filter(orel, prog).to_numpy()
        H.assert_same_bag(got, want, str(prog[0].op))
    # pushed down into the scan: same rows
    got = ctx.scan([c.pattern(c.V(0), c.K(sal), c.V(2))], [progs[1]])[0].to_numpy()
    H.assert_same_bag(got, db.filter(orel, progs[1]).to_numpy(), "pushdown")


@pytest.mark.parametrize("q", ["cfg1", "cfg2", "cfg3", "star3"])
@pytest.mark.parametrize("mode", [0, 1])
def test_employee_queries_vs_oracle(ctx, emp, q, mode):
    """BASELINE.md §4 queries: fused star join (scan + direct build + multiway probe) vs oracle columnar AND faithful modes"""
    d, db = emp
    js, pats, filt = datagen.employee_queries(d)[q]
    got = ctx.star_join(js, pats, filt)
    want = db.bgp(pats, filt, mode=mode)
    assert sorted(got.slots) == sorted(want.slots)
    H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), q)
    got2 = ctx.bgp_execute(pats, filt)
    H.assert_same_bag(got2.to_numpy(sorted(got2.slots)), want.to_numpy(sorted(want.slots)), q + " via kb_bgp_execute")


def test_star_join_is_deterministic_and_ordered(ctx, emp):
    """KOLIBRIE_ORDERED=1: output in store order, identical from run to run. Default mode: same bag, row order unspecified
    (like the reference, whose row order is hash-iteration order)."""
    d, db = emp
    js, pats, filt = datagen.employee_queries(d)["cfg2"]
    a = ctx.star_join(js, pats, filt).to_numpy([0, 1, 2, 3])
    b = ctx.star_join(js, pats, filt).to_numpy([0, 1, 2, 3])
    if ORDERED:
        assert np.array_equal(a, b), "same query twice -> identical row order"
        assert (np.diff(a[:, 0].astype(np.int64)) > 0).all(), "probe order = store order = ascending subject"
    else:
        H.assert_same_bag(a, b, "same query twice")


def test_star_join_multivalued_falls_back_to_chained(ctx):
    """1:N predicates (duplicate keys on the build side) cannot use the direct table: same bag through the chained path"""
    rng = np.random.default_rng(3)
    n = 4000
    subj = rng.integers(0, 600, n)
    tr = np.unique(np.stack([subj, rng.integers(100, 103, n), rng.integers(1000, 1040, n)], axis=1).astype(np.uint32), axis=0)
    ctx.store_load(tr[:, 0], tr[:, 1], tr[:, 2])
    db = O.Db(tr[:, 0], tr[:, 1], tr[:, 2])
    pats = [c.pattern(c.V(0), c.K(100), c.V(1)), c.pattern(c.V(0), c.K(101), c.V(2)), c.pattern(c.V(0), c.K(102), c.V(3))]
    want = db.bgp(pats).to_numpy([0, 1, 2, 3])
    assert len(want) > n  # real 1:N blow-up
    for _ in range(2):  # second run takes the cached "multi-valued" route directly
        H.assert_same_bag(ctx.star_join(0, pats).to_numpy([0, 1, 2, 3]), want, "1:N star")
    # a pattern that shares a NON-join variable with another (quirk Q3) must still be a natural join
    pats2 = [c.pattern(c.V(0), c.K(100), c.V(1)), c.pattern(c.V(0), c.K(101), c.V(1))]
    H.assert_same_bag(ctx.star_join(0, pats2).to_numpy([0, 1]), db.bgp(pats2).to_numpy([0, 1]), "shared non-join variable")


@pytest.mark.parametrize("seed", range(4))
def test_hash_join_shapes_vs_oracle(ctx, seed):
    """binary natural joins: 1 and 2 common variables, 1:N both ways, empty sides, cartesian product"""
    rng = np.random.default_rng(seed)

    def rel(slots, n, hi):
        cols = [rng.integers(0, hi, n).astype(np.uint32) for _ in slots]
        return ctx.rel_from_host(slots, cols), O.rel_from_host(slots, cols)

    for (ls, ln, rs, rn, hi) in [((0, 1), 3000, (1, 2), 5000, 200), ((0, 1, 2), 2500, (1, 2, 3), 1800, 12), ((0, 1), 700, (0, 1), 900, 30),
                                 ((0, 1), 0, (1, 2), 50, 10), ((0, 1), 40, (2, 3), 30, 10), ((0,), 3000, (0, 5), 10, 4)]:
        (gl, ol), (gr, orr) = rel(ls, ln, hi), rel(rs, rn, hi)
        got = ctx.hash_join(gl, gr)
        want = O.hash_join(ol, orr)
        assert sorted(got.slots) == sorted(want.slots)
        H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), f"{ls}x{rs}")


@pytest.mark.parametrize("csr", ["1", "0"])
def test_join_fanout_grouped_and_chained(csr, monkeypatch):
    """1:N / N:M joins with skewed fan-out through BOTH multimap layouts: the key-grouped (CSR) directory (default for one dense key
    column) and the chained table (KOLIBRIE_CSR_JOIN=0, and always for sparse key ranges / several key columns)"""
    monkeypatch.setenv("KOLIBRIE_CSR_JOIN", csr)
    cx = c.Context(0)
    try:
        rng = np.random.default_rng(17)

        def both(slots, cols):
            cols = [np.ascontiguousarray(x, dtype=np.uint32) for x in cols]
            return cx.rel_from_host(slots, cols), O.rel_from_host(slots, cols)

        hot = np.full(700, 77, np.uint32)  # one key with 700 build rows ...
        bkeys = np.concatenate([hot, rng.integers(0, 5000, 20000).astype(np.uint32)])
        pkeys = np.concatenate([np.full(2000, 77, np.uint32), rng.integers(0, 9000, 40000).astype(np.uint32)])  # ... probed 2000 times; keys 5000..8999 miss
        cases = {
            "skewed 1:N": (((0, 1), [bkeys, rng.integers(0, 1 << 20, len(bkeys))]), ((0, 2, 3), [pkeys, rng.integers(0, 50, len(pkeys)), rng.integers(0, 50, len(pkeys))])),
            "key-only build side": (((0,), [bkeys[:3000]]), ((0, 2), [pkeys[:5000], rng.integers(0, 50, 5000)])),
            "sparse key range": (((0, 1), [bkeys * 100003, bkeys]), ((0, 2), [pkeys * 100003, pkeys])),
            "single row each": (((0, 1), [[5], [6]]), ((0, 2), [[5], [7]])),
            "no key in common": (((0, 1), [[1, 2, 3], [4, 5, 6]]), ((0, 2), [[7, 8], [9, 9]])),
            "exact tile multiples": (((0, 1), [np.arange(2048) % 64, np.arange(2048)]), ((0, 2), [np.arange(1024) % 128, np.arange(1024)])),
        }
        for name, ((ls, lc), (rs, rc)) in cases.items():
            (gl, ol), (gr, orr) = both(ls, lc), both(rs, rc)
            for a, b, oa, ob in ((gl, gr, ol, orr), (gr, gl, orr, ol)):
                got = cx.hash_join(a, b)
                want = O.hash_join(oa, ob)
                assert sorted(got.slots) == sorted(want.slots)
                H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), f"{name} (csr={csr})")
    finally:
        cx.close()


def test_bgp_path_join_vs_oracle(ctx):
    """object->subject path (no star variable): scan all patterns in one pass, then chained joins"""
    tr = random_store(11, 20000, n_terms=400, n_preds=4)
    ctx.store_load(tr[:, 0], tr[:, 1], tr[:, 2])
    db = O.Db(tr[:, 0], tr[:, 1], tr[:, 2])
    pats = [c.pattern(c.V(0), c.K(100), c.V(1)), c.pattern(c.V(1), c.K(101), c.V(2)), c.pattern(c.V(2), c.K(102), c.V(3))]
    got = ctx.bgp_execute(pats, project=[0, 3])
    want = db.bgp(pats, project=[0, 3])
    H.assert_same_bag(got.to_numpy([0, 3]), want.to_numpy([0, 3]), "3-hop path")


def test_group_aggregate_vs_oracle(ctx, emp):
    d, db = emp
    js, pats, _ = datagen.employee_queries(d)["cfg3"]
    rel = ctx.star_join(js, pats)
    orel = db.bgp(pats)
    all_aggs = [(c.AGG_COUNT, 0), (c.AGG_SUM, 2), (c.AGG_MIN, 2), (c.AGG_MAX, 2), (c.AGG_AVG, 2)]
    # all five at once (general kernel), then one variable + one aggregate (the single-key kernel): 3 groups, and thousands of
    # groups (more than a CTA's shared table holds)
    cases = [(gs, all_aggs) for gs in ([1], [2], [1, 4])] + [(gs, [a]) for gs in ([1], [2]) for a in all_aggs] + [([1], [])]
    for gslots, aggs in cases:
        g = ctx.group_aggregate(rel, gslots, aggs)
        w = db.group(orel, gslots, aggs)

        def table(x):
            keys = np.stack(x["keys"], axis=1)
            order = np.lexsort(tuple(keys[:, k] for k in range(keys.shape[1] - 1, -1, -1)))
            return keys[order], x["counts"][order], [v[order] for v in x["values"]]

        gk, gc, gv = table(g)
        wk, wc, wv = table(w)
        assert np.array_equal(gk, wk) and np.array_equal(gc, wc)
        for a, b in zip(gv, wv):
            # salaries are integers: sums stay exact in f64 (< 2^53), so equality is exact; AVG within 1 ulp-ish
            assert np.allclose(a, b, rtol=1e-12, atol=0)


def test_star_join_aggregate_fused_vs_oracle(ctx, emp):
    """kb_star_join_aggregate: GROUP BY folded into the index probe kernel (no joined row is written) for one group variable and at
    most one aggregate; every other shape, and a store without index, takes join + group — all must equal the oracle's group over
    the oracle's join"""
    d, db = emp
    js, pats, _ = datagen.employee_queries(d)["cfg3"]          # slots: e=0, t=1, s=2, n=3, c=4
    _, pats2, filt2 = datagen.employee_queries(d)["cfg2"]

    def table(x):
        keys = np.stack(x["keys"], axis=1)
        order = np.lexsort(tuple(keys[:, k] for k in range(keys.shape[1] - 1, -1, -1)))
        return keys[order], x["counts"][order], [v[order] for v in x["values"]]

    def check(pp, ff, gslots, aggs, what):
        g, n_rows = ctx.star_join_aggregate(js, pp, ff, gslots, aggs)
        orel = db.bgp(pp, ff)
        w = db.group(orel, gslots, aggs)
        gk, gc, gv = table(g)
        wk, wc, wv = table(w)
        assert n_rows == len(orel.to_numpy(sorted(orel.slots))), what
        assert np.array_equal(gk, wk) and np.array_equal(gc, wc), what
        for a, b in zip(gv, wv):
            assert np.allclose(a, b, rtol=1e-12, atol=0), what

    one = [[(c.AGG_COUNT, 0)], [(c.AGG_SUM, 2)], [(c.AGG_MIN, 2)], [(c.AGG_MAX, 2)], [(c.AGG_AVG, 2)], []]
    for indexed in (True, False):
        if indexed:
            ctx.build_index()
        before = ctx.get_stats()["kernel_launches"]
        for aggs in one:
            check(pats, None, [1], aggs, f"by title {aggs} indexed={indexed}")            # 3 groups: the CTA table
            check(pats, None, [2], aggs, f"by salary {aggs} indexed={indexed}")           # thousands of groups: past the CTA table, past 4096 slots
            check(pats2, filt2, [1], aggs, f"FILTER + by title {aggs} indexed={indexed}")  # typed pre-filter on the probe slice
        check(pats, None, [1, 4], [(c.AGG_COUNT, 0)], "two group variables: join + group")
        check(pats, None, [1], [(c.AGG_COUNT, 0), (c.AGG_SUM, 2)], "two aggregates: join + group")
        f_post = [c.fop(c.F_NE_ID, slot=1, id=d.ids["Manager"]), c.fop(c.F_CMP_NUM, slot=2, cmp=c.CMP_GT, value=70000.0), c.fop(c.F_AND)]
        check(pats, f_post, [1], [(c.AGG_AVG, 2)], "filters on two patterns")
        if indexed:  # COUNT by title with the index: one probe launch + the table init, nothing else
            n0 = ctx.get_stats()["kernel_launches"]
            ctx.star_join_aggregate(js, pats, None, [1], [(c.AGG_COUNT, 0)])
            assert ctx.get_stats()["kernel_launches"] - n0 <= 2
        assert ctx.get_stats()["kernel_launches"] > before
        ctx.store_load(d.s, d.p, d.o)  # drops the index for the second pass


def test_legacy_ffi_symbol(ctx):
    """perform_hash_join_cuda as Kolibrie's hash_join_cuda calls it (cuda_join.rs:28-60): ascending indices, literal honoured"""
    d = datagen.employee_dataset(60000)  # 360 000 triples: beyond the reference stub's ~303 K clamp (cuda_join.cu:81-88)
    pred = d.ids["foaf:title"]
    want = O.legacy_select(d.p, d.o, pred)
    got = c.legacy_hash_join_cuda(d.s, d.p, d.o, pred)
    assert np.array_equal(got, want) and len(got) == 60000
    lit = d.ids["Developer"]
    assert np.array_equal(c.legacy_hash_join_cuda(d.s, d.p, d.o, pred, lit), O.legacy_select(d.p, d.o, pred, lit))
    assert len(c.legacy_hash_join_cuda(d.s[:0], d.p[:0], d.o[:0], pred)) == 0
    # the same symbol from the library name Kolibrie links (libcudajoin.so)
    assert np.array_equal(c.legacy_hash_join_cuda(d.s, d.p, d.o, pred, libpath=c.LEGACY_LIB_PATH), want)


def test_legacy_vs_reference_cuda_stub():
    """The reference's OWN cuda_join.cu compiled for sm_100a, run on a B200: the index SET it returned for a seeded input inside the
    range its clamped grid covers is stored in tests/golden/reference/cuda_stub_salary.npz (sorted: the reference's order is atomicAdd
    arrival order). Our symbol must return that set for the same input."""
    import os

    from tests.golden.reference.make_reference_golden import stub_input

    golden = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "cuda_stub_salary.npz"))
    s, p, o, pred, digest = stub_input()
    assert digest == str(golden["input_sha256"]) and pred == int(golden["predicate"]), "the seeded input differs from the stored one"
    theirs = golden["indices"]
    ours = c.legacy_hash_join_cuda(s, p, o, pred)
    assert len(theirs) == 30000 and np.array_equal(theirs, ours)


def test_star_join_host_one_shot(ctx, emp):
    d, db = emp
    js, pats, filt = datagen.employee_queries(d)["cfg2"]
    rows, slots = ctx.star_join_host(d.s, d.p, d.o, js, pats, filt)
    ctx.dict_numeric_load(d.num_or0, d.is_num)
    want = db.bgp(pats, filt)
    H.assert_same_bag(rows[:, [slots.index(s) for s in sorted(slots)]], want.to_numpy(sorted(want.slots)), "host one-shot")
    ctx.store_load(d.s, d.p, d.o)


def test_partition_for_shuffle(ctx, emp):
    d, db = emp
    rel = ctx.scan([c.pattern(c.V(0), c.K(d.ids["foaf:title"]), c.V(1))])[0]
    base = rel.to_numpy([0, 1])
    for g in (2, 8):
        part, offs = ctx.partition(rel, 1, g)
        rows = part.to_numpy([0, 1])
        assert offs[0] == 0 and offs[-1] == len(base)
        for r in range(g):
            chunk = rows[offs[r]:offs[r + 1]]
            assert all(c.lib().kb_shard_of(int(k), g) == r for k in np.unique(chunk[:, 1]))
        H.assert_same_bag(rows, base, "partition is a permutation")


def test_errors_are_reported_not_swallowed(ctx):
    with pytest.raises(c.KolibrieError) as e:
        ctx.scan([c.pattern(c.V(0), c.K(c.KB_ID_NONE), c.V(1))])
    assert e.value.status == c.KB_E_INVALID
    with pytest.raises(c.KolibrieError) as e:
        ctx.star_join(9, [c.pattern(c.V(0), c.K(1), c.V(1)), c.pattern(c.V(0), c.K(2), c.V(2))])
    assert e.value.status == c.KB_E_INVALID
    with pytest.raises(c.KolibrieError) as e:
        ctx.filter(ctx.rel_from_host([0], [np.arange(4, dtype=np.uint32)]), [c.fop(c.F_AND)])
    assert e.value.status == c.KB_E_INVALID


@pytest.mark.parametrize("claimed_rank", [1, 2])
def test_sharded_store_key_compaction(claimed_rank):
    """one rank's shard of a 4-way subject-sharded store: kb_set_sharding compacts the key domain of the direct tables
    (block-cyclic shard function). A context that CLAIMS the wrong rank must notice (foreign subjects) and stay correct."""
    world, rank = 4, 1
    d = datagen.employee_shard(60000, rank, world, prefix=20000)
    assert (np.array([c.lib().kb_shard_of(int(x), world) for x in d.s[::997]]) == rank).all()
    ctx2 = c.Context(0)
    try:
        ctx2.set_sharding(claimed_rank, world)
        ctx2.store_load(d.s, d.p, d.o)
        ctx2.dict_numeric_load(d.num_or0, d.is_num)
        db = O.Db(d.s, d.p, d.o, d.num_or0, d.is_num)
        for q in ("cfg2", "cfg3"):
            js, pats, filt = datagen.employee_queries(d)[q]
            got = ctx2.star_join(js, pats, filt)
            want = db.bgp(pats, filt)
            H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), f"{q} claimed rank {claimed_rank}")
        assert ctx2.get_stats()["fused_scan_builds"] >= 2
    finally:
        ctx2.close()


@pytest.mark.parametrize("q", ["cfg1", "cfg2", "cfg3", "star3"])
def test_index_path_vs_oracle(ctx, emp, q):
    """kb_store_build_index (= build_all_indexes): star joins read predicate slices instead of scanning the store; same bag"""
    d, db = emp
    n_pred, ms = ctx.build_index()
    assert n_pred == 6
    before = ctx.get_stats()["index_joins"]
    js, pats, filt = datagen.employee_queries(d)[q]
    got = ctx.star_join(js, pats, filt)
    assert ctx.get_stats()["index_joins"] == before + 1, "the index path must have been taken"
    want = db.bgp(pats, filt)
    H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), q)
    # a filter on the PROBE-side pattern and one spanning two patterns
    js, pats, _ = datagen.employee_queries(d)["cfg2"]
    f2 = [c.fop(c.F_CMP_NUM, slot=2, cmp=c.CMP_GT, value=60000.0), c.fop(c.F_EQ_ID, slot=1, id=d.ids["Manager"]), c.fop(c.F_AND),
          c.fop(c.F_NE_ID, slot=3, id=int(d.s[0])), c.fop(c.F_AND)]
    got = ctx.star_join(js, pats, f2)
    want = db.bgp(pats, f2)
    H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), "compound filter")
    # an append that repeats existing subjects makes the predicates multi-valued: the maintained index loses its tables for them and
    # the query must still agree with the oracle on the new store (a delete drops the index altogether)
    ctx.store_append(d.s[:6], d.p[:6], d.o[:6], tag=77)
    got = ctx.star_join(js, pats, filt if q != "cfg1" else None)
    s2, p2, o2 = np.concatenate([d.s, d.s[:6]]), np.concatenate([d.p, d.p[:6]]), np.concatenate([d.o, d.o[:6]])
    want = O.Db(s2, p2, o2, d.num_or0, d.is_num).bgp(pats, filt if q != "cfg1" else None)
    H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), "after a duplicating append")
    ctx.store_delete(d.s[:6], d.p[:6], d.o[:6])
    n0 = ctx.get_stats()["index_joins"]
    ctx.star_join(js, pats, filt if q != "cfg1" else None)
    assert ctx.get_stats()["index_joins"] == n0, "a delete drops the index: the next query scans"


def test_index_path_multivalued_and_missing_predicate(ctx):
    rng = np.random.default_rng(5)
    n = 5000
    tr = np.unique(np.stack([rng.integers(0, 700, n), rng.integers(100, 103, n), rng.integers(1000, 1040, n)], axis=1).astype(np.uint32), axis=0)
    ctx.store_load(tr[:, 0], tr[:, 1], tr[:, 2])
    assert ctx.build_index()[0] == 3
    db = O.Db(tr[:, 0], tr[:, 1], tr[:, 2])
    pats = [c.pattern(c.V(0), c.K(100), c.V(1)), c.pattern(c.V(0), c.K(101), c.V(2)), c.pattern(c.V(0), c.K(102), c.V(3))]
    want = db.bgp(pats).to_numpy([0, 1, 2, 3])
    for _ in range(2):
        H.assert_same_bag(ctx.star_join(0, pats).to_numpy([0, 1, 2, 3]), want, "1:N star with index")
    none = ctx.star_join(0, [c.pattern(c.V(0), c.K(100), c.V(1)), c.pattern(c.V(0), c.K(999), c.V(2))])
    assert none.n_rows == 0 and sorted(none.slots) == [0, 1, 2]
    # object-keyed star: ?a P1 ?x . ?b P2 ?x joined on the object
    pats_o = [c.pattern(c.V(1), c.K(100), c.V(0)), c.pattern(c.V(2), c.K(101), c.V(0))]
    H.assert_same_bag(ctx.star_join(0, pats_o).to_numpy([0, 1, 2]), db.bgp(pats_o).to_numpy([0, 1, 2]), "object star")


@pytest.mark.parametrize("n_subj", [1, 1023, 1024, 3017, 40000])
def test_index_kernel_shapes(ctx, n_subj):
    """the one-launch index join (probe_index_kernel): every build side is a persistent table. T = 1..4 tables, typed / general /
    no pre-filter on the probe slice, filters on looked-up values, object-keyed joins, ragged last tiles, and the self-cleaning
    control block across many launches in a row"""
    rng = np.random.default_rng(n_subj)
    subj = np.arange(50, 50 + n_subj, dtype=np.uint32)
    base = 50 + n_subj
    vals = np.arange(base, base + 64, dtype=np.uint32)            # 64 numeric literals
    uniq = base + 64 + rng.permutation(n_subj).astype(np.uint32)  # a unique, dense object per subject (inverse functional)
    few = np.arange(base + 64 + n_subj, base + 64 + n_subj + 3, dtype=np.uint32)
    n_ids = int(few[-1]) + 1
    num = np.zeros(n_ids)
    isn = np.zeros(n_ids, np.uint8)
    num[vals] = np.linspace(-5.0, 250.5, 64)
    isn[vals] = 1
    cols = []
    for pid, ob in ((100, vals[rng.integers(0, 64, n_subj)]), (101, uniq), (102, few[rng.integers(0, 3, n_subj)]), (103, vals[rng.integers(0, 64, n_subj)]),
                    (104, few[rng.integers(0, 3, n_subj)])):
        keep = np.ones(n_subj, bool) if pid != 103 else rng.random(n_subj) < 0.7  # P103 is missing for ~30 % of the subjects
        cols.append(np.stack([subj[keep], np.full(keep.sum(), pid, np.uint32), ob[keep]], axis=1))
    tr = np.concatenate(cols).astype(np.uint32)
    tr = tr[rng.permutation(len(tr))]
    ctx.dict_numeric_load(num, isn)
    ctx.store_load(tr[:, 0], tr[:, 1], tr[:, 2])
    assert ctx.build_index()[0] == 5
    db = O.Db(tr[:, 0], tr[:, 1], tr[:, 2], num, isn)
    P = lambda pid, v: c.pattern(c.V(0), c.K(pid), c.V(v))
    gt = lambda slot, v: [c.fop(c.F_CMP_NUM, slot=slot, cmp=c.CMP_GT, value=v)]
    cases = [
        ("T1 no filter", [P(100, 1), P(101, 2)], None),
        ("T2 typed pre-filter", [P(101, 1), P(100, 2), P(102, 3)], gt(2, 100.0)),
        ("T2 typed <=", [P(101, 1), P(100, 2), P(102, 3)], [c.fop(c.F_CMP_NUM, slot=2, cmp=c.CMP_LE, value=17.25)]),
        ("T3 partial predicate", [P(100, 1), P(101, 2), P(102, 3), P(103, 4)], gt(1, 0.0)),
        ("T4 everything", [P(100, 1), P(101, 2), P(102, 3), P(103, 4), P(104, 5)], None),
        ("general pre-filter (id equality AND numeric)", [P(102, 1), P(100, 2)], [c.fop(c.F_EQ_ID, slot=1, id=int(few[1])), c.fop(c.F_CMP_NUM, slot=2, cmp=c.CMP_LT, value=200.0), c.fop(c.F_AND)]),
        ("filter spanning two patterns", [P(100, 1), P(103, 2), P(101, 3)], [c.fop(c.F_PUSH_VAR, slot=1), c.fop(c.F_PUSH_VAR, slot=2), c.fop(c.F_SUB), c.fop(c.F_TRUTHY)]),
        ("two numeric filters on different patterns", [P(100, 1), P(103, 2), P(102, 3)], gt(1, 50.0) + gt(2, 20.0) + [c.fop(c.F_AND)]),
        ("filter on the subject", [P(100, 1), P(102, 2)], [c.fop(c.F_NE_ID, slot=0, id=int(subj[0]))]),
    ]
    before = ctx.get_stats()["index_joins"]
    for name, pats, filt in cases:
        for rep in range(2):  # the second launch starts from the control block the first one left behind
            got = ctx.star_join(0, pats, filt)
            want = db.bgp(pats, filt)
            H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), f"{name} (n={n_subj}, rep {rep})")
    assert ctx.get_stats()["index_joins"] == before + 2 * len(cases)
    # object-keyed: ?a P101 ?x . ?b P101 ?x (the persistent table is ytab)
    pats_o = [c.pattern(c.V(1), c.K(101), c.V(0)), c.pattern(c.V(2), c.K(101), c.V(0))]
    got = ctx.star_join(0, pats_o)
    H.assert_same_bag(got.to_numpy([0, 1, 2]), db.bgp(pats_o).to_numpy([0, 1, 2]), "object-keyed")
    # a scan-path query in between must not disturb the control block
    ctx.set_use_index(False)
    r = ctx.star_join(0, cases[1][1], cases[1][2])
    ctx.set_use_index(True)
    got = ctx.star_join(0, cases[1][1], cases[1][2])
    H.assert_same_bag(got.to_numpy(sorted(got.slots)), r.to_numpy(sorted(r.slots)), "index vs scan path")


@pytest.mark.parametrize("cmp", [c.CMP_GT, c.CMP_GE, c.CMP_LT, c.CMP_LE])
def test_star_scan_filter_boundaries(ctx, emp, cmp):
    """the star-shape scan kernel evaluates a strict comparison as a non-strict one against the neighbouring double: constants that
    equal stored values, infinities, NaN and signed zeros must still give the oracle's rows (scan path: index off)"""
    d, db = emp
    js, pats, _ = datagen.employee_queries(d)["cfg2"]
    present = float(d.salary_of_employee[7])
    for value in (present, present + 0.5, 30000.0, 149999.0, 0.0, -0.0, float("inf"), float("-inf"), float("nan"), 1e300, -1e300, 5e-324):
        filt = [c.fop(c.F_CMP_NUM, slot=2, cmp=cmp, value=value)]
        got = ctx.star_join(js, pats, filt)
        want = db.bgp(pats, filt)
        H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), f"cmp {cmp} value {value}")


def test_index_lookups_replace_scans(ctx):
    """IndexScan with a bound subject or object (index_manager.rs:253-340 cases; engine.rs:1248-1407): with the store index valid,
    (c P ?o), (?s P c) and (?s P ?o) are answered from the predicate's slice — direct table for unique columns, key-grouped directory
    for multi-valued ones — and must not launch a scan kernel; answers = the oracle's scan"""
    rng = np.random.default_rng(21)
    n = 60000
    # predicate 100: functional (unique subjects); 101: multi-valued both ways; 102: sparse object ids (no directory -> scan)
    s100 = rng.permutation(20000)[:15000].astype(np.uint32) + 1000
    t100 = np.stack([s100, np.full(len(s100), 100), rng.integers(500, 900, len(s100))], axis=1)
    t101 = np.unique(np.stack([rng.integers(1000, 6000, n), np.full(n, 101), rng.integers(2000, 7000, n)], axis=1), axis=0)
    t102 = np.unique(np.stack([rng.integers(1000, 3000, 4000), np.full(4000, 102), rng.integers(0, 1 << 30, 4000)], axis=1), axis=0)
    tr = np.concatenate([t100, t101, t102]).astype(np.uint32)
    tr = tr[rng.permutation(len(tr))]
    ctx.store_load(tr[:, 0], tr[:, 1], tr[:, 2])
    db = O.Db(tr[:, 0], tr[:, 1], tr[:, 2])
    ctx.build_index()
    X, Y = 0, 1
    some_s100, some_s101, some_o101, some_o100 = int(s100[7]), int(t101[5, 0]), int(t101[9, 2]), int(t100[3, 2])
    cases = [("functional, bound subject", c.pattern(c.K(some_s100), c.K(100), c.V(Y)), True),
             ("functional, bound subject absent", c.pattern(c.K(999999), c.K(100), c.V(Y)), True),
             ("functional predicate, bound object (many subjects)", c.pattern(c.V(X), c.K(100), c.K(some_o100)), True),
             ("multi-valued, bound subject", c.pattern(c.K(some_s101), c.K(101), c.V(Y)), True),
             ("multi-valued, bound object", c.pattern(c.V(X), c.K(101), c.K(some_o101)), True),
             ("multi-valued, bound object absent", c.pattern(c.V(X), c.K(101), c.K(1)), True),
             ("whole slice", c.pattern(c.V(X), c.K(101), c.V(Y)), True),
             ("predicate absent", c.pattern(c.V(X), c.K(555), c.V(Y)), True),
             ("sparse objects, bound subject", c.pattern(c.K(int(t102[0, 0])), c.K(102), c.V(Y)), True),
             ("sparse objects, bound object: no directory", c.pattern(c.V(X), c.K(102), c.K(int(t102[0, 2]))), False),
             ("variable predicate", c.pattern(c.K(some_s101), c.V(Y), c.V(X)), False)]
    for what, pat, by_index in cases:
        scans0 = ctx.get_stats()["scan_launches"]
        got = ctx.scan([pat])[0]
        want = db.scan(pat)
        H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), what)
        launched = ctx.get_stats()["scan_launches"] - scans0
        if by_index and "whole slice" not in what:
            assert launched == 0, f"{what}: a scan kernel ran"
        if not by_index:
            assert launched >= 1, what
    # several patterns in one call: looked-up and scanned patterns mix; a pushed-down FILTER applies to looked-up rows too
    pats = [c.pattern(c.K(some_s101), c.K(101), c.V(Y)), c.pattern(c.V(X), c.V(2), c.K(some_o101)), c.pattern(c.V(X), c.K(100), c.V(Y))]
    flt = [None, None, [c.fop(c.F_NE_ID, slot=Y, id=some_o100)]]
    got = ctx.scan(pats, flt)
    for k in range(3):
        want = db.scan(pats[k], flt[k])
        H.assert_same_bag(got[k].to_numpy(sorted(got[k].slots)), want.to_numpy(sorted(want.slots)), f"mixed {k}")
    # a BGP whose patterns do not share one variable (left-deep joins over looked-up inputs)
    bgp = [c.pattern(c.K(some_s101), c.K(101), c.V(Y)), c.pattern(c.V(X), c.K(101), c.V(Y))]
    got = ctx.bgp_execute(bgp)
    want = db.bgp(bgp)
    H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), "path BGP")


def test_join_heavy_hitters_spread_over_the_grid(ctx):
    """1:N join whose fan-out is concentrated on a few probe rows (the transitive rule's join on the ancestor column, join_algorithm.rs:
    499-677 over a class tree): tiles whose expansion exceeds 32 768 rows are recorded and expanded by a second launch in pieces
    (probe_grouped_kernel<HEAVY>); same bag as the oracle, heavy keys adjacent, scattered, and mixed with ordinary rows"""
    rng = np.random.default_rng(23)
    n_build = 300_000
    bkey = rng.integers(100, 4000, n_build).astype(np.uint32)
    bkey[:120_000] = 7            # one key carried by 120 000 build rows
    bkey[120_000:170_000] = 9     # another by 50 000
    rng.shuffle(bkey)
    bpay = np.arange(n_build, dtype=np.uint32)
    for label, pkey in (("adjacent heavy rows", np.concatenate([np.full(20, 7), np.full(10, 9), rng.integers(100, 4000, 5000)])),
                        ("scattered heavy rows", rng.permutation(np.concatenate([np.full(12, 7), np.full(25, 9), rng.integers(0, 4000, 40000)]))),
                        ("one heavy row", np.concatenate([rng.integers(100, 4000, 2000), [7], rng.integers(100, 4000, 2000)]))):
        pkey = pkey.astype(np.uint32)
        ppay = np.arange(len(pkey), dtype=np.uint32) + 1_000_000
        gl, ol = ctx.rel_from_host([0, 1], [ppay, pkey]), O.rel_from_host([0, 1], [ppay, pkey])
        gr, orr = ctx.rel_from_host([1, 2], [bkey, bpay]), O.rel_from_host([1, 2], [bkey, bpay])
        got = ctx.hash_join(gl, gr)
        want = O.hash_join(ol, orr)
        assert got.n_rows == want.n_rows and got.n_rows > 200_000, label
        H.assert_same_bag(got.to_numpy(sorted(got.slots)), want.to_numpy(sorted(want.slots)), label)
