"""Parity tests proper: the CUDA path (through the C ABI) against the oracle, the committed golden vectors
and -- when the prebuilt reference library travelled with the repo -- the unmodified reference itself.
Bar: bit-exact (all arithmetic is u16/u32/u64 integer)."""
import numpy as np
import pytest

import bitmagic_b200 as bm
import gen
import golden_util as gu
import orclib
import refanswers as ra
from refanswers import same

pytestmark = pytest.mark.gpu

C = bm.F_OPT_COMPRESS


def gpu_aggregate(ctx, ps, op, g0, g1, flags, dset=None):
    own = dset is None
    if own:
        dset = bm.DeviceSet.upload(ctx, ps)
    res = bm.aggregate(ctx, dset, op, g0, g1, flags)
    kind, pop, dig, nr = res.meta()
    total, any_ = res.total()
    fk, off, bits, gaps = res.fetch()
    assert np.array_equal(fk, kind)
    bv = bm.result_to_bvector(fk, off, bits, gaps)
    blocks = np.stack([bv.block_words(c) for c in range(kind.size)])
    gflat = np.concatenate([bv.blocks[c] for c in range(kind.size) if kind[c] == bm.BLK_GAP]) \
        if (kind == bm.BLK_GAP).any() else np.zeros(0, np.uint16)
    res.free()
    if own:
        dset.free()
    return dict(kind=kind, pop=pop, dig=dig, nr=nr, total=total, any=any_, blocks=blocks, gflat=gflat)


def check_vs_oracle(ctx, ps, op, g0, g1, flags, dset=None):
    got = gpu_aggregate(ctx, ps, op, g0, g1, flags, dset)
    okind, opop, odig, onr, oblk, ogap = orclib.oracle_aggregate(ps, op, g0, g1, flags)
    assert np.array_equal(got["blocks"], oblk)
    assert np.array_equal(got["pop"], opop)
    assert np.array_equal(got["dig"], odig)
    assert np.array_equal(got["nr"], onr)
    assert np.array_equal(got["kind"], okind)
    assert got["total"] == int(opop.sum()) and got["any"] == bool(opop.sum())
    glen = np.where(okind == bm.BLK_GAP, (ogap[:, 0] >> 3) + 1, 0)
    oflat = np.concatenate([ogap[c, :glen[c]] for c in range(len(okind))]) if glen.sum() else np.zeros(0, np.uint16)
    assert np.array_equal(got["gflat"], oflat)
    return got


@pytest.mark.parametrize("name", ["agg_mixed", "agg_edge", "agg_zipf"])
def test_aggregate_vs_golden(ctx, name):
    ps, cases = gu.load_agg(name)
    dset = bm.DeviceSet.upload(ctx, ps)
    for case in cases:
        got = gpu_aggregate(ctx, ps, case["op"], case["g0"], case["g1"], case["flags"], dset)
        xor = case["op"] == bm.OP_XOR
        gu.check_agg_case(case, got["kind"], got["pop"], got["blocks"], None if xor else got["gflat"], check_kind=not xor)
        assert got["any"] == case["any"]
    dset.free()


@pytest.mark.parametrize("op", [bm.OP_OR, bm.OP_AND, bm.OP_AND_SUB, bm.OP_XOR])
@pytest.mark.parametrize("seed", [1, 2])
def test_aggregate_random_mixed_vs_oracle(ctx, op, seed):
    rng = np.random.default_rng(100 * op + seed)
    kw = dict(p_null=0.04, p_full=0.03) if op in (bm.OP_AND, bm.OP_AND_SUB) else {}
    vecs = gen.mixed_vectors(rng, 24, 9, **kw)
    ps = bm.PackedSet.pack(vecs)
    dset = bm.DeviceSet.upload(ctx, ps)
    for trial in range(4):
        perm = rng.permutation(24)
        if op == bm.OP_AND_SUB:
            na = int(rng.integers(1, 4)); g0, g1 = perm[:na], perm[na:na + int(rng.integers(0, 20))]
        elif op == bm.OP_AND:
            g0, g1 = perm[: int(rng.integers(1, 5))], None
        else:
            g0, g1 = perm[: int(rng.integers(1, 25))], None
        for flags in (0, C):
            check_vs_oracle(ctx, ps, op, g0, g1, flags, dset)
    dset.free()


def test_gap_stream_and_gather_paths_agree(ctx):
    """Sorted member lists take the TMA-streamed GAP path, tuning key 0 = 1 forces the gather path: same bits."""
    rng = np.random.default_rng(8)
    vecs = [bm.BVector.random(4, 0.4 / (k + 1), rng).optimize() for k in range(300)]
    vecs[7].set_full(1)
    ps = bm.PackedSet.pack(vecs)
    dset = bm.DeviceSet.upload(ctx, ps)
    try:
        for mode in (0, 1):
            ctx.set_tuning(0, mode)
            check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [0, 1], list(range(2, 300)), C, dset)
            check_vs_oracle(ctx, ps, bm.OP_OR, list(range(100, 300)), None, C, dset)
            check_vs_oracle(ctx, ps, bm.OP_AND, [280, 290, 299], None, 0, dset)          # GAP sources in the AND group
            check_vs_oracle(ctx, ps, bm.OP_AND_SUB, list(range(250, 254)), list(range(100, 250)), C, dset)  # both lists streamed
            check_vs_oracle(ctx, ps, bm.OP_XOR, list(range(60, 300)), None, 0, dset)
            check_vs_oracle(ctx, ps, bm.OP_OR, list(range(299, 99, -1)), None, 0, dset)   # descending -> gather
            check_vs_oracle(ctx, ps, bm.OP_OR, [100, 299], None, 0, dset)                 # sparse subset -> gather
            check_vs_oracle(ctx, ps, bm.OP_OR, list(range(100, 300, 2)), None, C, dset)   # non-members inside the window -> per-block stream
            check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [0, 150], list(range(100, 300)), C, dset)   # an AND member inside the SUB window
            check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [3], list(range(60, 300)) + [5], C, dset)   # unsorted tail member
    finally:
        ctx.set_tuning(0, 0)
    dset.free()


def test_gap_flat_and_raw_formats(ctx):
    """BMB200_DESC_GAP_FLAT / _PAD: GAP blocks in the flat-streamable form (lead pad 0xFFFF iff first run is 0) and raw
    GAP blocks must give identical results everywhere (aggregate flat / stream / gather paths, rs_index build, rank, select)."""
    rng = np.random.default_rng(21)
    vecs = gen.mixed_vectors(rng, 20, 5, p_null=0.05, p_gap=0.7) + gen.edge_vectors(5)
    plain, padded = bm.PackedSet.pack(vecs, gap_flat=False), bm.PackedSet.pack(vecs)
    assert (padded.desc >> 31).any() and not (plain.desc >> 30).any()
    isgap = (padded.desc & 3) == bm.BLK_GAP
    assert ((padded.desc[isgap] >> 30) & 1).all() and not (padded.desc[isgap] >> 31).all()   # first-run-1 blocks carry no pad
    d0, d1 = bm.DeviceSet.upload(ctx, plain), bm.DeviceSet.upload(ctx, padded)
    n = len(vecs)
    for op, g0, g1 in [(bm.OP_OR, list(range(n)), None), (bm.OP_AND_SUB, [0, 1], list(range(2, n))), (bm.OP_AND, [3, 4, 5], None),
                       (bm.OP_XOR, list(range(n)), None), (bm.OP_OR, list(range(n - 1, -1, -1)), None)]:
        a = gpu_aggregate(ctx, plain, op, g0, g1, C, d0)
        b = check_vs_oracle(ctx, padded, op, g0, g1, C, d1)
        assert np.array_equal(a["blocks"], b["blocks"]) and np.array_equal(a["kind"], b["kind"])
    for v in (0, 7, n - 2):
        r0, r1 = bm.DeviceRS(ctx, d0, v), bm.DeviceRS(ctx, d1, v)
        for x, y in zip(r0.export(), r1.export()):
            assert np.array_equal(x, y)
        pos = rng.integers(0, 5 * 65536, 2000).astype(np.uint64)
        assert np.array_equal(r0.rank(pos), r1.rank(pos))
        rk = rng.integers(0, r0.total() + 2, 2000).astype(np.uint64)
        (p0, f0), (p1, f1) = r0.select(rk), r1.select(rk)
        assert np.array_equal(f0, f1) and np.array_equal(p0[f0], p1[f1])
        r0.free(); r1.free()
    d0.free(); d1.free()


@pytest.mark.parametrize("seed", [3, 4])
def test_flat_window_all_gap_styles(ctx, seed):
    """The FLAT consumer (whole-pool OR / SUB groups, >= 16 GAP blocks per column) on every GAP style the generator knows:
    sparse bits, few long runs (multi-word runs), ~1270 runs, word-aligned runs, mostly-ones blocks (first run = 1, long
    runs), all-zero / all-one GAP blocks; dense and sparse live masks (test-first and always-atomic modes)."""
    rng = np.random.default_rng(seed)
    vecs = gen.mixed_vectors(rng, 56, 6, p_null=0.03, p_full=0.0, p_gap=0.85) + gen.edge_vectors(6)[:2]
    dense = bm.BVector(6)
    for nb in range(6):
        dense.set_bits(nb, rng.integers(0, 2**32, 2048, dtype=np.uint64).astype(np.uint32) | rng.integers(0, 2**32, 2048, dtype=np.uint64).astype(np.uint32))
    sparse = bm.BVector.random(6, 0.02, rng)
    vecs = [dense, sparse] + vecs
    n = len(vecs)
    ps = bm.PackedSet.pack(vecs)
    raw = bm.PackedSet.pack(vecs, gap_flat=False)
    dset, draw = bm.DeviceSet.upload(ctx, ps), bm.DeviceSet.upload(ctx, raw)
    for op, g0, g1 in [(bm.OP_OR, list(range(2, n)), None), (bm.OP_OR, list(range(1, n)), None),
                       (bm.OP_AND_SUB, [0], list(range(2, n))), (bm.OP_AND_SUB, [1], list(range(2, n))),
                       (bm.OP_AND_SUB, [0, 1], list(range(2, n))), (bm.OP_AND_SUB, [0], list(range(10, 40)))]:
        for flags in (0, C):
            a = check_vs_oracle(ctx, ps, op, g0, g1, flags, dset)
            b = gpu_aggregate(ctx, raw, op, g0, g1, flags, draw)
            assert np.array_equal(a["blocks"], b["blocks"]) and np.array_equal(a["kind"], b["kind"])
    dset.free(); draw.free()


def test_pipeline_batch(ctx):
    """bmb200_aggregate_batch (aggregator::pipeline): every group equals its own single aggregate / the oracle;
    counts, OR target, counts-only mode; and the unmodified reference pipeline when its library is present."""
    rng = np.random.default_rng(31)
    vecs = gen.mixed_vectors(rng, 18, 6, p_null=0.05, p_full=0.03)
    ps = bm.PackedSet.pack(vecs)
    dset = bm.DeviceSet.upload(ctx, ps)
    groups = []
    for _ in range(9):
        perm = rng.permutation(18)
        na = int(rng.integers(1, 4)); ns = int(rng.integers(0, 8))
        groups.append((sorted(perm[:na].tolist()), sorted(perm[na:na + ns].tolist())))
    groups.append(([0], []))
    groups.append(([2, 3], [2]))                      # empty by construction
    nb = ps.n_blocks
    res = bm.aggregate_batch(ctx, dset, bm.OP_AND_SUB, groups, C | bm.F_OR_TARGET)
    kind, pop, dig, nr = res.meta()
    totals = res.group_totals(len(groups))
    fk, off, bits, gaps = res.fetch()
    union = np.zeros((nb, 2048), np.uint32)
    for g, (g0, g1) in enumerate(groups):
        okind, opop, odig, onr, oblk, ogap = orclib.oracle_aggregate(ps, bm.OP_AND_SUB, g0, g1, C)
        sl = slice(g * nb, (g + 1) * nb)
        assert np.array_equal(kind[sl], okind) and np.array_equal(pop[sl], opop) and np.array_equal(dig[sl], odig) and np.array_equal(nr[sl], onr)
        assert totals[g] == int(opop.sum())
        bv = bm.result_to_bvector(fk[sl], off[sl], bits, gaps)
        assert np.array_equal(np.stack([bv.block_words(c) for c in range(nb)]), oblk)
        union |= oblk
    o = res.or_target(nb)
    obv = bm.result_to_bvector(*o.fetch())
    assert np.array_equal(np.stack([obv.block_words(c) for c in range(nb)]), union)
    o.free(); res.free()
    # counts only
    res = bm.aggregate_batch(ctx, dset, bm.OP_AND_SUB, groups, bm.F_COUNT_ONLY)
    assert np.array_equal(res.group_totals(len(groups)), totals)
    res.free()
    # host mirror: Pipeline / Aggregator.combine_and_sub(pipeline)
    pipe = bm.Pipeline(make_results=True, compute_counts=True)
    for g0, g1 in groups:
        a = pipe.add()
        for v in g0: a.add(vecs[v], 0)
        for v in g1: a.add(vecs[v], 1)
    pipe.set_or_target()
    pipe.complete()
    bm.Aggregator(ctx).combine_and_sub(pipe)
    assert pipe.get_bv_count_vector() == [int(t) for t in totals]
    assert pipe.get_bv_res_vector()[-1] is None and pipe.get_bv_res_vector()[0] is not None
    assert np.array_equal(np.stack([pipe.or_target.block_words(c) for c in range(nb)]), union)
    rc, rkind, rpop, rblk, rok, rob = ra.ref_pipeline(ps, groups, want_or=True)
    assert same(rc, totals)
    assert same(rblk, np.stack([
        np.stack([bm.result_to_bvector(fk[g * nb:(g + 1) * nb], off[g * nb:(g + 1) * nb], bits, gaps).block_words(c) for c in range(nb)])
        for g in range(len(groups))]))
    assert same(rob, union)
    dset.free()


def test_edge_cases(ctx):
    vecs = gen.edge_vectors(4)
    ps = bm.PackedSet.pack(vecs)
    dset = bm.DeviceSet.upload(ctx, ps)
    n = len(vecs)
    cases = [(bm.OP_OR, list(range(n)), None), (bm.OP_OR, [0, 1], None), (bm.OP_OR, [5], None), (bm.OP_OR, [3, 4], None),
             (bm.OP_OR, [2, 2], None), (bm.OP_AND, [2, 3], None), (bm.OP_AND, [0, 2], None), (bm.OP_AND, [2, 2], None),
             (bm.OP_AND, [5, 2], None), (bm.OP_AND_SUB, [2], [0]), (bm.OP_AND_SUB, [2], [5]), (bm.OP_AND_SUB, [2, 3], [1, 4]),
             (bm.OP_AND_SUB, [3], [2]), (bm.OP_AND_SUB, [1], []), (bm.OP_AND_SUB, [2], [1]), (bm.OP_XOR, [2, 3], None),
             (bm.OP_XOR, [0, 1, 4], None), (bm.OP_XOR, [2, 2], None), (bm.OP_XOR, [5], None)]
    for op, g0, g1 in cases:
        for flags in (0, C):
            check_vs_oracle(ctx, ps, op, g0, g1, flags, dset)
    # count-only mode returns the same totals and stores nothing
    res = bm.aggregate(ctx, dset, bm.OP_AND_SUB, [2, 3], [1, 4], bm.F_COUNT_ONLY)
    _, opop, *_ = orclib.oracle_aggregate(ps, bm.OP_AND_SUB, [2, 3], [1, 4], 0)
    assert res.total()[0] == int(opop.sum())
    assert np.array_equal(res.meta()[1], opop)
    res.free()
    # column sub-range
    res = bm.aggregate(ctx, dset, bm.OP_OR, list(range(n)), None, 0, nb_from=1, nb_to=3)
    _, opop, *_ = orclib.oracle_aggregate(ps, bm.OP_OR, list(range(n)), None, 0, 1, 3)
    assert np.array_equal(res.meta()[1], opop)
    res.free()
    dset.free()


def test_large_groups_chunked_classification(ctx):
    """> 1024 group members exercises the multi-chunk classification path; duplicates are legal."""
    rng = np.random.default_rng(42)
    vecs = [bm.BVector.random(3, 0.02 / (1 + k % 7), rng) for k in range(40)]
    for k in range(10, 40):
        vecs[k].optimize()
    ps = bm.PackedSet.pack(vecs)
    dset = bm.DeviceSet.upload(ctx, ps)
    g = rng.integers(0, 40, 2500)
    check_vs_oracle(ctx, ps, bm.OP_OR, g, None, C, dset)
    check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [0, 1], g, C, dset)
    check_vs_oracle(ctx, ps, bm.OP_XOR, g[:1500], None, 0, dset)
    dset.free()


def test_flat_windows_over_several_classification_passes(ctx):
    """C5 shape in small: 2600 sparse GAP vectors -> three member passes per column, each streaming its own flat window;
    the live mask goes from dense (always-atomic form) to sparse (test-first form) inside one column."""
    nv, nbk = 2600, 2
    dens = np.full(nv, 0.0025)
    dens[::97] = 0.006
    seed = np.arange(7000, 7000 + nv, dtype=np.uint64)
    dset = bm.DeviceSet.synth(ctx, nv, nbk, dens, seed, True)
    ps = dset.download()
    assert (ps.kinds() == bm.BLK_GAP).all()
    check_vs_oracle(ctx, ps, bm.OP_OR, list(range(nv)), None, C, dset)
    check_vs_oracle(ctx, ps, bm.OP_OR, list(range(5, 2300)), None, 0, dset)
    check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [0, 1, 2], list(range(3, nv)), C, dset)
    check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [7], list(range(1000, 2400)), C, dset)
    dset.free()


def test_upload_vectors_and_host_mirror_api(ctx):
    """bm::aggregator-style surface: add/combine_*; 2-operand bit_*; count_*."""
    rng = np.random.default_rng(9)
    vecs = gen.mixed_vectors(rng, 8, 4)
    ps = bm.PackedSet.pack(vecs)
    agg = bm.Aggregator(ctx)
    for v in vecs[:5]:
        agg.add(v)
    for v in vecs[5:]:
        agg.add(v, 1)
    agg.set_optimization(bm.OPT_COMPRESS)
    t = agg.combine_or()
    _, _, _, _, oblk, _ = orclib.oracle_aggregate(ps, bm.OP_OR, range(5), None, C)
    assert np.array_equal(np.stack([t.block_words(c) for c in range(4)]), oblk)
    t, found = agg.combine_and_sub()
    okind, opop, _, _, oblk, _ = orclib.oracle_aggregate(ps, bm.OP_AND_SUB, range(5), range(5, 8), C)
    assert np.array_equal(np.stack([t.block_words(c) for c in range(4)]), oblk) and found == bool(opop.sum())
    assert np.array_equal(t.kind, okind)
    a, b = vecs[0], vecs[1]
    for f, op, g0, g1 in [(bm.bit_and, bm.OP_AND, [0, 1], None), (bm.bit_or, bm.OP_OR, [0, 1], None),
                          (bm.bit_xor, bm.OP_XOR, [0, 1], None), (bm.bit_sub, bm.OP_AND_SUB, [0], [1])]:
        r = f(a, b, ctx=ctx)
        _, opop, _, _, oblk, _ = orclib.oracle_aggregate(ps, op, g0, g1, 0)
        assert np.array_equal(np.stack([r.block_words(c) for c in range(4)]), oblk)
        assert r.count() == int(opop.sum())
    assert bm.count_and(a, b, ctx=ctx) == int(orclib.oracle_aggregate(ps, bm.OP_AND, [0, 1], None, 0)[1].sum())
    assert bm.count_sub(a, b, ctx=ctx) == int(orclib.oracle_aggregate(ps, bm.OP_AND_SUB, [0], [1], 0)[1].sum())
    assert agg.combine_or([]).n_blocks == 0 and agg.combine_and_sub([], [])[1] is False


def test_aggregate_host_end_to_end_call(ctx):
    rng = np.random.default_rng(3)
    ps = bm.PackedSet.pack(gen.mixed_vectors(rng, 10, 6))
    kind, pop, dig, nr, total = bm.aggregate_host(ctx, ps, bm.OP_AND_SUB, [0, 1], list(range(2, 10)), C)
    okind, opop, odig, onr, *_ = orclib.oracle_aggregate(ps, bm.OP_AND_SUB, [0, 1], list(range(2, 10)), C)
    assert np.array_equal(kind, okind) and np.array_equal(pop, opop) and np.array_equal(dig, odig) and total == int(opop.sum())


def test_rs_index_rank_select_vs_golden(ctx):
    ps, vs = gu.load_rs("rs_mixed")
    dset = bm.DeviceSet.upload(ctx, ps)
    for v, g in enumerate(vs):
        rs = bm.DeviceRS(ctx, dset, v)
        bc, sc, sb = rs.export()
        assert rs.total() == int(g["total"])
        if int(g["total"]):
            assert np.array_equal(bc, g["bcount"])
            nz = g["bcount"] > 0
            assert np.array_equal(sc[nz], g["sub"][nz])
            assert np.array_equal(sb, g["sb"])
        assert np.array_equal(rs.rank(g["pos"]), g["rank_out"]) or int(g["total"]) == 0
        pos, found = rs.select(g["rank"])
        assert np.array_equal(found, g["sel_found"])
        assert np.array_equal(pos[found], g["sel_pos"][g["sel_found"]])
        rs.free()
    dset.free()


def test_rs_index_vs_oracle_including_full_and_edges(ctx):
    rng = np.random.default_rng(17)
    vecs = gen.mixed_vectors(rng, 4, 300, p_null=0.3, p_full=0.15, p_gap=0.3)
    full = bm.BVector(300)
    for nb in range(300):
        full.set_full(nb)                       # RankFindTest: rank(i) == i+1, select(rank) == i  (t.cpp:4975-5090)
    vecs.append(full)
    ps = bm.PackedSet.pack(vecs)
    dset = bm.DeviceSet.upload(ctx, ps)
    for v in range(ps.n_vec):
        rs = bm.DeviceRS(ctx, dset, v)
        obc, osc, osb = orclib.oracle_rs_build(ps, v)
        bc, sc, sb = rs.export()
        assert np.array_equal(bc, obc) and np.array_equal(sc, osc) and np.array_equal(sb, osb)
        pos = np.concatenate([rng.integers(0, 300 * 65536, 5000), [0, 65535, 65536, 300 * 65536 - 1, 300 * 65536 + 5]]).astype(np.uint64)
        assert np.array_equal(rs.rank(pos), orclib.oracle_rank(ps, v, pos))
        tot = rs.total()
        rank = np.concatenate([rng.integers(0, tot + 2, 5000), [0, 1, tot, tot + 1]]).astype(np.uint64)
        p, f = rs.select(rank)
        op, of = orclib.oracle_select(ps, v, rank)
        assert np.array_equal(f, of) and np.array_equal(p[f], op[of])
        rs.free()
    i = rng.integers(0, 300 * 65536, 1000).astype(np.uint64)
    rs = bm.DeviceRS(ctx, dset, ps.n_vec - 1)
    assert np.array_equal(rs.rank(i), i + 1)
    p, f = rs.select(i + 1)
    assert f.all() and np.array_equal(p, i)
    rs.free()
    dset.free()


def test_synth_set_matches_its_own_contract(ctx):
    """The device generator: kinds follow optimize(), sizes add up, and aggregation over it matches the oracle."""
    nv, nbk = 64, 5
    dens = np.array([0.5 / (k + 1) for k in range(nv)])
    seed = np.arange(1000, 1000 + nv, dtype=np.uint64)
    dset = bm.DeviceSet.synth(ctx, nv, nbk, dens, seed, True)
    ps = dset.download()
    kinds = ps.kinds()
    assert (kinds[:, 0] == bm.BLK_BIT).all() and (kinds[:, -1] == bm.BLK_GAP).all()
    for v in range(nv):
        bv = ps.vector(v)
        d = bv.count() / (nbk * 65536)
        assert abs(d - dens[v]) < 0.02 + 0.1 * dens[v]
        for nb in range(nbk):
            k, data = ps.block(v, nb)
            if k == bm.BLK_GAP:
                assert (int(data[0]) >> 3) < 1276 and data[-1] == 65535 and (np.diff(data[1:].astype(int)) > 0).all()
            if k == bm.BLK_BIT:
                assert bm.hostfmt.calc_change(data) >= 1276
    check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [0, 1], list(range(2, nv)), C, dset)
    check_vs_oracle(ctx, ps, bm.OP_OR, list(range(nv)), None, 0, dset)
    d2 = bm.DeviceSet.synth(ctx, nv, nbk, dens, seed, True).download()    # deterministic
    assert np.array_equal(d2.bit_pool, ps.bit_pool) and np.array_equal(d2.gap_pool, ps.gap_pool)
    dset.free()


def test_against_unmodified_reference(ctx):
    rng = np.random.default_rng(77)
    vecs = gen.mixed_vectors(rng, 16, 6, p_null=0.05)
    ps = bm.PackedSet.pack(vecs)
    dset = bm.DeviceSet.upload(ctx, ps)
    for op, g0, g1, flags in [(bm.OP_OR, range(16), None, 0), (bm.OP_OR, range(16), None, C), (bm.OP_AND, [0, 1, 2], None, C),
                              (bm.OP_AND_SUB, [0, 1], range(2, 16), C)]:
        got = gpu_aggregate(ctx, ps, op, list(g0), list(g1) if g1 is not None else None, flags, dset)
        rkind, rpop, rblk, rgap, rany = ra.ref_aggregate(ps, op, list(g0), list(g1) if g1 is not None else None, flags)
        assert same(got["blocks"], rblk) and same(got["pop"], rpop) and same(got["kind"], rkind)
        assert got["any"] == rany
    dset.free()


def test_full_size_properties_c2_shape(ctx):
    """BASELINE config 2 shape at reduced vector count but full block geometry: size-independent properties
    (OR idempotence, AND-SUB subset/complement identities, checksum of popcounts vs sampled oracle columns)."""
    nv, nbk = 64, 512
    dens = np.full(nv, 0.05); seed = np.arange(100, 100 + nv, dtype=np.uint64)
    dset = bm.DeviceSet.synth(ctx, nv, nbk, dens, seed, False)
    r_or = bm.aggregate(ctx, dset, bm.OP_OR, np.arange(nv), None, 0)
    r_or2 = bm.aggregate(ctx, dset, bm.OP_OR, np.concatenate([np.arange(nv), np.arange(nv)]), None, 0)   # idempotent
    assert np.array_equal(r_or.meta()[1], r_or2.meta()[1])
    # |A| = |A & B| + |A - B|
    a = bm.aggregate(ctx, dset, bm.OP_OR, [0], None, bm.F_COUNT_ONLY).total()[0]
    ab = bm.aggregate(ctx, dset, bm.OP_AND, [0, 1], None, bm.F_COUNT_ONLY).total()[0]
    a_b = bm.aggregate(ctx, dset, bm.OP_AND_SUB, [0], [1], bm.F_COUNT_ONLY).total()[0]
    assert a == ab + a_b
    # |A ^ B| = |A | B| - |A & B|
    x = bm.aggregate(ctx, dset, bm.OP_XOR, [0, 1], None, bm.F_COUNT_ONLY).total()[0]
    o = bm.aggregate(ctx, dset, bm.OP_OR, [0, 1], None, bm.F_COUNT_ONLY).total()[0]
    assert x == o - ab
    # sampled columns against the oracle
    pop = r_or.meta()[1]
    for nb in (0, 255, 256, 511):
        ps = dset.download(nb, nb + 1)
        _, opop, *_ = orclib.oracle_aggregate(ps, bm.OP_OR, np.arange(nv), None, 0)
        assert pop[nb] == opop[0]
    dset.free()


def test_cxx_binding_against_reference_bvector_level():
    """bm::b200::aggregator<bm::bvector<>> (bitmagic_b200/include/bmb200_aggregator.hpp) vs bm::aggregator<> on real
    bvectors: compare()==0, calc_stat kinds, rs_index fields, and the reference's own count_to/select running on
    the GPU-built index.  The binary is built in the build container (it needs the reference headers)."""
    import subprocess
    exe = orclib.ORACLE_DIR / "_ref" / "test_cxx_binding"
    if not exe.exists():
        pytest.skip("oracle/_ref/test_cxx_binding not built (needs /root/reference at build time)")
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "OK:" in r.stdout


def test_more_than_65536_blocks_64bit_address_range(ctx):
    """n_blocks > 65536 (beyond the 32-bit address mode of the reference): aggregate + rs_index + rank/select vs the oracle."""
    nbk = 66000
    rng = np.random.default_rng(64)
    vs = []
    for k in range(3):
        v = bm.BVector(nbk)
        for nb in sorted(set(rng.integers(0, nbk, 40).tolist() + [0, 65535, 65536, nbk - 1])):
            w = hf_bits(rng, 0.01 * (k + 1))
            if k == 2:
                v.set_gap(nb, bm.hostfmt.bits_to_gap(hf_bits(rng, 0.001)))
            else:
                v.set_bits(nb, w)
        vs.append(v)
    vs[1].set_full(65537)
    ps = bm.PackedSet.pack(vs)
    dset = bm.DeviceSet.upload(ctx, ps)
    for op, g0, g1 in [(bm.OP_OR, [0, 1, 2], None), (bm.OP_AND_SUB, [0], [1, 2])]:
        res = bm.aggregate(ctx, dset, op, g0, g1, C)
        kind, pop, dig, nr = res.meta()
        okind, opop, odig, onr, _, _ = orclib.oracle_aggregate(ps, op, g0, g1, C)
        assert np.array_equal(kind, okind) and np.array_equal(pop, opop) and np.array_equal(dig, odig) and np.array_equal(nr, onr)
        res.free()
    rs = bm.DeviceRS(ctx, dset, 1)
    obc, osc, osb = orclib.oracle_rs_build(ps, 1)
    bc, sc, sb = rs.export()
    assert np.array_equal(bc, obc) and np.array_equal(sc, osc) and np.array_equal(sb, osb)
    pos = np.concatenate([rng.integers(0, nbk * 65536, 3000), [2**32 - 1, 2**32, 2**32 + 65536 + 5, nbk * 65536 - 1]]).astype(np.uint64)
    assert np.array_equal(rs.rank(pos), orclib.oracle_rank(ps, 1, pos))
    rank = rng.integers(0, rs.total() + 2, 3000).astype(np.uint64)
    p, f = rs.select(rank); op_, of = orclib.oracle_select(ps, 1, rank)
    assert np.array_equal(f, of) and np.array_equal(p[f], op_[of]) and int(p[f].max()) >= 2**32
    rs.rebuild()
    assert np.array_equal(rs.rank(pos), orclib.oracle_rank(ps, 1, pos))
    rs.free(); dset.free()


def hf_bits(rng, d):
    return bm.hostfmt.bits_to_words(rng.random(65536) < d)


def test_adopt_device_memory_and_no_leaks(ctx):
    """bmb200_set_adopt_device over torch-owned HBM; repeated create/free cycles return all device memory."""
    import ctypes as Cc
    import torch
    from bitmagic_b200 import capi
    rng = np.random.default_rng(5)
    ps = bm.PackedSet.pack(gen.mixed_vectors(rng, 8, 5))
    dev = torch.device("cuda:0")
    def up(a, pad=0):
        t = torch.zeros(a.nbytes + pad, dtype=torch.uint8, device=dev)
        t[: a.nbytes] = torch.from_numpy(a.view(np.uint8)).to(dev)
        return t
    t_desc, t_bb, t_gb = up(ps.desc), up(ps.bit_base), up(ps.gap_base)
    t_bp, t_gp = up(ps.bit_pool, 512), up(ps.gap_pool, 512)        # caller-owned pools need the 512-byte read slack
    c = capi.PackedSetC(ps.n_vec, ps.n_blocks, t_desc.data_ptr(), t_bb.data_ptr(), t_gb.data_ptr(), t_bp.data_ptr(), t_gp.data_ptr())
    h = Cc.c_void_p(0)
    ctx.check(capi.lib().bmb200_set_adopt_device(ctx._h, Cc.byref(c), Cc.byref(h)), "set_adopt_device")
    dset = capi.DeviceSet(ctx, h)
    g0, g1 = [0, 1], [2, 3, 4, 5, 6, 7]
    res = bm.aggregate(ctx, dset, bm.OP_AND_SUB, g0, g1, C)
    okind, opop, *_ = orclib.oracle_aggregate(ps, bm.OP_AND_SUB, g0, g1, C)
    kind, pop, _, _ = res.meta()
    assert np.array_equal(kind, okind) and np.array_equal(pop, opop)
    res.free(); dset.free()
    assert bool((t_bp[: ps.bit_pool.nbytes].cpu().numpy().view(np.uint32) == ps.bit_pool).all())   # adopted memory untouched, still owned by torch
    ctx.trim(); ctx.sync(); torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(20):
        d = bm.DeviceSet.upload(ctx, ps)
        r = bm.aggregate(ctx, d, bm.OP_OR, list(range(8)), None, C)
        rs = bm.DeviceRS(ctx, d, 3)
        r.fetch(); rs.rank(np.arange(10, dtype=np.uint64))
        rs.free(); r.free(); d.free()
    ctx.sync()
    assert torch.cuda.mem_get_info(0)[0] >= free0 - (4 << 20), "device memory leaked across create/free cycles"   # incl. the one parked arena
    ctx.trim()
    assert torch.cuda.mem_get_info(0)[0] >= free0 - (2 << 20)


def check_scan(ctx, ps, dset, pred, search, plane0, npl, uni, flags=C):
    res = bm.scan(ctx, dset, pred, search, plane0, npl, uni, flags)
    kind, pop, dig, nr = res.meta()
    nv = len(search)
    tot = res.group_totals(nv)
    fk, off, bits, gaps = res.fetch()
    bv = bm.result_to_bvector(fk, off, bits, gaps)
    blocks = np.stack([bv.block_words(c) for c in range(kind.size)])
    res.free()
    okind, opop, odig, onr, oblk, ogap = orclib.oracle_scan(ps, pred, search, plane0, npl, uni, flags)
    assert np.array_equal(blocks, oblk), f"scan pred {pred}: bits differ"
    assert np.array_equal(pop, opop) and np.array_equal(dig, odig) and np.array_equal(nr, onr) and np.array_equal(kind, okind)
    assert np.array_equal(tot, opop.reshape(nv, -1).sum(1))
    for c in np.nonzero(okind == bm.BLK_GAP)[0]:
        n = (int(ogap[c, 0]) >> 3) + 1
        assert np.array_equal(bv.blocks[c], ogap[c, :n])
    return blocks


def test_scan_vs_oracle_random_planes(ctx):
    """bmb200_scan on planes of every block kind (NULL / FULL / bit / GAP, both GAP storage forms), plane window inside a larger
    set, universe given / absent, 1..40 planes, values above the top plane."""
    import test_oracle_vs_reference as tor
    rng = np.random.default_rng(77)
    vecs = gen.mixed_vectors(rng, 44, 3, p_null=0.15, p_full=0.1, p_gap=0.45)
    for flat in (True, False):
        ps = bm.PackedSet.pack(vecs, gap_flat=flat)
        dset = bm.DeviceSet.upload(ctx, ps)
        for plane0, npl, uni in [(2, 40, 43), (0, 7, 1), (10, 1, bm.NO_UNIVERSE), (5, 13, bm.NO_UNIVERSE)]:
            top = (1 << npl) - 1
            vals = [0, 1, top, top // 3, int(rng.integers(0, top + 1)), top + 1 if npl < 64 else top]
            for pred in (bm.SCAN_EQ, bm.SCAN_GT, bm.SCAN_GE, bm.SCAN_LT, bm.SCAN_LE):
                check_scan(ctx, ps, dset, pred, vals, plane0, npl, uni, C if pred % 2 else 0)
            check_scan(ctx, ps, dset, bm.SCAN_RANGE, [[0, top], [3, 3], [top // 2, top // 4], [1, top + 5]], plane0, npl, uni)
        dset.free()


@pytest.mark.parametrize("nullable", [False, True])
def test_scan_against_reference_sparse_vector_scanner(ctx, nullable):
    """The real bm::sparse_vector<unsigned>'s own planes -> GPU scan == bm::sparse_vector_scanner<> results, and the host mirror
    (SparseVector / SparseVectorScanner) gives the same sets from the raw values."""
    import test_oracle_vs_reference as tor
    vals, nulls = tor.scan_inputs(9 + nullable, nullable=nullable)
    planes = ra.ref_sv_planes(vals, nulls)
    ps = bm.PackedSet.pack(planes)
    npl = len(planes) - 1
    dset = bm.DeviceSet.upload(ctx, ps)
    sv = bm.SparseVector.from_values(vals, nulls)
    sc = bm.SparseVectorScanner(sv, ctx)
    fn = {bm.SCAN_EQ: sc.find_eq, bm.SCAN_GT: sc.find_gt, bm.SCAN_GE: sc.find_ge, bm.SCAN_LT: sc.find_lt, bm.SCAN_LE: sc.find_le, bm.SCAN_RANGE: sc.find_range}
    for pred, search in tor.SCAN_CASES:
        blocks = check_scan(ctx, ps, dset, pred, search, 0, npl, npl)
        counts, rkind, rpop, rblk = ra.ref_sv_scan(vals, nulls, pred, search)
        assert same(blocks, rblk)
        got = fn[pred](np.array(search, np.uint64))
        nb = ps.n_blocks
        assert same(np.concatenate([np.stack([bv.block_words(c) for c in range(nb)]) for bv in got]), rblk)
    assert sc.count_eq(77) == int(((vals == 77) & (nulls == 0 if nulls is not None else True)).sum())
    assert sc.find_zero().count() == int(((vals == 0) & (nulls == 0 if nulls is not None else True)).sum())
    sc.close(); dset.free()


@pytest.mark.parametrize("name", ["scan_plain", "scan_nullable"])
def test_scan_vs_golden(ctx, name):
    """bmb200_scan on the committed planes of a real bm::sparse_vector<unsigned> == the committed scanner answers."""
    ps, vals, nulls, cases = gu.load_scan(name)
    npl = ps.n_vec - 1
    dset = bm.DeviceSet.upload(ctx, ps)
    for case in cases:
        blocks = check_scan(ctx, ps, dset, case["pred"], case["search"], 0, npl, npl)
        assert np.array_equal(blocks, case["blk"])
    dset.free()


@pytest.mark.parametrize("seed", [1, 2])
def test_shift_right_and_vs_oracle(ctx, seed):
    """OP_SHIFT_R_AND (aggregator::combine_shift_right_and): every block kind in the current and the previous block of a source,
    shifts below and above one word / one word-quad, repeated sources, sub-ranges, both GAP storage forms, the Python mirror."""
    import test_oracle_vs_reference as tor
    vecs = tor.shift_and_inputs(seed, n_vec=12, n_blocks=5)
    rng = np.random.default_rng(seed)
    for flat in (True, False):
        ps = bm.PackedSet.pack(vecs, gap_flat=flat)
        dset = bm.DeviceSet.upload(ctx, ps)
        for n in (1, 2, 3, 5, 12, 33, 34, 70, 130, 200):
            g = rng.integers(0, len(vecs), n) if n > len(vecs) else rng.permutation(len(vecs))[:n]
            check_vs_oracle(ctx, ps, bm.OP_SHIFT_R_AND, g, None, C if n % 2 else 0, dset)
        # a shard: columns [2, 5) of a set that also holds the halo column 1 (and 0) -- equals the same columns of the full result
        g = rng.permutation(len(vecs))[:6]
        res = bm.aggregate(ctx, dset, bm.OP_SHIFT_R_AND, g, None, 0, nb_from=2, nb_to=5)
        kind, pop, dig, nr = res.meta(); res.free()
        okind, opop, odig, onr, oblk, ogap = orclib.oracle_aggregate(ps, bm.OP_SHIFT_R_AND, g, None, 0)
        assert np.array_equal(pop, opop[2:5]) and np.array_equal(dig, odig[2:5]) and np.array_equal(kind, okind[2:5])
        # long chains over FULL / dense blocks keep bits alive: same vector repeated
        full_like = max(range(len(vecs)), key=lambda v: vecs[v].count())
        got = check_vs_oracle(ctx, ps, bm.OP_SHIFT_R_AND, [full_like] * 40, None, C, dset)
        assert got["total"] > 0
        dset.free()
    agg = bm.Aggregator(ctx)
    res, found = agg.combine_shift_right_and(vecs[:3])
    okind, opop, odig, onr, oblk, ogap = orclib.oracle_aggregate(bm.PackedSet.pack(vecs[:3], 6), bm.OP_SHIFT_R_AND, [0, 1, 2], None, 0)
    assert found == bool(opop.sum()) and np.array_equal(np.stack([res.block_words(c) for c in range(6)]), oblk)


def _check_decoded_set(ctx, dset, nv, nb, kinds, blks, gapsf, label):
    ps = dset.download()
    isgap = (ps.desc & 3) == bm.BLK_GAP
    assert ((ps.desc[isgap] >> 30) & 1).all()                      # decoded GAP blocks are in the flat-streamable form
    for v in range(nv):
        bv = ps.vector(v)
        assert np.array_equal(bv.kind, kinds[v]), f"{label} vector {v}: kinds {bv.kind} vs {kinds[v]}"
        assert np.array_equal(np.stack([bv.block_words(c) for c in range(nb)]), blks[v]), f"{label} vector {v}: bits"
        flat = [bv.blocks[c] for c in range(nb) if bv.kind[c] == bm.BLK_GAP]
        assert np.array_equal(np.concatenate(flat) if flat else np.zeros(0, np.uint16), gapsf[v]), f"{label} vector {v}: GAP words"
    return ps


@pytest.mark.parametrize("name", ["blobs", "blobs_entropy"])
def test_deserialize_to_device_vs_golden_and_oracle(ctx, name):
    """bmb200_set_upload_blobs: serializer BLOBs (committed fixtures written by the reference; "blobs" = levels 0..2, explicit-length
    encodings, host token walk; "blobs_entropy" = levels 3..6, gamma / interpolative / super-block encodings, token walk + entropy
    decode on the GPU) decoded on the GPU == bm::deserialize (block kinds, bits, GAP words); the decoded set then aggregates
    like the plainly uploaded one; streams the decoder does not cover and truncated streams are refused loudly."""
    nv, nb, blobs, kinds, blks, gapsf = gu.load_blobs(name)
    for level, bl in blobs.items():
        dset = bm.DeviceSet.upload_blobs(ctx, bl, nb)
        ps = _check_decoded_set(ctx, dset, nv, nb, kinds[level], blks, gapsf[level], f"{name} level {level}")
        check_vs_oracle(ctx, ps, bm.OP_OR, list(range(nv)), None, C, dset)
        check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [0, 1], list(range(2, nv)), C, dset)
        rs = bm.DeviceRS(ctx, dset, 3)
        pos = np.arange(0, nb * 65536, 997, dtype=np.uint64)
        assert np.array_equal(rs.rank(pos), orclib.oracle_rank(ps, 3, pos))
        rs.free(); dset.free()
    top = max(blobs)
    # a mixed set: every vector at a different level (host-walkable and entropy-coded BLOBs side by side)
    levels = sorted(blobs)
    mixed = [blobs[levels[v % len(levels)]][v] for v in range(nv)]
    dset = bm.DeviceSet.upload_blobs(ctx, mixed, nb)
    _check_decoded_set(ctx, dset, nv, nb, [kinds[levels[v % len(levels)]][v] for v in range(nv)], blks,
                       [gapsf[levels[v % len(levels)]][v] for v in range(nv)], f"{name} mixed levels")
    dset.free()
    # fewer columns than the BLOBs hold: the tail is decoded (to find the token ends) but not stored
    dset = bm.DeviceSet.upload_blobs(ctx, blobs[top], nb - 3)
    ps = dset.download()
    for v in range(nv):
        assert np.array_equal(np.stack([ps.vector(v).block_words(c) for c in range(nb - 3)]), blks[v][: nb - 3])
    dset.free()
    bad = blobs[top][0].copy(); bad[0] |= 1 << 6                       # BM_HM_HXOR header (XOR-reference compression): not covered
    with pytest.raises(bm.BMB200Error) as e:
        bm.DeviceSet.upload_blobs(ctx, [bad], nb)
    assert e.value.code == bm.capi.ERR_UNSUPPORTED
    for v in range(min(nv, 6)):                                        # truncated streams: rejected, never read past the end
        with pytest.raises(bm.BMB200Error):
            bm.DeviceSet.upload_blobs(ctx, [blobs[top][v][: max(2, blobs[top][v].size // 2)]], nb)
    if orclib.have_ref():                                              # fresh BLOBs of the real serializer, all levels
        import test_oracle_vs_reference as tor
        vecs = tor.entropy_inputs(7) if name == "blobs_entropy" else tor.blob_inputs()
        psr = bm.PackedSet.pack(vecs)
        for level in range(0, 7):
            bl = [orclib.ref_serialize(psr, v, level) for v in range(psr.n_vec)]
            want = [orclib.ref_deserialize(b, psr.n_blocks) for b in bl]
            dset = bm.DeviceSet.upload_blobs(ctx, bl, psr.n_blocks)
            got = dset.download()
            for v in range(psr.n_vec):
                bv = got.vector(v)
                assert np.array_equal(bv.kind, want[v][0]), f"level {level} vector {v}: kinds"
                assert np.array_equal(np.stack([bv.block_words(c) for c in range(psr.n_blocks)]), want[v][2]), f"level {level} vector {v}: bits"
                for c in range(psr.n_blocks):
                    if bv.kind[c] == bm.BLK_GAP:
                        assert np.array_equal(bv.blocks[c], want[v][3][c][: bv.blocks[c].size]), f"level {level} vector {v} column {c}: GAP words"
            dset.free()
    if orclib.have_ref(True):                                          # BM64ADDR streams (64-bit header fields)
        import test_oracle_vs_reference as tor
        vecs = tor.entropy_inputs(3) if name == "blobs_entropy" else tor.blob_inputs()
        psr = bm.PackedSet.pack(vecs)
        bl = [orclib.ref_serialize(psr, v, 6 if name == "blobs_entropy" else 2, addr64=True) for v in range(psr.n_vec)]
        dset = bm.DeviceSet.upload_blobs(ctx, bl, psr.n_blocks)
        got = dset.download()
        for v in range(psr.n_vec):
            assert np.array_equal(np.stack([got.vector(v).block_words(c) for c in range(psr.n_blocks)]),
                                  np.stack([vecs[v].block_words(c) for c in range(psr.n_blocks)])), f"64-bit stream, vector {v}"
        dset.free()


def test_sharded_rs_device_callables_two_shards_one_gpu():
    """ShardedRS over the device kernels: the vector is cut into two block-range shards that both live on this GPU (each with its own
    DeviceSet + DeviceRS, queried through the *_dev entry points on torch CUDA tensors); the two shards' contributions are summed by
    hand (what the all_reduce does) and must equal the unsharded oracle -- positions past the end, rank 0 and ranks above the
    cardinality included."""
    import torch
    from bitmagic_b200.sharding import ShardedRS, device_rs_callables, shard_range
    rng = np.random.default_rng(78)
    n_blocks = 600
    vec = gen.mixed_vectors(rng, 1, n_blocks, p_null=0.3, p_full=0.1, p_gap=0.4)[0]
    whole = bm.PackedSet.pack([vec])
    card = vec.count()
    dev = torch.device("cuda", 0)
    ctx = bm.Context(0)                                    # a context of its own, bound to torch's current stream
    ctx.set_stream(torch.cuda.current_stream(dev).cuda_stream)
    try:
        pos = np.concatenate([rng.integers(0, n_blocks * 65536, 20000), [0, 65535, 65536, 256 * 65536 - 1, 256 * 65536, n_blocks * 65536 - 1,
                              n_blocks * 65536, n_blocks * 65536 + 999]]).astype(np.int64)
        rk = np.concatenate([rng.integers(1, card + 1, 20000), [0, 1, card, card + 1, card + 77]]).astype(np.int64)
        tpos, trk = torch.from_numpy(pos).to(dev), torch.from_numpy(rk).to(dev)
        totals = [vec.slice(*shard_range(n_blocks, 2, r)).count() for r in range(2)]

        class TwoShards:                                   # stands in for torch.distributed: shard cardinalities known, no reduction
            def __init__(self, r): self.r = r
            def is_initialized(self): return True
            def get_world_size(self): return 2
            def get_rank(self): return self.r
            def all_gather_into_tensor(self, out, t): out.copy_(torch.tensor(totals, dtype=torch.int64, device=out.device))
            def all_reduce(self, t): pass

        acc_rank = torch.zeros_like(tpos); acc_pos = torch.zeros_like(trk); acc_found = torch.zeros_like(trk, dtype=torch.bool)
        for r in range(2):
            lo, hi = shard_range(n_blocks, 2, r)
            dset = bm.DeviceSet.upload(ctx, bm.PackedSet.pack([vec.slice(lo, hi)]))
            rs = bm.DeviceRS(ctx, dset, 0)
            assert rs.total() == totals[r]
            srs = ShardedRS(rs.total(), *device_rs_callables(rs), n_blocks, TwoShards(r), dev)
            acc_rank += srs.rank(tpos)
            p, f = srs.select(trk)
            acc_pos += p; acc_found |= f
            torch.cuda.synchronize(dev)
            rs.free(); dset.free()
        want_rank = orclib.oracle_rank(whole, 0, pos.astype(np.uint64)).astype(np.int64)
        want_pos, want_found = orclib.oracle_select(whole, 0, rk.astype(np.uint64))
        assert np.array_equal(acc_rank.cpu().numpy(), want_rank)
        assert np.array_equal(acc_found.cpu().numpy(), want_found)
        assert np.array_equal(acc_pos.cpu().numpy()[want_found], want_pos.astype(np.int64)[want_found])
    finally:
        ctx.close()


def test_find_first_and_sub_with_range_hints(ctx):
    """Aggregator.find_first_and_sub + set_range_hint (aggregator::find_first_and_sub, src/bmaggregator.h:1457-1549) against the first
    position of the oracle's AND-SUB result restricted the way the reference restricts it: block range for a multi-block hint,
    block range + in-block mask for a one-block hint."""
    rng = np.random.default_rng(77)
    vecs = gen.mixed_vectors(rng, 9, 12, p_null=0.2)
    ps = bm.PackedSet.pack(vecs)
    agg = bm.Aggregator(ctx)
    for g0, g1 in (([0, 1], [2, 3]), ([4], []), ([5, 6, 7], [8]), ([0, 1, 2, 3, 4], [5])):
        okind, _, _, _, want_blocks, _ = orclib.oracle_aggregate(ps, bm.OP_AND_SUB, g0, g1, 0)
        want_blocks = want_blocks.copy(); want_blocks[okind == bm.BLK_FULL] = 0xFFFFFFFF; want_blocks[okind == bm.BLK_NULL] = 0
        allpos = np.flatnonzero(np.unpackbits(np.ascontiguousarray(want_blocks).view(np.uint8), bitorder="little"))
        for hint in (None, (3 * 65536 + 5, 8 * 65536 + 100), (2 * 65536 + 1000, 2 * 65536 + 40000), (11 * 65536, 12 * 65536 - 1), (65536 * 5 + 7, 65536 * 5 + 7)):
            agg.reset_range_hint()
            pos = allpos
            if hint is not None:
                one = agg.set_range_hint(*hint)
                assert one == ((hint[0] >> 16) == (hint[1] >> 16))
                if one:
                    pos = allpos[(allpos >= hint[0]) & (allpos <= hint[1])]
                else:
                    pos = allpos[(allpos >= (hint[0] >> 16) * 65536) & (allpos < ((hint[1] >> 16) + 1) * 65536)]
            found, idx = agg.find_first_and_sub([vecs[k] for k in g0], [vecs[k] for k in g1])
            assert found == bool(pos.size), (g0, g1, hint)
            if found:
                assert idx == int(pos[0]), (g0, g1, hint, idx, int(pos[0]))
    agg.reset_range_hint()
    assert agg.find_first_and_sub([], [vecs[0]]) == (False, 0)


def test_c1_config_bit_and_count(ctx):
    """BASELINE configs[0]: two bvectors of 2^20 bits, 10 % random fill: bit_and + count() and count_and through the C ABI == the oracle
    (and the reference when its library travelled); bytes touched = 3 * 16 * 8192."""
    vecs = gen.c1_vectors()
    ps = bm.PackedSet.pack(vecs)
    t = bm.bit_and(vecs[0], vecs[1], bm.OPT_NONE, ctx)
    want = np.stack([vecs[0].block_words(c) & vecs[1].block_words(c) for c in range(16)])
    assert np.array_equal(np.stack([t.block_words(c) for c in range(16)]), want)
    okind, opop, odig, onr, oblk, ogap = orclib.oracle_aggregate(ps, bm.OP_AND, [0, 1], None, 0)
    assert np.array_equal(oblk, want) and t.count() == int(opop.sum()) == bm.count_and(vecs[0], vecs[1], ctx)
    assert bm.count_or(vecs[0], vecs[1], ctx) == vecs[0].count() + vecs[1].count() - t.count()
    rkind, rpop, rblk, rcnt = ra.ref_binop(ps, 1, 0, 1)
    assert same(rblk, want) and rcnt == t.count() == ra.ref_count_op(ps, 1, 0, 1)


# ----------------------------------------------------------------------------------------------------------------------
# round 2: full-size parity in the test records, generator pinned on the reference, residency / e2e paths
# ----------------------------------------------------------------------------------------------------------------------
def _host_mem_gb():
    try:
        return int(next(ln for ln in open("/proc/meminfo") if ln.startswith("MemAvailable")).split()[1]) / 2**20
    except Exception:
        return 0.0


def test_device_generator_equals_host_generator_bit_for_bit(ctx):
    """bmb200_synth_set (CUDA) and oracle/bm_synth.c (host, pinned on bvector::optimize() by the CPU tests) are two independent
    implementations of the benchmark generator: every array of the packed set must be identical -- so the bench's inputs are
    exactly what the reference arm and the parity check regenerate on the host."""
    import os
    for nv, nbk, dens, opt in ((48, 7, np.array([0.5 / (k + 1) for k in range(48)]), True), (9, 5, np.full(9, 0.05), False),
                               (33, 4, np.concatenate([np.full(30, 0.0025), [0.0, 1.0, 0.0098]]), True)):
        seed = np.arange(31, 31 + nv, dtype=np.uint64) * np.uint64(7919)
        dset = bm.DeviceSet.synth(ctx, nv, nbk, dens, seed, opt)
        ps = dset.download()
        hs = orclib.HostSynth(nv, nbk, dens, seed, opt, threads=min(4, os.cpu_count() or 1))
        for a in ("desc", "bit_base", "gap_base", "bit_pool", "gap_pool"):
            assert np.array_equal(getattr(ps, a), getattr(hs.ps, a)), f"{a} differs (n_vec={nv})"
        hs.free(); dset.free()


REF_THREADS = 8          # reference workers for the all-column checks (their answers are recorded per thread count)


def _all_column_parity(ctx, nv, nbk, dens, seed, optimize, op, g0, g1, flags, threads):
    dset = bm.DeviceSet.synth(ctx, nv, nbk, dens, seed, optimize)
    res = bm.aggregate(ctx, dset, op, g0, g1, flags)
    kind, pop, dig, nr = res.meta()
    total, _ = res.total()
    hs = orclib.HostSynth(nv, nbk, dens, seed, optimize, threads=threads)
    assert hs.ps.stored_bytes() == dset.stored_bytes()
    tot, k, p, d, gl = ra.ref_job(hs.ps, op, g0, g1, flags, threads=threads)
    hs.free()
    assert tot == total
    assert same(k, kind), "block kinds"
    assert same(p, pop), "popcounts"
    assert same(d, dig), "digests"
    assert same(gl, np.where(kind == bm.BLK_GAP, nr, 0)), "GAP lengths"
    res.free(); dset.free()
    return int(total)


def test_c2_full_size_all_columns_vs_reference(ctx):
    """BASELINE config 2 at FULL size (combine_or over 256 x 2^28 bits, 5 %, bit-blocks = 8 GiB): kind, popcount and digest of
    all 4096 result columns against the unmodified reference (all host cores) on host-regenerated inputs."""
    import os
    if _host_mem_gb() < 24:
        pytest.skip("needs ~20 GB of host memory")
    nv, nbk = 256, 4096
    dens = np.full(nv, 0.05); seed = np.arange(100, 100 + nv, dtype=np.uint64)
    tot = _all_column_parity(ctx, nv, nbk, dens, seed, False, bm.OP_OR, np.arange(nv, dtype=np.uint32), None, bm.F_OPT_NONE, REF_THREADS)
    assert tot > 0.99 * nbk * 65536           # 0.95^256: practically all ones


def test_c3_quarter_size_all_columns_vs_reference(ctx):
    """BASELINE config 3's recipe on 4096 of its 16384 block columns (the bench line itself carries the full-size check): AND-SUB
    over 1024 Zipf vectors, every column's kind / popcount / digest / GAP length against the unmodified reference."""
    import os
    if _host_mem_gb() < 12:
        pytest.skip("needs ~10 GB of host memory")
    nv, nbk = 1024, 4096
    dens = np.array([0.5 / (k + 1) for k in range(nv)]); seed = np.arange(1000, 1000 + nv, dtype=np.uint64)
    _all_column_parity(ctx, nv, nbk, dens, seed, True, bm.OP_AND_SUB, np.array([0, 1], np.uint32), np.arange(2, nv, dtype=np.uint32), C, REF_THREADS)


@pytest.mark.parametrize("optimize", [False, True])
def test_c4_full_size_rs_index_rank_select_vs_reference64(ctx, optimize):
    """BASELINE config 4 at FULL size: one 2^32-bit vector (65536 blocks, 1 %), rs_index fields + 10 M count_to + 10 M select,
    ALL answers against the unmodified reference built with -DBM64ADDR (oracle/_ref/libbmref64.so)."""
    if _host_mem_gb() < 6:
        pytest.skip("needs ~4 GB of host memory")
    nbk, nq = 65536, 10_000_000
    dset = bm.DeviceSet.synth(ctx, 1, nbk, np.array([0.01]), np.array([7], np.uint64), optimize)
    rs = bm.DeviceRS(ctx, dset, 0)
    total = rs.total()
    bc, sc, sb = rs.export()
    rng = np.random.default_rng(8)
    pos = rng.integers(0, nbk * 65536, nq, dtype=np.uint64)
    rank = rng.integers(1, total + 1, nq, dtype=np.uint64)
    rank[:3] = (0, total, total + 1)                     # select fails for rank 0 and rank > count
    g_rank = rs.rank(pos)
    g_sel, g_found = rs.select(rank)
    ps = dset.download()
    rbc, rsc, rsb, rtot = ra.ref_rs_build(ps, 0, addr64=True)
    assert rtot == total and same(rbc, bc) and same(rsb, sb)
    assert same(np.where(bc > 0, sc, 0), rsc)                 # sub-counts of the non-empty blocks
    r_rank, r_sel, r_found = ra.ref_rank_select(ps, 0, pos, rank, addr64=True)
    assert same(g_rank, r_rank)
    assert same(g_found, r_found) and not g_found[0] and g_found[1] and not g_found[2]
    assert same(np.where(g_found, g_sel, 0), r_sel)
    rs.free(); dset.free()


def test_upload_vectors_pipeline_many_chunks_and_threads(ctx):
    """bmb200_set_upload_vectors: threaded packing through the pinned staging ring.  A set whose columns exceed one slot several
    times over (forced small by 1 host thread vs many) must arrive bit-exact and aggregate like the plainly uploaded packed set."""
    rng = np.random.default_rng(5)
    vecs = gen.mixed_vectors(rng, 40, 48, p_null=0.05)
    ps = bm.PackedSet.pack(vecs)
    for threads in (1, 0, 7):
        ctx.set_tuning(bm.capi.TUNE_HOST_THREADS, threads)
        dset = bm.DeviceSet.upload_vectors(ctx, vecs)
        back = dset.download()
        for a in ("desc", "bit_base", "gap_base", "bit_pool", "gap_pool"):
            assert np.array_equal(getattr(back, a), getattr(ps, a)), f"{a} (threads={threads})"
        check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [0, 1, 2], list(range(3, 40)), C, dset)
        dset.free()
    ctx.set_tuning(bm.capi.TUNE_HOST_THREADS, 0)


def test_upload_slabs_dma_plus_device_gather_equals_host_packing(ctx):
    """bmb200_set_upload_slabs: blocks that live inside a few host slabs (what a slab-backed bm::bvector<> allocator holds) cross
    PCIe as they lie and are gathered into the arena on the device -- the arena must equal the host-packed one byte for byte
    (descriptors, prefix sums, bit pool, FLAT GAP pool incl. lead pads and zero fill), pinned or pageable slabs, with and without
    the prefetch; a block outside every slab makes the call fall back to the packing path (same result)."""
    rng = np.random.default_rng(11)
    vecs = gen.mixed_vectors(rng, 70, 40, p_null=0.05)
    ps = bm.PackedSet.pack(vecs)
    launches0 = ctx.launch_count()
    for kw in (dict(pinned=True), dict(pinned=False, slab_bytes=300_000), dict(pinned=True, prefetch=True, slab_bytes=4 << 20), dict(pinned=False, stray=True)):
        dset = bm.DeviceSet.upload_slabs(ctx, vecs, **kw)
        back = dset.download()
        for a in ("desc", "bit_base", "gap_base", "bit_pool", "gap_pool"):
            assert np.array_equal(getattr(back, a), getattr(ps, a)), f"{a} ({kw})"
        check_vs_oracle(ctx, ps, bm.OP_AND_SUB, [0, 1, 2], list(range(3, 70)), C, dset)
        check_vs_oracle(ctx, ps, bm.OP_OR, list(range(70)), None, C, dset)
        dset.free()
    assert ctx.launch_count() > launches0
    ctx.trim()


@pytest.mark.parametrize("flavour", ["e2e", "e2e_slab"])
def test_e2e_harness_real_bvectors_cold_warm_and_check(ctx, flavour):
    """oracle/_ref/libbmb200_e2e.so (bench.py's e2e leg): bm::b200::aggregator on real bm::bvector<> objects -- cold call, warm call
    on a bm::b200::device_set, and the reference aggregator on the same bvectors (compare() == 0 + calc_stat kinds).
    libbmb200_e2e_slab.so is the same harness on bm::b200::slab_bvector (page-locked slab allocator; cold upload = slab DMA +
    device gather)."""
    import ctypes as Ct
    so = orclib.ORACLE_DIR / "_ref" / f"libbmb200_{flavour}.so"
    if not so.exists():
        pytest.skip(f"oracle/_ref/{so.name} not built (needs /root/reference at build time)")
    lib = Ct.CDLL(str(so)); lib.e2e_create_empty.restype = Ct.c_void_p; lib.e2e_free.restype = None
    nv, nbk = 96, 2304                                   # 9 top-level blocks: the result store runs on several host threads (>= 2048 columns)
    dens = np.array([0.5 / (k + 1) for k in range(nv)]); seed = np.arange(1000, 1000 + nv, dtype=np.uint64)
    dset = bm.DeviceSet.synth(ctx, nv, nbk, dens, seed, True)
    node = Ct.c_int(-1)
    h = Ct.c_void_p(lib.e2e_create_empty(nv, nbk, 0, 0, Ct.byref(node)))
    assert h
    from bitmagic_b200.capi import packed_c, ptr
    for lo in range(0, nbk, 256):
        ps = dset.download(lo, min(nbk, lo + 256))
        c = packed_c(ps.n_vec, ps.n_blocks, ps.desc, ps.bit_base, ps.gap_base, ps.bit_pool, ps.gap_pool)
        assert lib.e2e_append(h, Ct.byref(c), lo, 3) == 0
    for op, g0, g1, compress in ((bm.OP_AND_SUB, np.array([0, 1], np.uint32), np.arange(2, nv, dtype=np.uint32), 1),
                                 (bm.OP_OR, np.arange(10, nv, dtype=np.uint32), np.zeros(0, np.uint32), 1),
                                 (bm.OP_OR, np.arange(nv, dtype=np.uint32), np.zeros(0, np.uint32), 0)):
        want = bm.aggregate(ctx, dset, op, g0, g1 if g1.size else None, C if compress else 0).total()[0]
        ms = np.zeros(2); cnt = Ct.c_uint64(0); h2d = Ct.c_uint64(0); d2h = Ct.c_uint64(0)
        assert lib.e2e_cold(h, op, compress, ptr(g0), g0.size, ptr(g1), g1.size, 2, ptr(ms), Ct.byref(cnt), Ct.byref(h2d), Ct.byref(d2h)) == 0
        assert cnt.value == want and h2d.value >= dset.stored_bytes()
        eq = Ct.c_int(0); rc_ = Ct.c_uint64(0); rms = Ct.c_double(0)
        assert lib.e2e_check(h, op, compress, ptr(g0), g0.size, ptr(g1), g1.size, Ct.byref(eq), Ct.byref(rc_), Ct.byref(rms)) == 0
        assert eq.value == 1 and rc_.value == want, "cold result bvector differs from bm::aggregator"
        wms = np.zeros(3)
        assert lib.e2e_warm(h, op, compress, ptr(g0), g0.size, ptr(g1), g1.size, 1, 3, ptr(wms), Ct.byref(cnt), Ct.byref(d2h)) == 0
        assert cnt.value == want
        assert lib.e2e_check(h, op, compress, ptr(g0), g0.size, ptr(g1), g1.size, Ct.byref(eq), Ct.byref(rc_), Ct.byref(rms)) == 0
        assert eq.value == 1, "warm (resident device_set) result bvector differs from bm::aggregator"
    lib.e2e_free(h)
    dset.free()


def test_deserialize_to_device_superblock_members_at_capacity_levels(ctx):
    """Super-block token whose member blocks have exactly 124 / 252 / 508 / 1276 / 1277 runs (gap_block_set_no_ret thresholds,
    src/bm.h:4800): kinds, GAP words incl. the header level bits and bits decoded on the GPU == bm::deserialize."""
    v = gen.superblock_threshold_vector()
    ps = bm.PackedSet.pack([v])
    for level in (5, 6):
        blob = ra.ref_serialize(ps, 0, level)
        rkind, rpop, rblk, rgap = ra.ref_deserialize(blob, ps.n_blocks)
        dset = bm.DeviceSet.upload_blobs(ctx, [blob], ps.n_blocks)
        bv = dset.download().vector(0)
        assert same(bv.kind, rkind)
        for c in range(ps.n_blocks):
            if rkind[c] == bm.BLK_GAP:
                n = (int(bv.blocks[c][0]) >> 3) + 1
                assert n == bv.blocks[c].size and same(np.pad(bv.blocks[c], (0, orclib.GAP_MAX_WORDS - n)), rgap[c]), f"level {level} block {c}"
            elif rkind[c] == bm.BLK_BIT:
                assert same(bv.blocks[c], rblk[c])
        dset.free()


def test_binop_result_kinds_vs_reference(ctx):
    """bmb200_binop (bvector::bit_or / bit_and / bit_xor / bit_sub): bits, popcounts AND block kinds of every column against the real
    3-operand ops, for every pairing of NULL / FULL / bit / GAP argument blocks and both opt modes; GAP x GAP goes through the
    device merge (gap_merge_kernel), incl. identical, disjoint and nested run lists."""
    rng = np.random.default_rng(21)
    vecs = gen.mixed_vectors(rng, 6, 40, p_null=0.15, p_full=0.1, p_gap=0.45) + gen.edge_vectors(40)[:4]
    gap_only = bm.BVector(40)
    for nb in range(40):                                      # a GAP-only vector and an exact copy of it
        gap_only.set_gap(nb, bm.hostfmt.bits_to_gap(gen.block_with_runs(rng, int(rng.integers(2, 900)))))
    vecs += [gap_only, gap_only.slice(0, 40)]
    ps = bm.PackedSet.pack(vecs, 40)
    dset = bm.DeviceSet.upload(ctx, ps)
    n = len(vecs)
    ops = {0: bm.OP_OR, 1: bm.OP_AND, 2: bm.capi.OP_SUB, 3: bm.OP_XOR}
    pairs = [(a, b) for a in range(n) for b in range(n) if a != b]
    for compress in (False, True):
        for (a, b) in pairs[:: 3 if compress else 2]:
            for rop, gop in ops.items():
                rkind, rpop, rblk, rcnt = ra.ref_binop(ps, rop, a, b, compress)
                res = bm.capi.binop(ctx, dset, gop, a, b, C if compress else 0)
                kind, pop, dig, nr = res.meta()
                fk, off, bits, gaps = res.fetch()
                bv = bm.result_to_bvector(fk, off, bits, gaps)
                res.free()
                assert same(kind, rkind), f"kinds: op {rop} ({a},{b}) compress={compress}: {kind}"
                assert same(pop, rpop) and int(pop.sum()) == rcnt
                assert same(np.stack([bv.block_words(c) for c in range(40)]), rblk)
    dset.free()


def test_sharded_aggregator_cxx_two_ranks_nccl(tmp_path):
    """bm::b200::sharded_aggregator (C++ binding) on 2 GPUs, one process per GPU: block-range shards, the library's own NCCL exchange
    (bmb200_comm_init / bmb200_exchange_popcounts, id passed through a file) vs bm::aggregator on the full vectors.  Needs >= 2 GPUs."""
    import subprocess
    import torch
    exe = orclib.ORACLE_DIR / "_ref" / "test_sharded"
    if not exe.exists():
        pytest.skip("oracle/_ref/test_sharded not built (needs /root/reference at build time)")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (NCCL refuses two ranks on one device)")
    idf = tmp_path / "nccl_id.bin"
    procs = [subprocess.Popen([str(exe), str(r), "2", str(idf)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and "OK:" in o, f"rank {r}:\n{o[-2000:]}"
