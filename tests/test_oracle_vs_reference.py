"""Pins oracle/bm_oracle.c (the plain-C restatement) against the UNMODIFIED reference (oracle/_ref/libbmref.so).  The
reference's answers come from tests/refanswers.py: live where the reference library was built, recorded
(tests/golden/ref_answers*.npz) everywhere else."""
import numpy as np
import pytest

import bitmagic_b200 as bm
import gen
import orclib
import refanswers as ra
from refanswers import same

# BLOBs written by the reference's serializer are these tests' inputs: too large to store in full, so they run where the
# reference library was built (tests/test_golden.py covers committed BLOB fixtures everywhere)
needs_serializer = pytest.mark.skipif(not orclib.have_ref(), reason="needs the reference library (oracle/_ref) for fresh BLOBs")

OPS = [(bm.OP_OR, "or"), (bm.OP_AND, "and"), (bm.OP_AND_SUB, "and_sub")]


def _groups(rng, n_vec, op):
    if op == bm.OP_AND_SUB:
        na = int(rng.integers(1, 4))
        perm = rng.permutation(n_vec)
        return perm[:na], perm[na:]
    if op == bm.OP_AND:
        return rng.permutation(n_vec)[: int(rng.integers(2, 5))], None
    return rng.permutation(n_vec)[: int(rng.integers(1, n_vec + 1))], None


@pytest.mark.parametrize("op,name", OPS)
@pytest.mark.parametrize("compress", [0, 1])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_aggregate_oracle_matches_reference(op, name, compress, seed):
    rng = np.random.default_rng(1000 * op + 10 * seed + compress)
    kw = dict(p_null=0.05, p_full=0.03) if op != bm.OP_OR else {}
    vecs = gen.mixed_vectors(rng, 10, 5, **kw)
    ps = bm.PackedSet.pack(vecs)
    g0, g1 = _groups(rng, 10, op)
    flags = bm.F_OPT_COMPRESS if (compress or op == bm.OP_AND_SUB) else 0   # combine_and_sub always compresses
    okind, opop, odig, onr, oblk, ogap = orclib.oracle_aggregate(ps, op, g0, g1, flags)
    rkind, rpop, rblk, rgap, rany = ra.ref_aggregate(ps, op, g0, g1, flags)
    assert same(oblk, rblk)              # compare()==0
    assert same(opop, rpop)              # count()
    assert same(okind, rkind)            # calc_stat block kinds
    assert same(ogap, rgap)                        # GAP encodings (rows zero past their length on both sides)
    assert rany == bool(opop.sum())
    # the reference's own independent check: the "horizontal" path (tests/stress/t.cpp:10887-10921)
    hkind, hpop, hblk, _, _ = ra.ref_aggregate(ps, op, g0, g1, flags, horizontal=True)
    assert same(oblk, hblk)


def test_aggregate_edge_cases_match_reference():
    vecs = gen.edge_vectors(4)
    ps = bm.PackedSet.pack(vecs)
    n = len(vecs)
    cases = [(bm.OP_OR, list(range(n)), None), (bm.OP_OR, [0, 1], None), (bm.OP_OR, [5], None),
             (bm.OP_OR, [3, 4], None), (bm.OP_AND, [2, 3], None), (bm.OP_AND, [0, 2], None),
             (bm.OP_AND, [2, 2], None), (bm.OP_AND_SUB, [2], [0]), (bm.OP_AND_SUB, [2], [5]),
             (bm.OP_AND_SUB, [2, 3], [1, 4]), (bm.OP_AND_SUB, [3], [2]), (bm.OP_AND_SUB, [1], [])]
    for op, g0, g1 in cases:
        for flags in (0, bm.F_OPT_COMPRESS):
            if op == bm.OP_AND_SUB:
                flags = bm.F_OPT_COMPRESS
            okind, opop, odig, onr, oblk, ogap = orclib.oracle_aggregate(ps, op, g0, g1, flags)
            rkind, rpop, rblk, rgap, rany = ra.ref_aggregate(ps, op, g0, g1, flags)
            assert same(oblk, rblk), (op, g0, g1)
            assert same(opop, rpop), (op, g0, g1)
            assert same(okind, rkind), (op, g0, g1, flags, okind, rkind)


def test_xor_matches_reference_bit_xor():
    rng = np.random.default_rng(5)
    vecs = gen.mixed_vectors(rng, 6, 4)
    ps = bm.PackedSet.pack(vecs)
    for a, b in [(0, 1), (2, 3), (4, 5), (1, 1)]:
        okind, opop, odig, onr, oblk, _ = orclib.oracle_aggregate(ps, bm.OP_XOR, [a, b], None, bm.F_OPT_COMPRESS)
        rkind, rpop, rblk, rcnt = ra.ref_binop(ps, 3, a, b, compress=True)
        assert same(oblk, rblk)
        assert int(opop.sum()) == rcnt == ra.ref_count_op(ps, 3, a, b)
    # 3-way chain
    _, opop, _, _, oblk, _ = orclib.oracle_aggregate(ps, bm.OP_XOR, [0, 1, 2], None, 0)
    _, _, rblk, _, _ = ra.ref_aggregate(ps, bm.OP_XOR, [0, 1, 2], None, 0)
    assert same(oblk, rblk)


def test_two_operand_ops_match_reference():
    rng = np.random.default_rng(11)
    vecs = gen.mixed_vectors(rng, 4, 6)
    ps = bm.PackedSet.pack(vecs)
    for a, b in [(0, 1), (2, 3), (1, 2)]:
        for refop, op, g0, g1 in [(0, bm.OP_OR, [a, b], None), (1, bm.OP_AND, [a, b], None), (2, bm.OP_AND_SUB, [a], [b])]:
            _, opop, _, _, oblk, _ = orclib.oracle_aggregate(ps, op, g0, g1, 0)
            _, rpop, rblk, rcnt = ra.ref_binop(ps, refop, a, b)
            assert same(oblk, rblk)
            assert int(opop.sum()) == rcnt == ra.ref_count_op(ps, refop, a, b)


def test_optimize_classification_and_bit_to_gap():
    """calc_change / bit_to_gap / the opt_compress classification vs bvector::optimize on the reference."""
    rng = np.random.default_rng(3)
    v = bm.BVector(8)
    for nb, runs in enumerate([1, 2, 3, 1274, 1275, 1276, 1277, 4000]):
        v.set_bits(nb, gen.block_with_runs(rng, runs))
    ps = bm.PackedSet.pack([v])
    rkind, rpop, rblk, rgap = ra.ref_optimize(ps, 0)
    import ctypes as C
    for nb in range(8):
        w = np.ascontiguousarray(v.blocks[nb])
        runs = orclib.oracle().orc_bit_block_calc_change(orclib.ptr(w))
        exp = bm.BLK_GAP if 1 < runs < 1276 else bm.BLK_BIT
        if runs == 1:
            exp = bm.BLK_FULL if w[0] else bm.BLK_NULL
        assert rkind[nb] == exp, (nb, runs, rkind[nb])
        if exp == bm.BLK_GAP:
            out = np.zeros(70000, np.uint16)
            ln = orclib.oracle().orc_bit_to_gap(orclib.ptr(out), orclib.ptr(w))
            assert ln == runs
            assert same(np.pad(out[:ln + 1], (0, orclib.GAP_MAX_WORDS - ln - 1)), rgap[nb])
            # host mirror (product-side numpy helper) agrees too
            assert same(bm.hostfmt.bits_to_gap(w), out[:ln + 1])


@pytest.mark.parametrize("seed", [1, 2])
def test_rs_index_and_queries_match_reference(seed):
    rng = np.random.default_rng(seed)
    vecs = gen.mixed_vectors(rng, 3, 600, p_null=0.2, p_full=0.1, p_gap=0.4) + gen.edge_vectors(600)[:5]
    ps = bm.PackedSet.pack(vecs)
    for v in range(ps.n_vec):
        obc, osc, osb = orclib.oracle_rs_build(ps, v)
        rbc, rsc, rsb, rtot = ra.ref_rs_build(ps, v)
        if rtot == 0:
            assert obc.sum() == 0
            continue
        assert same(obc, rbc)
        # the reference does not define sub_count for NULL blocks beyond 0 (ra.ref_rs_build zeroes it there)
        assert same(np.where(obc > 0, osc, 0), rsc)
        assert same(osb, rsb)
        pos = rng.integers(0, 600 * 65536, 3000).astype(np.uint64)
        rank = rng.integers(0, rtot + 3, 3000).astype(np.uint64)
        rr, rp, rf = ra.ref_rank_select(ps, v, pos, rank)
        assert same(orclib.oracle_rank(ps, v, pos), rr)
        op, of = orclib.oracle_select(ps, v, rank)
        assert same(of, rf)
        assert same(np.where(of, op, 0), rp)     # positions where found (ra.ref_rank_select zeroes the rest)


def test_reference_known_answers_sample16():
    """samples/bvsample16/sample16.cpp:95-130 expected outputs:
    OR -> 0..10,10000,20000 ; AND -> 10000,20000 ; AND-SUB -> 20000 (see SURVEY 8c)."""
    nbk = 1
    def mk(pos):
        return bm.BVector.from_positions(pos, nbk)
    bv1 = mk([1, 2, 3, 10000, 20000]); bv2 = mk([0, 4, 5, 6, 10000, 20000]); bv3 = mk([7, 8, 9, 10, 10000, 20000])
    bv4 = mk([10000]);
    ps = bm.PackedSet.pack([bv1, bv2, bv3, bv4])
    for op, g0, g1, flags, want in ((bm.OP_OR, [0, 1, 2], None, 0, list(range(11)) + [10000, 20000]),
                                    (bm.OP_AND, [0, 1, 2], None, 0, [10000, 20000]),
                                    (bm.OP_AND_SUB, [0, 1, 2], [3], bm.F_OPT_COMPRESS, [20000])):
        blk = orclib.oracle_aggregate(ps, op, g0, g1, flags)[4]
        assert list(np.flatnonzero(bm.hostfmt.words_to_bits(blk[0]))) == want
        assert same(blk, ra.ref_aggregate(ps, op, g0, g1, flags)[2])      # the reference's bits: the same known answer


def test_pipeline_oracle_matches_reference():
    """aggregator::pipeline + combine_and_sub(TPipe&) (src/bmaggregator.h:222-341,1291-1453): counts, per-group
    results (kinds included) and the OR target equal the per-group oracle."""
    rng = np.random.default_rng(31)
    vecs = gen.mixed_vectors(rng, 14, 5, p_null=0.05, p_full=0.03)
    ps = bm.PackedSet.pack(vecs)
    groups = [([0, 1], [2, 3, 4]), ([5], []), ([2, 3], [2]), ([6, 7, 8], [9, 10, 11, 12, 13]), ([1], [0])]
    counts, rkind, rpop, rblk, rok, rob = ra.ref_pipeline(ps, groups, want_or=True)
    union = np.zeros((5, 2048), np.uint32)
    oblks = []
    for g, (g0, g1) in enumerate(groups):
        okind, opop, odig, onr, oblk, _ = orclib.oracle_aggregate(ps, bm.OP_AND_SUB, g0, g1, bm.F_OPT_COMPRESS)
        assert counts[g] == int(opop.sum())
        assert same(rpop[g], opop) and same(rkind[g], okind)
        oblks.append(oblk)
        union |= oblk
    assert same(np.stack(oblks), rblk)
    assert same(rob, union)


SCAN_CASES = [(bm.SCAN_EQ, [0, 17, 4999, 70000, 65536 + 77, 1 << 20]), (bm.SCAN_GT, [0, 100, 4998, 5000, 65535, 1 << 20]), (bm.SCAN_GE, [0, 1, 2500, 5000, 65536]),
              (bm.SCAN_LT, [0, 1, 3000, 9999, 70000]), (bm.SCAN_LE, [0, 4999, 12, 65536]), (bm.SCAN_RANGE, [[10, 20], [0, 0], [0, 4999], [30, 10], [4000, 1 << 22], [65536, 70000]])]


def scan_inputs(seed, n=150000, nullable=False):
    rng = np.random.default_rng(seed)
    vals = rng.integers(0, 5000, n).astype(np.uint32)
    vals[rng.random(n) < 0.3] = 0
    vals[n // 2: n // 2 + 4000] = 77                     # a long run of one value
    vals[rng.random(n) < 0.0008] |= np.uint32(1 << 16)   # a sparse high plane (GAP blocks); planes 13..15 stay absent
    nulls = (rng.random(n) < 0.1).astype(np.uint8) if nullable else None
    return vals, nulls


@pytest.mark.parametrize("nullable", [False, True])
def test_scan_oracle_matches_reference_scanner(nullable):
    """orc_scan (restated contract) == bm::sparse_vector_scanner<> on the reference's own optimize()d planes."""
    vals, nulls = scan_inputs(5 + nullable, nullable=nullable)
    planes = ra.ref_sv_planes(vals, nulls)
    ps = bm.PackedSet.pack(planes)
    npl = len(planes) - 1
    kinds = ps.kinds()
    assert npl == 17 and (kinds == bm.BLK_GAP).any() and (kinds == bm.BLK_BIT).any() and (kinds == bm.BLK_NULL).any()
    for pred, search in SCAN_CASES:
        okind, opop, odig, onr, oblk, ogap = orclib.oracle_scan(ps, pred, search, 0, npl, npl, bm.F_OPT_COMPRESS)
        counts, rkind, rpop, rblk = ra.ref_sv_scan(vals, nulls, pred, search)
        assert same(oblk, rblk), f"pred {pred}"
        assert same(opop, rpop)
        assert same(opop.reshape(len(search), -1).sum(1), counts)


def shift_and_inputs(seed, n_vec=10, n_blocks=5):
    """Vectors dense enough that (T >> 1) & v keeps bits alive for a few steps, all block kinds, carries across block borders."""
    rng = np.random.default_rng(seed)
    vecs = gen.mixed_vectors(rng, n_vec, n_blocks, p_null=0.08, p_full=0.25, p_gap=0.3)
    for v in vecs[: n_vec // 2]:                       # dense bit / GAP blocks with bits at both block borders
        for nb in range(n_blocks - 1):
            w = rng.integers(0, 2**32, 2048, dtype=np.uint64).astype(np.uint32) | rng.integers(0, 2**32, 2048, dtype=np.uint64).astype(np.uint32)
            w[0] |= 1; w[2047] |= 0x80000000
            if nb % 2:
                v.set_bits(nb, w)
        v.kind[n_blocks - 1] = bm.BLK_NULL; v.blocks.pop(n_blocks - 1, None)    # spare column for the carry out of the last block
    for v in vecs:
        v.kind[n_blocks - 1] = bm.BLK_NULL; v.blocks.pop(n_blocks - 1, None)
    return vecs


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_shift_right_and_oracle_matches_reference(seed):
    """orc_aggregate(OP_SHIFT_R_AND) == aggregator::combine_shift_right_and on real bvectors (bits, kinds, GAP bytes)."""
    vecs = shift_and_inputs(seed)
    ps = bm.PackedSet.pack(vecs)
    rng = np.random.default_rng(seed)
    for n in (1, 2, 3, 7, 10, 40):
        g = rng.integers(0, len(vecs), n) if n > len(vecs) else rng.permutation(len(vecs))[:n]
        for flags in (0, bm.F_OPT_COMPRESS):
            okind, opop, odig, onr, oblk, ogap = orclib.oracle_aggregate(ps, bm.OP_SHIFT_R_AND, g, None, flags)
            rkind, rpop, rblk, rgap, rany = ra.ref_aggregate(ps, bm.OP_SHIFT_R_AND, g, None, flags)
            assert same(oblk, rblk), f"n={n}"
            assert same(opop, rpop) and rany == bool(opop.sum())
            assert same(okind, rkind)
            assert same(ogap, rgap)
    # closed form: result[p] = AND_k v_k[p - (n-1-k)]
    g = [0, 1, 2]
    _, _, _, _, oblk, _ = orclib.oracle_aggregate(ps, bm.OP_SHIFT_R_AND, g, None, 0)
    bits = [np.unpackbits(np.concatenate([vecs[v].block_words(c) for c in range(ps.n_blocks)]).view(np.uint8), bitorder="little") for v in g]
    want = np.roll(bits[0], 2) & np.roll(bits[1], 1) & bits[2]
    want[:2] = 0                                        # v_0 contributes zeros shifted in from before position 0
    got = np.unpackbits(oblk.reshape(-1).view(np.uint8), bitorder="little")
    assert got.any() and same(got, want)


def blob_inputs(seed=5, n_blocks=12):
    """Vectors that make the serializer pick every explicit-length block encoding: mixed kinds, edge GAP blocks, a single-bit
    block, a narrow interval, sparse words (0-runs / digest0), an almost-full block, long zero / one block runs."""
    rng = np.random.default_rng(seed)
    vecs = gen.mixed_vectors(rng, 10, n_blocks, p_null=0.15, p_full=0.15, p_gap=0.4) + gen.edge_vectors(n_blocks)
    v = bm.BVector(n_blocks)
    w = np.zeros(2048, np.uint32); w[100] = 1 << 7; v.set_bits(0, w)
    w = np.zeros(2048, np.uint32); w[500:520] = rng.integers(1, 2**32, 20, dtype=np.uint64).astype(np.uint32); v.set_bits(1, w)
    w = np.zeros(2048, np.uint32); w[::64] = 0xFFFF0000; v.set_bits(2, w)
    w = np.full(2048, 0xFFFFFFFF, np.uint32); w[7] = 0xFFFFFFF7; v.set_bits(3, w)
    w = np.zeros(2048, np.uint32); w[3] = 5; w[900] = 1 << 31; w[2047] = 1; v.set_bits(4, w)
    for nb in range(6, n_blocks):
        v.set_full(nb)
    vecs.append(v)
    v = bm.BVector(n_blocks); v.set_gap(n_blocks - 1, gen.gap_from_runs([65534, 65535], 0)); v.set_gap(0, gen.gap_from_runs([0, 65535], 1)); vecs.append(v)
    return vecs


def entropy_inputs(seed=20260923):
    """The vectors behind tests/golden/blobs_entropy.npz (tests/gen.entropy_vectors)."""
    return gen.entropy_vectors(np.random.default_rng(seed))


# entropy-coded tokens the serializer of this reference version emits at levels 3..6 (measured); all must be met by the corpus
ENTROPY_TOKENS = (21, 23, 61, 62, 63, 65, 66, 67, 68)


@needs_serializer
def test_deserialize_oracle_matches_reference():
    """orc_deserialize == bm::deserialize on BLOBs written by bm::serializer<> at every compression level (0..6): bits, block
    kinds and GAP bytes, over vectors that make the serializer use every encoding it has (token histogram checked)."""
    hist = orclib.oracle_token_hist()
    seen = np.zeros(256, np.uint64)
    for vecs in (blob_inputs(), entropy_inputs(), entropy_inputs(7)):
        ps = bm.PackedSet.pack(vecs)
        for level in range(0, 7):
            for v in range(ps.n_vec):
                blob = ra.ref_serialize(ps, v, level)
                rkind, rpop, rblk, rgap = ra.ref_deserialize(blob, ps.n_blocks)
                assert same(rblk, np.stack([vecs[v].block_words(c) for c in range(ps.n_blocks)]))
                rc, kind, blk, gaps = orclib.oracle_deserialize(blob, ps.n_blocks)
                assert rc == 0, f"level {level} vector {v}: rc={rc}"
                assert same(blk, rblk) and same(kind, rkind) and same(gaps, rgap), f"level {level} vector {v}"
    seen += hist
    orclib.oracle_token_hist(False)
    for t in ENTROPY_TOKENS + (11, 16, 18, 19, 22, 24, 30, 34):
        assert seen[t] > 0, f"serializer token {t} not exercised"
    vecs = blob_inputs(); ps = bm.PackedSet.pack(vecs)
    # truncated / corrupt streams are rejected, not read past the end
    blob = ra.ref_serialize(ps, 0, 2)
    assert orclib.oracle_deserialize(blob[: blob.size // 2], ps.n_blocks)[0] != 0


@needs_serializer
def test_64bit_address_blobs_oracle_and_device_decoder_host_build():
    """BLOBs written by the BM64ADDR build of the reference (BM_HM_64_BIT header, 64-bit size field and block-run counts): the oracle
    and the host build of the product's walker / decoder == the BM64ADDR bm::deserialize."""
    for vecs in (blob_inputs(), entropy_inputs(3)):
        ps = bm.PackedSet.pack(vecs)
        for level in (0, 2, 4, 6):
            for v in range(ps.n_vec):
                blob = ra.ref_serialize(ps, v, level, addr64=True)
                assert blob[0] & (1 << 5)
                rkind, rpop, rblk, rgap = ra.ref_deserialize(blob, ps.n_blocks, addr64=True)
                assert same(rblk, np.stack([vecs[v].block_words(c) for c in range(ps.n_blocks)]))
                rc, kind, blk, gaps = orclib.oracle_deserialize(blob, ps.n_blocks)
                assert rc == 0 and same(blk, rblk) and same(kind, rkind) and same(gaps, rgap), f"level {level} vector {v}"
                rc, kind, dec, gw, blk, gaps, n = orclib.blob_host_check(blob, ps.n_blocks)
                assert rc == 0 and same(kind, rkind), f"level {level} vector {v}"
                for c in np.flatnonzero(dec):
                    assert same(blk[c], rblk[c]) if kind[c] == bm.BLK_BIT else same(gaps[c], rgap[c])


@needs_serializer
def test_bookmarked_blobs_oracle_and_device_decoder_host_build():
    """BLOBs written with serializer::set_bookmarks(true, interval): the oracle skips the marks; the product's walker cuts the stream
    at them (ent_find_segments) and walks every segment on its own -- both == bm::deserialize."""
    vecs = gen.entropy_vectors(np.random.default_rng(5), n_vec=8, n_blocks=40)
    ps = bm.PackedSet.pack(vecs)
    max_segments = 0
    for level in (2, 4, 6):
        for interval in (4, 16):
            for v in range(ps.n_vec):
                blob = ra.ref_serialize_bookmarks(ps, v, level, interval)
                rkind, rpop, rblk, rgap = ra.ref_deserialize(blob, ps.n_blocks)
                assert same(rblk, np.stack([vecs[v].block_words(c) for c in range(ps.n_blocks)]))
                rc, kind, blk, gaps = orclib.oracle_deserialize(blob, ps.n_blocks)
                assert rc == 0 and same(blk, rblk) and same(kind, rkind) and same(gaps, rgap)
                rc, kind, dec, gw, blk, gaps, n = orclib.blob_host_check(blob, ps.n_blocks)
                assert rc == 0 and same(kind, rkind), f"level {level} interval {interval} vector {v}"
                max_segments = max(max_segments, orclib.blob_host_check.last_segments)
                for c in np.flatnonzero(dec):
                    assert same(blk[c], rblk[c]) if kind[c] == bm.BLK_BIT else same(gaps[c], rgap[c])
    assert max_segments >= 8


@needs_serializer
def test_device_decoder_host_build_matches_reference():
    """The product's BLOB walker + entropy decoder (bitmagic_b200/csrc/blob_entropy.cuh), built for the host as a checker
    (oracle/blob_host_check.cpp: same functions, a team of one lane instead of a warp), == bm::deserialize: block kinds for every
    block, and for every block that came from an entropy-coded token the exact bits / GAP words pass 2 stores in the arena."""
    n_ent = 0
    for vecs in (blob_inputs(), entropy_inputs(), entropy_inputs(7)):
        ps = bm.PackedSet.pack(vecs)
        for level in range(0, 7):
            for v in range(ps.n_vec):
                blob = ra.ref_serialize(ps, v, level)
                rkind, rpop, rblk, rgap = ra.ref_deserialize(blob, ps.n_blocks)
                rc, kind, dec, gw, blk, gaps, n = orclib.blob_host_check(blob, ps.n_blocks)
                assert rc == 0, f"level {level} vector {v}: rc={rc}"
                n_ent += n
                assert same(kind, rkind), f"level {level} vector {v}: kinds"
                for c in np.flatnonzero(dec):
                    if kind[c] == bm.BLK_BIT:
                        assert same(blk[c], rblk[c]), f"level {level} vector {v} column {c}: bits"
                    else:
                        assert same(gaps[c], rgap[c]), f"level {level} vector {v} column {c}: GAP words"
    assert n_ent > 500
    # truncated streams and a header the decoder does not cover are rejected
    vecs = entropy_inputs(); ps = bm.PackedSet.pack(vecs)
    blob = ra.ref_serialize(ps, 2, 5)
    assert orclib.blob_host_check(blob[: blob.size // 2], ps.n_blocks)[0] != 0
    bad = blob.copy(); bad[0] |= 1 << 6                           # BM_HM_HXOR: XOR-reference compression is not covered
    assert orclib.blob_host_check(bad, ps.n_blocks)[0] == 202


def test_c1_config_bit_and_count():
    """BASELINE configs[0]: two bvectors of 2^20 bits, 10 % random fill: t.bit_and(a, b, opt_none); t.count() and bm::count_and(a, b)
    on the reference == the oracle (the reference's own CPU-runnable case; the GPU runs it in test_gpu_parity.py)."""
    vecs = gen.c1_vectors()
    ps = bm.PackedSet.pack(vecs)
    rkind, rpop, rblk, rcnt = ra.ref_binop(ps, 1, 0, 1)
    okind, opop, odig, onr, oblk, ogap = orclib.oracle_aggregate(ps, bm.OP_AND, [0, 1], None, 0)
    want = np.stack([vecs[0].block_words(c) & vecs[1].block_words(c) for c in range(16)])
    assert same(rblk, want) and same(oblk, want) and same(okind, rkind)
    assert rcnt == int(opop.sum()) == ra.ref_count_op(ps, 1, 0, 1) == int(np.unpackbits(want.view(np.uint8)).sum())
    assert 9000 < rcnt < 12000                                      # 2^20 * 0.01 = 10 486 expected


@needs_serializer
def test_multi_superblock_blobs_with_bookmarks():
    """BLOBs that span more than one 256-block super-block (super-block position lists next to ordinary tokens, 24-bit bookmark offsets,
    sync marks): oracle and the host build of the product's decoder == bm::deserialize."""
    rng = np.random.default_rng(31)
    nbk = 270
    vecs = gen.entropy_vectors(rng, n_vec=5, n_blocks=nbk)
    v = bm.BVector(nbk)
    for nb in range(0, nbk, 3):
        bits = np.zeros(65536, np.uint8); bits[rng.choice(65536, size=int(rng.integers(1, 30)), replace=False)] = 1
        v.set_gap(nb, bm.hostfmt.bits_to_gap(bm.hostfmt.bits_to_words(bits)))
    vecs.append(v)
    ps = bm.PackedSet.pack(vecs)
    n_ent = 0
    for level, interval in ((5, 0), (6, 16), (6, 256)):
        for vi in range(ps.n_vec):
            blob = ra.ref_serialize_bookmarks(ps, vi, level, interval) if interval else ra.ref_serialize(ps, vi, level)
            rkind, rpop, rblk, rgap = ra.ref_deserialize(blob, ps.n_blocks)
            rc, kind, blk, gaps = orclib.oracle_deserialize(blob, ps.n_blocks)
            assert rc == 0 and same(blk, rblk) and same(kind, rkind) and same(gaps, rgap), f"oracle: level {level} vector {vi}"
            rc, kind, dec, gw, blk, gaps, n = orclib.blob_host_check(blob, ps.n_blocks)
            assert rc == 0 and same(kind, rkind), f"decoder: level {level} vector {vi}"
            n_ent += n
            for c in np.flatnonzero(dec):
                assert same(blk[c], rblk[c]) if kind[c] == bm.BLK_BIT else same(gaps[c], rgap[c])
    assert n_ent > 1000


def test_host_synth_blocks_are_what_optimize_stores():
    """The benchmark generator, host form (oracle/bm_synth.c): its optimize()d set must hold exactly what the REAL
    bvector::optimize(opt_compress) makes of the raw (all bit-block) set -- block kinds, GAP words, bits -- so 'stored the way
    optimize() would store it' is pinned on the reference, not on the generator's own threshold.  Also: AVX-512 form == scalar form."""
    nv, nb = 40, 6
    dens = np.array([0.5 / (k + 1) for k in range(nv)]); dens[7] = 0.0; dens[9] = 1.0; dens[11] = 0.0098; dens[12] = 0.0097   # 11/12 straddle the 1276-run threshold
    seed = np.arange(1000, 1000 + nv, dtype=np.uint64)
    opt = orclib.HostSynth(nv, nb, dens, seed, True, threads=3)
    raw = orclib.HostSynth(nv, nb, dens, seed, False, threads=2)
    kinds_seen = set()
    for v in range(nv):
        kind, pop, blocks, gaps = ra.ref_optimize(raw.ps, v)
        for c in range(nb):
            k, data = opt.ps.block(v, c)
            assert k == kind[c], f"vector {v} block {c}: generator stores kind {k}, optimize() makes {kind[c]}"
            kinds_seen.add(int(k))
            if k == bm.BLK_GAP:
                n = (int(np.asarray(data)[0]) >> 3) + 1
                assert same(np.pad(np.asarray(data), (0, orclib.GAP_MAX_WORDS - n)), gaps[c])
            elif k == bm.BLK_BIT:
                assert same(np.asarray(data), blocks[c])
    assert kinds_seen == {bm.BLK_NULL, bm.BLK_FULL, bm.BLK_BIT, bm.BLK_GAP}
    k11 = {int(opt.ps.block(11, c)[0]) for c in range(nb)} | {int(opt.ps.block(12, c)[0]) for c in range(nb)}
    assert k11 == {bm.BLK_BIT, bm.BLK_GAP}, "the threshold vectors should produce both kinds"
    orclib.oracle().orc_synth_force_scalar(1)
    try:
        sc = orclib.HostSynth(nv, nb, dens, seed, True, threads=4)
    finally:
        orclib.oracle().orc_synth_force_scalar(0)
    for a in ("desc", "bit_base", "gap_base", "bit_pool", "gap_pool"):
        assert same(getattr(sc.ps, a), getattr(opt.ps, a)), a


def test_ref_job_matches_oracle_all_columns():
    """The persistent reference job bench.py uses for its all-column parity (T workers, bvectors built once): kind / popcount /
    digest / GAP length of every column equal the C oracle's, for ragged worker ranges, with and without opt_compress."""
    nv, nb = 48, 11
    dens = np.array([0.5 / (k + 1) for k in range(nv)])
    seed = np.arange(77, 77 + nv, dtype=np.uint64)
    hs = orclib.HostSynth(nv, nb, dens, seed, True, threads=2)
    for op, g0, g1, flags in ((bm.OP_AND_SUB, [0, 1], list(range(2, nv)), bm.F_OPT_COMPRESS), (bm.OP_OR, list(range(5, nv)), None, bm.F_OPT_COMPRESS),
                              (bm.OP_OR, list(range(20, nv)), None, bm.F_OPT_NONE), (bm.OP_AND, [3, 4, 5], None, bm.F_OPT_COMPRESS)):
        ok, op_, od, onr, _, _ = orclib.oracle_aggregate(hs.ps, op, g0, g1, flags)
        for threads in (1, 3, 11):
            tot, k, p, d, gl = ra.ref_job(hs.ps, op, g0, g1, flags, threads=threads)
            assert tot == int(op_.sum())
            assert same(k, ok) and same(p, op_) and same(d, od)
            assert same(gl, np.where(ok == bm.BLK_GAP, onr, 0))


def test_superblock_members_at_the_gap_capacity_levels():
    """Members of a super-block token (set_sblock_bienc_v3) are rebuilt with set_bit_no_check under BM_GAP (gap_block_set_no_ret,
    src/bm.h:4800): a block stays GAP while runs <= 1276 and sits on the smallest level with runs <= glen[level] - 4 -- NOT the
    deserialize_gap rule (gap_calc_level(runs + 1)).  Oracle and the host build of the product's decoder == bm::deserialize, headers included."""
    v = gen.superblock_threshold_vector()
    ps = bm.PackedSet.pack([v])
    for level in (5, 6):
        blob = ra.ref_serialize(ps, 0, level)
        h = orclib.oracle_token_hist(True)
        rkind, rpop, rblk, rgap = ra.ref_deserialize(blob, ps.n_blocks)
        rc, kind, blk, gaps = orclib.oracle_deserialize(blob, ps.n_blocks)
        orclib.oracle_token_hist(False)
        assert h[68] == 1, "the vector should serialize as one super-block token"
        assert rc == 0 and same(kind, rkind) and same(blk, rblk) and same(gaps, rgap)
        by_runs = {r: (int(kind[2 * i]), (int(gaps[2 * i][0]) >> 1) & 3) for i, r in enumerate(gen.SB_MEMBER_RUNS)}   # == the reference's
        assert by_runs[124] == (bm.BLK_GAP, 0) and by_runs[125] == (bm.BLK_GAP, 1) and by_runs[252] == (bm.BLK_GAP, 1) and by_runs[508] == (bm.BLK_GAP, 2)
        assert by_runs[1276] == (bm.BLK_GAP, 3) and by_runs[1277][0] == bm.BLK_BIT
        rc, kind, dec, gw, blk, gaps, n = orclib.blob_host_check(blob, ps.n_blocks)
        assert rc == 0 and same(kind, rkind)
        for c in np.flatnonzero(dec):
            assert same(blk[c], rblk[c]) if kind[c] == bm.BLK_BIT else same(gaps[c], rgap[c])
