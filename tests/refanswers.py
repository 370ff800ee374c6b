"""The unmodified reference's answers, live or recorded.

Tests that compare against the reference call these functions instead of ``orclib.ref_*``.  Where the reference library
(oracle/_ref/, compiled from the reference sources) is present, the call runs it; everywhere else the answer comes from
tests/golden/ref_answers*.npz, recorded from the same library on the same inputs.  A call is found again by a SHA-256 of its
function name and every argument (packed sets included), so an answer is only ever used for exactly the inputs it was
computed on; a call that was never recorded fails, it does not skip.

Large output arrays are kept as a SHA-256 of their values (``Digest``): tests compare them with ``same()``, which is an exact
equality test either way.  Outputs a test reads element by element are kept in full.

Recording: with the reference library present, run the tests with ``BMB200_REF_RECORD=<file.npz>``; every answer the run
needs is written there when the process ends.
"""
from __future__ import annotations

import atexit
import hashlib
import json
import os
from pathlib import Path

import numpy as np

import orclib

GOLDEN = Path(__file__).resolve().parent / "golden"
DIGEST_ABOVE = 1024          # output arrays larger than this many bytes are kept as a digest unless kept in full


class Digest:
    """SHA-256 of an integer / bool array's values and shape (dtype-independent, like np.array_equal)."""

    def __init__(self, hexdigest: str):
        self.hex = hexdigest

    @classmethod
    def of(cls, a) -> "Digest":
        if isinstance(a, Digest):
            return a
        a = np.asarray(a)
        h = hashlib.sha256(repr(a.shape).encode())
        h.update(memoryview(np.ascontiguousarray(a.astype(np.uint64, copy=False))).cast("B"))
        return cls(h.hexdigest()[:32])

    def __eq__(self, other):
        if not isinstance(other, Digest):
            return NotImplemented
        n = min(len(self.hex), len(other.hex))
        return n >= 16 and other.hex[:n] == self.hex[:n]

    def __hash__(self):
        return hash(self.hex[:16])

    def __repr__(self):
        return f"Digest({self.hex[:16]})"


def same(a, b) -> bool:
    """np.array_equal that also accepts a Digest, or a list of row digests, on either side."""
    if isinstance(b, list) and b and isinstance(b[0], Digest):
        a, b = b, a
    if isinstance(a, list) and a and isinstance(a[0], Digest):
        return len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    if isinstance(a, Digest) or isinstance(b, Digest):
        return Digest.of(a) == Digest.of(b)
    return bool(np.array_equal(a, b))


# ------------------------------------------------------------------------------------------------------------ call keys
def _feed(h, x):
    if isinstance(x, np.ndarray):
        h.update(b"A" + x.dtype.str.encode() + repr(x.shape).encode())
        h.update(memoryview(np.ascontiguousarray(x)).cast("B"))
    elif hasattr(x, "bit_pool") and hasattr(x, "desc"):              # hostfmt.PackedSet
        h.update(b"P%d,%d" % (x.n_vec, x.n_blocks))
        for a in (x.desc, x.bit_base, x.gap_base, x.bit_pool, x.gap_pool):
            _feed(h, np.asarray(a))
    elif isinstance(x, (list, tuple, range)):
        h.update(b"L%d[" % len(x))
        for y in x:
            _feed(h, y)
        h.update(b"]")
    elif isinstance(x, dict):
        for k in sorted(x):
            h.update(str(k).encode() + b"=")
            _feed(h, x[k])
    elif isinstance(x, np.generic):
        _feed(h, x.item())
    elif x is None or isinstance(x, (bool, int, float, str)):
        h.update(b"S" + repr(x).encode())
    else:
        raise TypeError(f"cannot key a reference call on {type(x).__name__}")


def call_key(name, args, kw) -> str:
    h = hashlib.sha256(name.encode())
    _feed(h, list(args))
    _feed(h, kw)
    return h.hexdigest()[:32]


# ------------------------------------------------------------------------------------------------------------ the store
_store = None
_recorded = {}
_record_to = os.environ.get("BMB200_REF_RECORD")


def _load():
    global _store
    if _store is None:
        _store = {}
        for f in sorted(GOLDEN.glob("ref_answers*.npz")):
            z = np.load(f, allow_pickle=False)
            for key, spec in json.loads(str(z["__index__"])).items():
                _store[key] = (spec, z)
    return _store


def _encode(out, keep, small=DIGEST_ABOVE):
    """-> (json spec, {name: array}) of one call's output; arrays beyond `small` bytes become digests unless kept."""
    single = not isinstance(out, tuple)
    items = (out,) if single else out
    spec, arrays = [], {}
    for i, x in enumerate(items):
        if isinstance(x, np.ndarray) and not (keep is True or i in keep) and x.nbytes > small:
            spec.append(["d", Digest.of(x).hex])
        elif isinstance(x, np.ndarray):
            spec.append(["a", i]); arrays[str(i)] = x
        elif isinstance(x, Digest):
            spec.append(["d", x.hex])
        elif isinstance(x, list) and x and isinstance(x[0], Digest):
            spec.append(["r", [d.hex[:16] for d in x]])
        else:
            spec.append(["s", x.item() if isinstance(x, np.generic) else x])
    return {"single": single, "items": spec}, arrays


def _decode(spec, get):
    items = []
    for tag, v in spec["items"]:
        items.append(Digest(v) if tag == "d" else [Digest(d) for d in v] if tag == "r" else get(v) if tag == "a" else v)
    return items[0] if spec["single"] else tuple(items)


def _dump():
    if not _recorded:
        return
    index, arrays = {}, {}
    for key, (spec, arrs) in _recorded.items():
        index[key] = spec
        for n, a in arrs.items():
            arrays[f"{key}.{n}"] = a
    np.savez_compressed(_record_to, __index__=np.array(json.dumps(index)), **arrays)


if _record_to:
    atexit.register(_dump)


def answer(name, fn, args, kw, keep=(), variant=False, rows=(), small=DIGEST_ABOVE):
    """The reference's answer to fn(*args, **kw): live when its library is present, else recorded.  Outputs listed in
    `rows` are kept as one digest per row (a list of Digest)."""
    key = call_key(name, args, kw)
    if orclib.have_ref(variant):
        out = fn(*args, **kw)
        if rows:
            out = tuple([Digest.of(r) for r in x] if i in rows else x for i, x in enumerate(out))
        spec, arrays = _encode(out, keep, small)
        spec["fn"] = name
        if _record_to and key not in _load():
            _recorded[key] = (spec, arrays)
        return _decode(json.loads(json.dumps(spec)), lambda i: arrays[str(i)])
    store = _load()
    assert key in store, (f"no recorded reference answer for {name} on these inputs (key {key}); record it with the reference "
                          "library present and BMB200_REF_RECORD=<file> (see tests/refanswers.py)")
    spec, z = store[key]
    return _decode(spec, lambda i: z[f"{key}.{i}"])


def _wrap(name, keep=(), variant_kw=None, rows=(), small=DIGEST_ABOVE):
    fn = getattr(orclib, name)

    def f(*args, **kw):
        variant = kw.get(variant_kw, False) if variant_kw else False
        return answer(name, fn, args, kw, keep, variant, rows, small)
    f.__name__ = name
    f.__doc__ = fn.__doc__
    return f


ref_aggregate = _wrap("ref_aggregate", variant_kw="addr64")
ref_binop = _wrap("ref_binop", small=0)
ref_count_op = _wrap("ref_count_op")
ref_optimize = _wrap("ref_optimize", keep=(0,), rows=(2, 3))
ref_pipeline = _wrap("ref_pipeline")
ref_sv_scan = _wrap("ref_sv_scan")
ref_serialize = _wrap("ref_serialize", keep=True, variant_kw="addr64")
ref_serialize_bookmarks = _wrap("ref_serialize_bookmarks", keep=True)
ref_deserialize = _wrap("ref_deserialize", variant_kw="addr64", rows=(2, 3))


def ref_rank_select(ps, v, pos, rank, addr64=False):
    """-> rank_out, pos_out (0 where not found), found: the reference's count_to / select (timings dropped)."""
    def run(ps, v, pos, rank, addr64=False):
        rr, rp, rf, _ = orclib.ref_rank_select(ps, v, pos, rank, addr64=addr64)
        return rr, np.where(rf, rp, 0).astype(np.uint64), rf
    return answer("ref_rank_select", run, (ps, v, pos, rank), dict(addr64=addr64), variant=addr64)


def ref_rs_build(ps, v, addr64=False):
    """-> bcount, sub_count (0 where bcount is 0: the reference leaves it undefined there), superblock counts, total"""
    def run(ps, v, addr64=False):
        bc, sc, sb, tot = orclib.ref_rs_build(ps, v, addr64=addr64)
        return bc, np.where(bc > 0, sc, 0).astype(np.uint64), sb, tot
    return answer("ref_rs_build", run, (ps, v), dict(addr64=addr64), variant=addr64)


def ref_job(ps, op, g0, g1=None, flags=0, threads=1):
    """The persistent reference job (orclib.RefJob) on `threads` workers, two passes -> total, kind, popcnt, digest and
    gap_len (0 where the column is not GAP) of every column."""
    def run(ps, op, g0, g1, flags, threads):
        job = orclib.RefJob(ps, op, g0, g1, flags, threads=threads)
        try:
            _, tot = job.run(2)
            k, p, d, gl = job.export()
            return tot, k, p, d, np.where(k == 3, gl, 0).astype(np.uint32)
        finally:
            job.free()
    return answer("ref_job", run, (ps, op, g0, g1, flags, threads), {})


def ref_sv_planes(values, nulls=None):
    """The reference bm::sparse_vector<unsigned>'s optimize()d planes + universe.  Returned as the host mirror's planes
    (bitmagic_b200.SparseVector) after checking that, packed, they equal the reference's planes array for array."""
    import bitmagic_b200 as bm

    def packed(planes):
        ps = bm.PackedSet.pack(planes)
        return (len(planes),) + tuple(Digest.of(a) for a in (ps.desc, ps.bit_base, ps.gap_base, ps.bit_pool, ps.gap_pool))
    sv = bm.SparseVector.from_values(values, nulls)
    mine = sv.planes + [sv.universe()]
    want = answer("ref_sv_planes", lambda v, n: packed(orclib.ref_sv_planes(v, n)), (values, nulls), {})
    assert packed(mine) == want, "the host mirror's planes differ from the reference sparse_vector's"
    return mine
