"""Pins the oracle's restatement against the REFERENCE'S OWN OBJECT CODE.

oracle/ref/Makefile compiles a few of the reference's leaf source files into
oracle/_ref/libotbref.so (hashfunc.c, pg_crc32c_sb8.c, bloomfilter.c,
heaptuple.c, bufpage.c, float.c, int8.c, locator.c, fnbufpage.c).
tests/golden/make_oracle_vs_ref_vectors.py ran that object code on the inputs
below and stored its answers in tests/golden/oracle_vs_ref.npz; every
comparison here is against those stored answers, so the tests run without the
reference.  Outputs too large to store (bloom filter words, forward-node pages)
are compared through SHA-256 digests of their bytes."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_ref.npz")


@pytest.fixture(scope="module")
def R():
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


# ---- the inputs (shared with the generator, which fed them to the reference)
def hash_inputs():
    rng = np.random.default_rng(42)
    i4 = [0, 1, -1, 17, 42, 2**31 - 1, -2**31] + rng.integers(-2**31, 2**31, 3000).tolist()
    i8 = [0, 1, -1, 2**32 + 1, -2**32, 2**63 - 1, -2**63] + rng.integers(-2**63, 2**63 - 1, 3000).tolist()
    f8 = [0.0, -0.0, 1.0, -1.5, 1e300, float("inf")] + rng.normal(0, 1e6, 500).tolist()
    blobs = [bytes(rng.integers(0, 256, n).astype(np.uint8)) for n in list(range(0, 40)) + [63, 64, 65, 255]]
    pairs = rng.integers(0, 2**32, (200, 2))
    return {"i4": np.array(i4, np.int64), "i8": np.array(i8, np.int64), "f8": np.array(f8), "blobs": blobs, "pairs": pairs}


def hash_inputs_digest(h):
    return digest(h["i4"], h["i8"], h["f8"], np.frombuffer(b"".join(h["blobs"]), np.uint8), h["pairs"].astype(np.int64))


BLOOM_ROWS = (10, 1000, 100000, 3000000)


def bloom_keys(nrows):
    L = O.lib()
    return [L.orc_hashint8new(i * 7919) for i in range(min(nrows, 5000))]


def bloom_probes():
    L = O.lib()
    return [L.orc_hashint8new(i) for i in range(2000)]


def float8_inputs():
    import opentenbase_b200 as g
    rng = np.random.default_rng(9)
    # (1e300 would make Sxx overflow: the reference raises ERROR there, the oracle reports status 6)
    vals = np.concatenate([rng.normal(1000, 300, 4000), [0.0, -0.0, 1e-300, 1e150, -1e150]])
    plan = O.make_plan(aggs=[(g.GX_AGG_AVG_F8, [(g.GX_OP_COL, 0, 0)]), (g.GX_AGG_SUM_F8, [(g.GX_OP_COL, 0, 0)])])
    return vals, plan


ATT = {O.GX_INT8: (8, 8), O.GX_INT4: (4, 4), O.GX_FLOAT8: (8, 8), O.GX_DATE: (4, 4), O.GX_CHAR: (1, 1), O.ORC_BPCHAR1: (-1, 4)}


def attrs(types):
    return ((C.c_int16 * len(types))(*[ATT[t][0] for t in types]), (C.c_int8 * len(types))(*[ATT[t][1] for t in types]))


def heap_inputs():
    rng = np.random.default_rng(13)
    types = [O.GX_INT8, O.GX_INT4, O.ORC_BPCHAR1, O.ORC_BPCHAR1, O.GX_FLOAT8, O.GX_CHAR, O.GX_DATE, O.GX_INT8]
    n = 400
    cols = [rng.integers(-2**62, 2**62, n), rng.integers(-2**31, 2**31, n).astype(np.int32),
            rng.integers(65, 90, n).astype(np.int8), rng.integers(65, 90, n).astype(np.int8), rng.normal(size=n),
            rng.integers(32, 127, n).astype(np.int8), rng.integers(-3000, 0, n).astype(np.int32), rng.integers(0, 2**40, n)]
    nulls = [None] + [(rng.random(n) < 0.25).astype(np.uint8) for _ in range(7)]
    nulls[4][:50] = 0
    for k in range(1, 8):
        nulls[k][:20] = 0                               # some tuples without any NULL (t_hoff 48)
    return types, cols, nulls


def heap_inputs_digest(cols, nulls):
    return digest(*cols, *[x for x in nulls if x is not None])


def heap_row(types, cols, nulls, i):
    """row i as the Datum words and isnull flags heap_form_tuple takes"""
    vals = (C.c_int64 * len(types))(*[int(np.asarray(c)[i].view(np.int64)) if np.asarray(c).dtype == np.float64 else int(np.asarray(c)[i]) for c in cols])
    isn = (C.c_uint8 * len(types))(*[0 if x is None else int(x[i]) for x in nulls])
    return vals, isn


FNPAGE_ID = (123456789012345, -7, 12, 3, 1, 2, 1)


def fnpage_inputs():
    rng = np.random.default_rng(99)
    cases = []
    for types, n, frac in [([O.GX_INT8, O.GX_INT8, O.GX_DATE, O.GX_INT4], 5000, 0.0),
                           ([O.GX_INT8, O.GX_INT4, O.ORC_BPCHAR1, O.GX_FLOAT8, O.GX_CHAR, O.GX_DATE, O.ORC_BPCHAR1, O.GX_INT8, O.GX_INT4], 3000, 0.2),
                           ([O.GX_CHAR], 700, 0.5), ([O.GX_FLOAT8] * 12, 900, 0.1)]:
        vals = np.zeros((n, len(types)), np.int64)
        for i, t in enumerate(types):
            vals[:, i] = (rng.integers(-2**62, 2**62, n) if t in (O.GX_INT8, O.GX_FLOAT8) else
                          rng.integers(-2**31, 2**31 - 1, n) if t in (O.GX_INT4, O.GX_DATE) else rng.integers(-128, 127, n))
        isn = (rng.random((n, len(types))) < frac).astype(np.uint8)
        isn[:40] = 0
        cases.append((types, n, vals, isn))
    return cases


# ---- the tests
def test_struct_layout_constants(R):
    flags, lower, upper, special, psv, linp, itemid, ctid, im2, bits = R["layout_page_offsets"].tolist()
    assert (flags, lower, upper, special, psv, linp, itemid) == (10, 16, 20, 24, 28, 44, 4)     # orc_heap.c PD_* / ORC_PAGE_HDR
    assert (ctid, im2, bits) == (32, 38, 47)                                                      # orc_internal.h HTH_*
    heap_header, hoff, infomask, minimal_header, minimal_offset, fnpage_header, invalid_shard = R["layout_sizes"].tolist()
    assert heap_header == 47 and hoff == 46 and infomask == 40
    assert minimal_header == 15 and minimal_offset == 32
    assert fnpage_header == 32 and invalid_shard == 4096


def test_hash_functions_against_reference_objects(R):
    L = O.lib()
    h = hash_inputs()
    np.testing.assert_array_equal(hash_inputs_digest(h), R["hash_inputs_digest"], err_msg="input stream changed: regenerate the vectors")
    i4, i8 = h["i4"].tolist(), h["i8"].tolist()
    for v, want in zip(i4, R["hash_i4"].tolist()):
        assert [L.orc_hashint4(v), L.orc_hashint4new(v), L.orc_hash_uint32(v & 0xFFFFFFFF), L.orc_murmurhash32(v & 0xFFFFFFFF),
                L.orc_evaluate_hashkey((C.c_int * 1)(O.GX_INT4), None, (C.c_int64 * 1)(v), 1)] == want, v
    for v, want in zip(i8, R["hash_i8"].tolist()):
        assert [L.orc_hashint8(v), L.orc_hashint8new(v),
                L.orc_evaluate_hashkey((C.c_int * 1)(O.GX_INT8), None, (C.c_int64 * 1)(v), 1)] == want, v
    for v, want in zip(range(-128, 128), R["hash_char"].tolist()):
        assert [L.orc_hashchar(v), L.orc_hashcharnew(v)] == want, v
    for v, want in zip(h["f8"].tolist(), R["hash_f8"].tolist()):
        assert [L.orc_hashfloat8(v), L.orc_hashfloat8new(v)] == want, v
    for b, want in zip(h["blobs"], R["hash_any"].tolist()):
        assert [L.orc_hash_any(b, len(b)), L.orc_hash_any_new(b, len(b))] == want, len(b)
    for (a, b), want in zip(h["pairs"].tolist(), R["hash_combine"].tolist()):
        assert L.orc_hash_combine(a, b) == want
    # two-column distribution key: rotate-then-xor order (locator.c:1611-1628)
    for a, b, want in zip(i8[:200], i4[:200], R["hash_key2"].tolist()):
        assert L.orc_evaluate_hashkey((C.c_int * 2)(O.GX_INT8, O.GX_INT4), None, (C.c_int64 * 2)(a, b), 2) == want
    # NULL distribution value hashes to 0 -> shard 0
    assert R["hash_key1_null"][0] == 0 == L.orc_evaluate_hashkey((C.c_int * 1)(O.GX_INT8), (C.c_uint8 * 1)(1), (C.c_int64 * 1)(12345), 1)


def test_bloom_filter_against_reference_object(R):
    L = O.lib()
    found = iter(R["bloom_find"])
    for nrows, logb, nwords, words in zip(R["bloom_rows"].tolist(), R["bloom_log_num_buckets"].tolist(),
                                          R["bloom_nwords"].tolist(), R["bloom_words_digest"]):
        assert nrows in BLOOM_ROWS
        ob = L.orc_bloom_create(nrows)
        assert (logb < 0) == (not ob)
        if logb < 0:
            continue
        assert logb == L.orc_bloom_log_num_buckets(ob)
        for k in bloom_keys(nrows):
            L.orc_bloom_insert(ob, k)
        nw = C.c_int64()
        ow = np.ctypeslib.as_array(C.cast(L.orc_bloom_words(ob, C.byref(nw)), C.POINTER(C.c_uint32)), (nw.value,))
        assert nw.value == nwords
        np.testing.assert_array_equal(digest(ow), words)          # identical bit patterns
        assert [L.orc_bloom_find(ob, p) for p in bloom_probes()] == next(found).tolist()
        L.orc_bloom_free(ob)
    assert R["bloom_1e9_gives_up"][0] == 1 and not L.orc_bloom_create(10**9)      # logNumBuckets > 20: gives up


def test_float8_transition_functions_against_reference_objects(R):
    """float8_accum / float8_combine / float8_avg / float8pl from float.o versus the oracle's
    aggregate states on the same input order."""
    vals, plan = float8_inputs()
    np.testing.assert_array_equal(digest(vals), R["float8_inputs_digest"], err_msg="input stream changed: regenerate the vectors")
    r, raw = O.exec_agg(O.Rel([O.GX_FLOAT8], [vals]), plan, keep_raw=True)
    np.testing.assert_array_equal(r.states[0, 0], R["float8_accum_state"])       # {N, Sx, Sxx} bit-identical
    assert r.aggs[0, 1] == R["float8pl_sum"][0]
    rc, avg = R["float8_avg"].tolist()
    assert rc == 0 and avg == r.aggs[0, 0]
    assert R["float8_avg_empty_rc"][0] == 1                                        # N == 0 -> NULL
    # combine: split the input in two, states must merge exactly like float8_combine
    h = len(vals) // 2
    r1, raw1 = O.exec_agg(O.Rel([O.GX_FLOAT8], [vals[:h]]), plan, keep_raw=True)
    r2, raw2 = O.exec_agg(O.Rel([O.GX_FLOAT8], [vals[h:]]), plan, keep_raw=True)
    np.testing.assert_array_equal(np.array([r1.states[0, 0], r2.states[0, 0]]), R["float8_combine_inputs"])
    comb = O.combine(plan, [raw1, raw2])
    np.testing.assert_array_equal(comb.states[0, 0], R["float8_combine"])
    assert R["float8_mul_mi"].tolist() == [1.1 * 3.3, 1.0 - 0.07]
    assert R["int8inc_41"][0] == 42


def test_heap_tuples_and_pages_against_reference_objects(R):
    """The oracle's heap_form_tuple / PageAddItem restatement produces the bytes the
    reference's heaptuple.o / bufpage.o produce; its deform agrees with heap_deform_tuple."""
    types, cols, nulls = heap_inputs()
    np.testing.assert_array_equal(heap_inputs_digest(cols, nulls), R["heap_inputs_digest"], err_msg="input stream changed: regenerate the vectors")
    rel = O.Rel(types, cols, nulls)
    pages = rel.pages().reshape(-1, 8192)
    # walk the oracle's first page and compare every tuple with the reference's
    pg = pages[0]
    lower = int(pg[16:20].copy().view(np.uint32)[0]); nlines = (lower - 44) // 4
    lens = R["heap_tuple_lens"].tolist()
    assert nlines == len(lens)
    ends = np.cumsum([0] + lens)
    for i in range(nlines):
        lp = int(pg[44 + 4 * i: 48 + 4 * i].copy().view(np.uint32)[0])
        off, ln = lp & 0x7FFF, lp >> 17
        mine = pg[off: off + ln]
        ref = R["heap_tuples"][ends[i]:ends[i + 1]]
        assert lens[i] == ln, f"tuple {i}: oracle length {ln} vs reference {lens[i]}"
        assert mine[46] == ref[46]                                            # t_hoff
        assert (int(mine[38]) | int(mine[39]) << 8) & 0x07FF == (int(ref[38]) | int(ref[39]) << 8) & 0x07FF   # natts
        assert (int(mine[40]) & 0x03) == (int(ref[40]) & 0x03)               # HEAP_HASNULL | HEAP_HASVARWIDTH
        np.testing.assert_array_equal(mine[47:], ref[47:])                   # null bitmap + padding + attribute data
        # the reference's deform of these tuple bytes gives back the inputs
        vals, isn = heap_row(types, cols, nulls, i)
        vo, no = R["heap_deform_vals"][i].tolist(), R["heap_deform_nulls"][i].tolist()
        assert no == list(isn)
        assert [v for v, z in zip(vo, no) if not z] == [v for v, z in zip(vals, isn) if not z]
    # page assembly: same line pointers, pd_lower, pd_upper
    assert R["heap_page_added"][0] == nlines
    rp = R["heap_page"]
    np.testing.assert_array_equal(rp[16:30], pg[16:30])                       # pd_lower, pd_upper, pd_special, pagesize_version
    np.testing.assert_array_equal(rp[44:lower], pg[44:lower])                 # ItemIdData array
    upper = int(pg[20:24].copy().view(np.uint32)[0])
    np.testing.assert_array_equal(rp[upper:], pg[upper:])                     # tuple area
    # and the next tuple really does not fit (heap_insert's fill rule)
    lp = int(pages[1][44:48].copy().view(np.uint32)[0])
    assert ((lp >> 17) + 7) // 8 * 8 > upper - lower - 4


def test_fnpages_against_reference_objects(R):
    """Forward-node pages (the redistribute wire format): the oracle's sender writes the bytes that heaptuple.o's
    heap_form_minimal_tuple_ptr + fnbufpage.o's FnPageInit write under FragmentSendAttrs' control flow, the reference's
    receiver (iterator macros of fnbufpage.h + heap_deform_tuple) read those bytes back into the inputs, and the
    oracle's receiver does too."""
    cases = fnpage_inputs()
    assert len(cases) == len(R["fnpage_pages"])
    for (types, n, vals, isn), k, pages, inputs, ref_ok in zip(cases, R["fnpage_pages"].tolist(), R["fnpage_pages_digest"],
                                                               R["fnpage_inputs_digest"], R["fnpage_ref_unpack_ok"].tolist()):
        np.testing.assert_array_equal(digest(vals, isn), inputs, err_msg="input stream changed: regenerate the vectors")
        assert k > 0
        frac = isn.any()
        cols = [vals[:, i].astype(O.NP_DTYPES[t]) if t != O.GX_FLOAT8 else vals[:, i].copy().view(np.float64) for i, t in enumerate(types)]
        nulls = [isn[:, i].copy() for i in range(len(types))] if frac else None
        mine = O.fnpage_pack(types, cols, nulls, O.OrcFnPageId(*FNPAGE_ID[:6], 0), True)
        assert len(mine) == k
        np.testing.assert_array_equal(digest(mine), pages)                    # the reference's bytes exactly
        assert ref_ok                                                         # the reference's receiver on these pages
        c2, n2 = O.fnpage_unpack(mine, types)
        for i in range(len(types)):
            np.testing.assert_array_equal(n2[i], isn[:, i])
            keep = isn[:, i] == 0
            np.testing.assert_array_equal(np.asarray(c2[i])[keep].view(np.uint8), np.asarray(cols[i])[keep].view(np.uint8))
