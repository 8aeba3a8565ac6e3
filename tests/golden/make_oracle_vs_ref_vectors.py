"""Generates tests/golden/oracle_vs_ref.npz: what the REFERENCE'S OWN OBJECT CODE (oracle/_ref/libotbref.so, built by
oracle/ref/Makefile from the reference's leaf sources) returns on the inputs of tests/test_oracle_vs_ref.py.
Run where the reference source tree exists:

    python -c "import __graft_entry__ as e; e.build()"      # builds oracle/_ref
    python tests/golden/make_oracle_vs_ref_vectors.py

The inputs are drawn from the same seeded generators as the test, and a digest of them is stored next to the
reference's answers, so the test can tell a changed input stream from a changed oracle.  Outputs too large to keep
(bloom filter words, forward-node pages) are stored as SHA-256 digests of their bytes: equal digests mean the oracle
produced the reference's bytes exactly."""
import ctypes as C
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle as O                                         # noqa: E402
import test_oracle_vs_ref as T                             # noqa: E402  (the test's own input generators)


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def load_ref():
    L = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libotbref.so"))
    u32, i32, i64, dbl = C.c_uint32, C.c_int32, C.c_int64, C.c_double
    for n, res, args in [("ref_hash_any", u32, [C.c_char_p, C.c_int]), ("ref_hash_uint32", u32, [u32]),
                         ("ref_hashint4", u32, [i32]), ("ref_hashint8", u32, [i64]), ("ref_hashchar", u32, [C.c_int8]),
                         ("ref_hashfloat8", u32, [dbl]), ("ref_hash_any_new", u32, [C.c_char_p, C.c_int]),
                         ("ref_hashint4new", u32, [i32]), ("ref_hashint8new", u32, [i64]), ("ref_hashcharnew", u32, [C.c_int8]),
                         ("ref_hashfloat8new", u32, [dbl]), ("ref_murmurhash32", u32, [u32]), ("ref_hash_combine", u32, [u32, u32]),
                         ("ref_evaluate_hashkey1", u32, [C.c_int, i64, C.c_int]), ("ref_evaluate_hashkey2", u32, [i64, i32]),
                         ("ref_bloom_init", C.c_void_p, [dbl, dbl]), ("ref_bloom_insert", None, [C.c_void_p, u32]),
                         ("ref_bloom_find", C.c_int, [C.c_void_p, u32]), ("ref_bloom_log_num_buckets", C.c_int, [C.c_void_p]),
                         ("ref_bloom_words", C.c_void_p, [C.c_void_p]),
                         ("ref_float8pl", dbl, [dbl, dbl]), ("ref_float8mul", dbl, [dbl, dbl]), ("ref_float8mi", dbl, [dbl, dbl]),
                         ("ref_float8_accum", None, [C.c_void_p, dbl]), ("ref_float8_combine", None, [C.c_void_p, C.c_void_p]),
                         ("ref_float8_avg", C.c_int, [C.c_void_p, C.c_void_p]), ("ref_int8inc", i64, [i64]),
                         ("ref_heap_form_tuple", C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
                         ("ref_heap_deform_tuple", None, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
                         ("ref_page_build", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
                         ("ref_page_offsets", None, [C.c_void_p]),
                         ("ref_fnpage_pack", C.c_int64, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                                         C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64]),
                         ("ref_fnpage_unpack", C.c_int64, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64])]:
        f = getattr(L, n); f.restype = res; f.argtypes = args
    return L


def layout(R, out):
    a = (C.c_int * 10)()
    R.ref_page_offsets(a)
    out["layout_page_offsets"] = np.array(list(a), np.int64)
    out["layout_sizes"] = np.array([R.ref_sizeof_heap_header(), R.ref_offsetof_hoff(), R.ref_offsetof_infomask(),
                                    R.ref_sizeof_minimal_header(), R.ref_minimal_tuple_offset(),
                                    R.ref_sizeof_fnpage_header(), R.ref_invalid_shardid()], np.int64)


def hashes(R, out):
    h = T.hash_inputs()
    out["hash_inputs_digest"] = T.hash_inputs_digest(h)
    i4, i8 = h["i4"].tolist(), h["i8"].tolist()
    u = np.uint32
    out["hash_i4"] = np.array([[R.ref_hashint4(v), R.ref_hashint4new(v), R.ref_hash_uint32(v & 0xFFFFFFFF),
                                R.ref_murmurhash32(v & 0xFFFFFFFF), R.ref_evaluate_hashkey1(0, v, 0)] for v in i4], u)
    out["hash_i8"] = np.array([[R.ref_hashint8(v), R.ref_hashint8new(v), R.ref_evaluate_hashkey1(1, v, 0)] for v in i8], u)
    out["hash_char"] = np.array([[R.ref_hashchar(v), R.ref_hashcharnew(v)] for v in range(-128, 128)], u)
    out["hash_f8"] = np.array([[R.ref_hashfloat8(v), R.ref_hashfloat8new(v)] for v in h["f8"].tolist()], u)
    out["hash_any"] = np.array([[R.ref_hash_any(b, len(b)), R.ref_hash_any_new(b, len(b))] for b in h["blobs"]], u)
    out["hash_combine"] = np.array([R.ref_hash_combine(a, b) for a, b in h["pairs"].tolist()], u)
    out["hash_key2"] = np.array([R.ref_evaluate_hashkey2(a, b) for a, b in zip(i8[:200], i4[:200])], u)
    out["hash_key1_null"] = np.array([R.ref_evaluate_hashkey1(1, 12345, 1)], u)


def bloom(R, out):
    rows = []
    for nrows in T.BLOOM_ROWS:
        rb = R.ref_bloom_init(float(nrows), 0.05)
        if rb is None:
            rows.append((nrows, -1, 0, np.zeros(32, np.uint8), np.zeros(0, np.uint8)))
            continue
        ob = O.lib().orc_bloom_create(nrows)                # only for the word count the test compares over
        nw = C.c_int64()
        O.lib().orc_bloom_words(ob, C.byref(nw))
        O.lib().orc_bloom_free(ob)
        for k in T.bloom_keys(nrows):
            R.ref_bloom_insert(rb, k)
        rw = np.ctypeslib.as_array(C.cast(R.ref_bloom_words(rb), C.POINTER(C.c_uint32)), (nw.value,)).copy()
        found = np.array([R.ref_bloom_find(rb, p) for p in T.bloom_probes()], np.uint8)
        rows.append((nrows, R.ref_bloom_log_num_buckets(rb), nw.value, digest(rw), found))
    out["bloom_rows"] = np.array([r[0] for r in rows], np.int64)
    out["bloom_log_num_buckets"] = np.array([r[1] for r in rows], np.int64)
    out["bloom_nwords"] = np.array([r[2] for r in rows], np.int64)
    out["bloom_words_digest"] = np.stack([r[3] for r in rows])
    out["bloom_find"] = np.stack([r[4] for r in rows if len(r[4])])
    out["bloom_1e9_gives_up"] = np.array([R.ref_bloom_init(1e9, 0.05) is None], np.uint8)


def float8(R, out):
    vals, plan = T.float8_inputs()
    out["float8_inputs_digest"] = digest(vals)
    state = (C.c_double * 3)(0.0, 0.0, 0.0)
    s = None
    for x in vals.tolist():
        R.ref_float8_accum(state, x)
        s = x if s is None else R.ref_float8pl(s, x)
    out["float8_accum_state"] = np.array(list(state))
    out["float8pl_sum"] = np.array([s])
    o = C.c_double()
    rc = R.ref_float8_avg(state, C.byref(o))
    out["float8_avg"] = np.array([rc, o.value])
    out["float8_avg_empty_rc"] = np.array([R.ref_float8_avg((C.c_double * 3)(0, 0, 0), C.byref(o))], np.int64)
    # float8_combine over the two halves' partial states, as the oracle computes them
    h = len(vals) // 2
    r1, _ = O.exec_agg(O.Rel([O.GX_FLOAT8], [vals[:h]]), plan, keep_raw=True)
    r2, _ = O.exec_agg(O.Rel([O.GX_FLOAT8], [vals[h:]]), plan, keep_raw=True)
    s1 = (C.c_double * 3)(*r1.states[0, 0]); s2 = (C.c_double * 3)(*r2.states[0, 0])
    out["float8_combine_inputs"] = np.array([list(s1), list(s2)])
    R.ref_float8_combine(s1, s2)
    out["float8_combine"] = np.array(list(s1))
    out["float8_mul_mi"] = np.array([R.ref_float8mul(1.1, 3.3), R.ref_float8mi(1.0, 0.07)])
    out["int8inc_41"] = np.array([R.ref_int8inc(41)], np.int64)


def heap(R, out):
    types, cols, nulls = T.heap_inputs()
    out["heap_inputs_digest"] = T.heap_inputs_digest(cols, nulls)
    attlen, attalign = T.attrs(types)
    rel = O.Rel(types, cols, nulls)
    pg = rel.pages().reshape(-1, 8192)[0]
    lower = int(pg[16:20].copy().view(np.uint32)[0]); nlines = (lower - 44) // 4
    buf = (C.c_uint8 * 1024)()
    tuples, lens, items = [], [], b""
    deform_vals = np.zeros((nlines, len(types)), np.int64); deform_nulls = np.zeros((nlines, len(types)), np.uint8)
    mine_lens = []
    for i in range(nlines):
        vals, isn = T.heap_row(types, cols, nulls, i)
        rl = R.ref_heap_form_tuple(len(types), attlen, attalign, vals, isn, buf, 1024)
        t = np.frombuffer(bytes(buf)[:rl], np.uint8).copy()
        tuples.append(t); lens.append(rl)
        # the deform and the page assembly are run on the ORACLE's tuple bytes, as the test compares them
        lp = int(pg[44 + 4 * i: 48 + 4 * i].copy().view(np.uint32)[0])
        mine = pg[lp & 0x7FFF: (lp & 0x7FFF) + (lp >> 17)].copy()
        vo, no = (C.c_int64 * len(types))(), (C.c_uint8 * len(types))()
        R.ref_heap_deform_tuple(len(types), attlen, attalign, mine.ctypes.data, len(mine), vo, no)
        deform_vals[i], deform_nulls[i] = list(vo), list(no)
        items += mine.tobytes(); mine_lens.append(len(mine))
    out["heap_tuples"] = np.concatenate(tuples)
    out["heap_tuple_lens"] = np.array(lens, np.int64)
    out["heap_deform_vals"] = deform_vals
    out["heap_deform_nulls"] = deform_nulls
    rpage = (C.c_uint8 * 8192)()
    added = R.ref_page_build(rpage, items, (C.c_int * len(mine_lens))(*mine_lens), len(mine_lens))
    out["heap_page_added"] = np.array([added], np.int64)
    out["heap_page"] = np.frombuffer(bytes(rpage), np.uint8).copy()


def fnpages(R, out):
    ks, page_digests, unpack_ok, in_digests = [], [], [], []
    for types, n, vals, isn in T.fnpage_inputs():
        attlen, attalign = T.attrs(types)
        cap = n // 20 + 4
        ref = np.zeros((cap, 8192), np.uint8)
        k = R.ref_fnpage_pack(len(types), attlen, attalign, vals.ctypes.data, isn.ctypes.data, n, *T.FNPAGE_ID, ref.ctypes.data, cap)
        vo = np.zeros((n, len(types)), np.int64); no = np.zeros((n, len(types)), np.uint8)
        got = R.ref_fnpage_unpack(ref.ctypes.data, k, len(types), attlen, attalign, vo.ctypes.data, no.ctypes.data, n)
        ks.append(k); page_digests.append(digest(ref[:k])); in_digests.append(digest(vals, isn))
        unpack_ok.append(got == n and np.array_equal(no, isn) and np.array_equal(vo[isn == 0], vals[isn == 0]))
    out["fnpage_pages"] = np.array(ks, np.int64)
    out["fnpage_pages_digest"] = np.stack(page_digests)
    out["fnpage_inputs_digest"] = np.stack(in_digests)
    out["fnpage_ref_unpack_ok"] = np.array(unpack_ok, np.uint8)


if __name__ == "__main__":
    R = load_ref()
    out = {}
    for f in (layout, hashes, bloom, float8, heap, fnpages):
        f(R, out)
    path = os.path.join(ROOT, "tests", "golden", "oracle_vs_ref.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")
