"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol
include/b200grb.h declares, the host-side handle logic (pending tuples, element access, row iterator,
dup/resize) behaves like the reference expects, and bulk operations FAIL LOUDLY without a GPU
(there is no CPU fallback).  No kernel is launched here."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import falkordb_b200 as fb
from falkordb_b200._lib import lib, obj, LIB_PATH
from falkordb_b200.grb import Matrix

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu():
    import torch
    return torch.cuda.is_available()


def header_symbols():
    src = open(os.path.join(ROOT, "include", "b200grb.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    funcs = set(re.findall(r"\b((?:GrB|GxB|LAGraph|LAGr|B200)_\w+)\s*\(", src))
    data = set()
    for m in re.finditer(r"extern\s+(?:const\s+)?\w+\s+([^;]+);", src):
        for name in m.group(1).split(","):
            data.add(name.strip().lstrip("*"))
    return funcs, data


def test_library_exports_every_declared_symbol():
    L = lib()
    funcs, data = header_symbols()
    assert len(funcs) > 60 and "GrB_mxm" in funcs and "GrB_DESC_RSC" in data and len(data) >= 31 + 9
    missing = [s for s in sorted(funcs | data) if not hasattr(L, s)]
    assert not missing, f"libb200grb.so does not export: {missing}"


def test_descriptor_table_is_distinct():
    _, data = header_symbols()
    descs = [d for d in data if d.startswith("GrB_DESC_")]
    assert len(descs) == 31
    assert len({obj(d).value for d in descs}) == 31


def test_element_ops_and_pending_semantics_host_only():
    fb.init()
    m = Matrix(8, 8, "u64")
    assert m.nvals() == 0 and m.get(1, 2) is None
    m.set(1, 2, 10)
    m.set(3, 4, 20)
    m.set(1, 2, 11)            # overwrite while pending: last write wins
    assert m.pending()
    assert m.get(1, 2) == 11 and m.get(3, 4) == 20 and m.nvals() == 2
    assert not m.pending()
    m.remove(3, 4)
    m.remove(7, 7)             # removing an absent entry is a no-op
    m.set(0, 0, 0)             # edge id 0 is a real value (tensor.rs:1427-1476)
    assert m.nvals() == 2 and m.get(0, 0) == 0 and m.contains(0, 0) and not m.contains(3, 4)
    assert list(m.iter()) == [(0, 0, 0), (1, 2, 11)]
    with pytest.raises(fb.GrbError):
        m.set(8, 0, 1)         # GrB_INVALID_INDEX


def test_row_iterator_ranges_and_seek():
    m = Matrix(100, 100, bool)
    want = sorted({(i, (i * 7) % 100) for i in range(0, 100, 3)} | {(i, (i * 11 + 3) % 100) for i in range(0, 100, 3)})
    for i, j in want:
        m.set(i, j)
    m.wait()
    assert list(m.iter()) == want
    assert list(m.iter(10, 20)) == [t for t in want if 10 <= t[0] <= 20]
    assert list(m.iter(1, 2)) == []          # rows 1..2 are empty
    assert list(m.iter(99, 99)) == [t for t in want if t[0] == 99]
    assert list(m.iter(98, 2 ** 64 - 1)) == [t for t in want if t[0] >= 98]


def test_bool_is_pattern_only_and_iso():
    m = Matrix(4, 4, bool)
    m.set(1, 1)
    assert m.is_iso() and m.get(1, 1) is True
    with pytest.raises(fb.GrbError):
        m.set(0, 0, False)      # stored false is never used on the path (versioned_matrix.rs:413-416)
    u = Matrix(4, 4, "u64")
    assert not u.is_iso()


def test_dup_copies_pending_and_resize_host():
    m = Matrix(64, 48, "u64")
    for i in range(64):
        m.set(i, (i * 7) % 48, i)
    d = m.dup()                  # pending work is copied, not finished (matrix.rs:691-698)
    assert d.nvals() == 64 and m.nvals() == 64
    g = m.grown(256, 192)
    assert (g.nrows(), g.ncols(), g.nvals()) == (256, 192, 64)
    assert set(g.iter()) == set(m.iter())
    assert (m.nrows(), m.ncols()) == (64, 48)
    g.resize(10, 10)             # shrink drops out-of-range entries
    assert set(g.iter()) == {t for t in m.iter() if t[0] < 10 and t[1] < 10}
    with pytest.raises(AssertionError, match="grown must not shrink"):
        m.grown(32, 48)


def test_huge_dimension_matrix_is_host_resident():
    """Tensor's `me` matrix is 2^60 x 2^60 hypersparse (tensor.rs:254): element ops + build + iterate on host."""
    n = 1 << 60
    me = Matrix(n, n, bool).into_hyper()
    keys = [((5 << 32) | 9, 17), ((5 << 32) | 9, 3), ((1 << 59), (1 << 59) + 1), ((5 << 32) | 9, 17)]
    me.build([k[0] for k in keys], [k[1] for k in keys])
    assert me.nvals() == 3                                  # duplicates collapse (matrix.rs:1686-1695)
    assert list(me.iter()) == sorted(set(keys))
    assert me.sparsity_status() == "hypersparse" and me.hyper_vector_count() == 2
    me.remove((5 << 32) | 9, 3)
    assert list(me.iter((5 << 32) | 9, (5 << 32) | 9)) == [((5 << 32) | 9, 17)]
    a = Matrix(n, n, bool)
    with pytest.raises(fb.GrbError) as e:
        a.lmxm(me)                                          # bulk algebra needs device-capable dims
    assert e.value.info in (-8, -7002)


def test_unsupported_semantics_fail_loudly():
    a, b, c = Matrix(4, 4), Matrix(4, 4), Matrix(4, 5)
    L = lib()
    assert L.GrB_mxm(c.h, None, None, obj("GxB_ANY_PAIR_BOOL"), a.h, b.h, None) in (-6, -7002)
    # a semiring off the path
    assert L.GrB_mxm(a.h, None, None, obj("GxB_ANY_BOOL"), a.h, b.h, None) == -8


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a box without a GPU")
def test_bulk_ops_fail_loudly_without_gpu():
    a, b = Matrix(4, 4), Matrix(4, 4)
    a.set(0, 1)
    b.set(1, 2)
    with pytest.raises(fb.GrbError) as e:
        a.lmxm(b)
    assert e.value.info == -7002 and "no CPU fallback" in str(e.value)
    with pytest.raises(fb.GrbError):
        fb.rmat(4)
    with pytest.raises(fb.GrbError):
        a.build([0], [0])


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "falkordb_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle", txt, re.M), f
                assert not re.search(r"#include\s*[\"<][^\n]*oracle", txt), f
                assert "liborc" not in txt and "orc_" not in re.sub(r"//[^\n]*", "", txt), f


def test_host_resident_set_ops_for_multi_edge_store():
    """Tensor.me (2^60 x 2^60) folds its deltas with eWiseAdd(RC) / masked copy / eWiseMult like any VersionedMatrix
    (versioned_matrix.rs:909-926, 799-816); those run on the hypersparse host form, no device involved."""
    n = 1 << 60
    K = (7 << 32) | 9
    m, dp, dm = Matrix(n, n, bool), Matrix(n, n, bool), Matrix(n, n, bool)
    m.build([K, K, K + 1, 5], [1, 2, 3, 4])
    dp.build([K, 99], [7, 1])
    dm.build([K], [2])
    new_m = Matrix(n, n, bool)
    new_m.element_wise_add(dm, m, dp, fb.Descriptor.RC)            # new_m<!dm,replace> = m u dp
    assert list(new_m.iter()) == [(5, 4), (99, 1), (K, 1), (K, 7), (K + 1, 3)]
    sel = Matrix(n, n, bool)
    sel.select(dm, m)                                             # sel<!dm,replace> = m
    assert list(sel.iter()) == [(5, 4), (K, 1), (K + 1, 3)]
    mask = Matrix(n, n, bool)
    mask.build([K, K, 42], [1, 2, 0])
    tomb = Matrix(n, n, bool)
    tomb.element_wise_multiply(mask, mask, m, None)               # tombstone_masked: dm<mask> = mask n m
    assert list(tomb.iter()) == [(K, 1), (K, 2)]
    assert m.intersection_nvals(mask) == 2
    ex = Matrix(n, n, bool)
    ex.set_pattern(None, m, None)
    ex.remove_all(dm)
    ex.set_pattern(None, dp, None)                                # extract(): (m \ dm) u dp
    assert ex.nvals() == 5 and ex.contains(K, 7) and not ex.contains(K, 2)
    t = m.transpose()
    assert list(t.iter()) == sorted((c, r) for r, c in m.iter())


def test_header_is_plain_c_and_container_layout_matches_the_reference(tmp_path):
    """include/b200grb.h must be consumable from C (the reference binds it with bindgen); the GxB_Container struct the
    reference memcpy's into its RDB stream has the size / offsets asserted in mod.rs:14191-14236"""
    import subprocess
    hdr = os.path.join(ROOT, "include", "b200grb.h")
    src = tmp_path / "layout.c"
    src.write_text('#include "%s"\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(void){ printf("%%zu %%zu %%zu %%zu %%zu %%zu\\n", sizeof(struct GxB_Container_struct),'
                   ' offsetof(struct GxB_Container_struct, format), offsetof(struct GxB_Container_struct, p),'
                   ' offsetof(struct GxB_Container_struct, Y), offsetof(struct GxB_Container_struct, iso),'
                   ' offsetof(struct GxB_Container_struct, void_future)); return 0; }\n' % hdr)
    exe = tmp_path / "layout"
    subprocess.run(["/usr/bin/gcc", "-std=c11", "-Wall", "-Werror", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert [int(x) for x in out] == [608, 128, 192, 320, 448, 480]


@pytest.mark.parametrize("seed,valued", [(1, True), (2, False), (3, True)])
def test_randomised_host_model_check_with_serialization_in_the_loop(seed, valued):
    """3,000 random host-only operations (set / remove / get / contains / nvals / wait / dup / resize / clear / ranged
    iteration / RDB encode-decode round trip) against a dict model -- the same style as the reference's LCG model check
    of VersionedMatrix (versioned_matrix.rs:1399-1472), one layer down, and runnable without a GPU"""
    import random
    from falkordb_b200 import serial
    rnd = random.Random(seed)
    nr, nc = 40, 70
    m = Matrix(nr, nc, "u64" if valued else bool)
    model = {}

    def check_equal(mm, mod, r, c):
        assert (mm.nrows(), mm.ncols()) == (r, c)
        want = sorted((i, j, v) if valued else (i, j) for (i, j), v in mod.items())
        assert list(mm.iter()) == want
        assert mm.nvals() == len(mod)

    for step in range(3000):
        op = rnd.random()
        i, j = rnd.randrange(nr), rnd.randrange(nc)
        if op < 0.40:
            v = rnd.randrange(0, 1 << 40) if valued else True
            m.set(i, j, v) if valued else m.set(i, j)
            model[(i, j)] = v
        elif op < 0.60:
            m.remove(i, j)
            model.pop((i, j), None)
        elif op < 0.75:
            got = m.get(i, j)
            assert got == model.get((i, j)), (step, i, j)
            assert m.contains(i, j) == ((i, j) in model)
        elif op < 0.80:
            assert m.nvals() == len(model)
        elif op < 0.84:
            m.wait()
            assert not m.pending()
        elif op < 0.88:
            lo = rnd.randrange(nr)
            hi = rnd.randrange(lo, nr)
            want = sorted((a, b, v) if valued else (a, b) for (a, b), v in model.items() if lo <= a <= hi)
            assert list(m.iter(lo, hi)) == want
        elif op < 0.91:
            d = m.dup()
            check_equal(d, model, nr, nc)
        elif op < 0.94:
            h2 = serial.decode_matrix(serial.encode_matrix(m.h))        # save / restore in the middle of the history
            check_equal(Matrix(0, 0, "u64" if valued else bool, _handle=h2), model, nr, nc)
            check_equal(m, model, nr, nc)
        elif op < 0.97:
            nr2, nc2 = rnd.randrange(max(1, nr - 8), nr + 9), rnd.randrange(max(1, nc - 8), nc + 9)
            m.resize(nr2, nc2)
            model = {(a, b): v for (a, b), v in model.items() if a < nr2 and b < nc2}
            nr, nc = nr2, nc2
        elif op < 0.975:
            m.clear()
            model = {}
        else:
            check_equal(m, model, nr, nc)
    check_equal(m, model, nr, nc)


def test_concurrent_callers_on_separate_and_shared_handles():
    """the reference calls the library from a pool of threads: writers on their own output handles, readers sharing input
    handles of one snapshot (SURVEY 8b threading).  ctypes drops the GIL inside each call, so these really overlap."""
    import threading
    shared = Matrix(200, 200, "u64")
    for i in range(200):
        shared.set(i, (i * 13) % 200, i + 1)
    shared.wait()
    errors = []

    def worker(t):
        try:
            import random
            rnd = random.Random(t)
            m = Matrix(64, 64, "u64")
            model = {}
            for _ in range(1500):
                i, j = rnd.randrange(64), rnd.randrange(64)
                r = rnd.random()
                if r < 0.5:
                    m.set(i, j, t * 1000 + i)
                    model[(i, j)] = t * 1000 + i
                elif r < 0.7:
                    m.remove(i, j)
                    model.pop((i, j), None)
                elif r < 0.9:
                    k = rnd.randrange(200)
                    assert shared.get(k, (k * 13) % 200) == k + 1          # concurrent readers of one handle
                else:
                    assert m.nvals() == len(model)
            assert sorted(model.items()) == [((a, b), v) for a, b, v in m.iter()]
            d = shared.dup()
            assert d.nvals() == 200
        except Exception as ex:      # noqa: BLE001 -- collected and re-raised in the main thread
            errors.append(repr(ex))

    ts = [threading.Thread(target=worker, args=(t,)) for t in range(6)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors


def test_plain_c_caller_links_and_runs_the_host_only_calls(tmp_path):
    """examples/c_abi_demo.c: a C11 program against include/b200grb.h + libb200grb.so (element ops, pending work, row
    iterator, GxB_Container save / restore) -- the calls bindgen's extern block resolves to in the reference"""
    import subprocess
    exe = tmp_path / "demo"
    libdir = os.path.join(ROOT, "falkordb_b200")
    subprocess.run(["/usr/bin/gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "c_abi_demo.c"), "-L", libdir, "-lb200grb", f"-Wl,-rpath,{libdir}", "-o", str(exe)],
                   check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    assert out == ["nvals 2", "rides: (0,3) (2,5)", "container 6x6 nvals 2 format 2 iso 1", "restored: (0,3) (2,5)"]


# ------------------------------------------------------------------------------------------ link closure
def test_every_symbol_the_reference_wrappers_link_resolves():
    """The reference's wrapper layer (matrix.rs, vector.rs, tensor.rs, versioned_matrix.rs, the traversal operators' direct
    calls, algo.BFS) must link against this library unchanged: every extern "C" function / static those files name
    (tests/golden/reference_ffi_symbols.json, extracted by tests/golden/make_ffi_symbols.py) is a dynamic symbol here."""
    import json
    import subprocess
    doc = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_ffi_symbols.json")))
    assert len(doc["functions"]) >= 70 and len(doc["statics"]) >= 35
    for must in ("GrB_mxm", "GrB_Vector_clear", "GrB_Vector_wait", "GrB_Vector_setElement_UINT64", "GrB_Vector_resize",
                 "GrB_Vector_removeElement", "GxB_Vector_Iterator_attach", "GxB_Vector_Iterator_seek",
                 "GxB_Vector_Iterator_getIndex", "GxB_Vector_Iterator_next", "LAGr_BreadthFirstSearch_Extended"):
        assert must in doc["functions"], must
    nm = subprocess.check_output(["nm", "-D", "--defined-only", LIB_PATH], text=True)
    exported = {ln.split()[-1] for ln in nm.splitlines() if ln.strip()}
    missing = [f"{k} ({v['first_use']})" for k, v in {**doc["functions"], **doc["statics"]}.items() if k not in exported]
    assert not missing, f"unresolved reference symbols: {missing}"


def _vec_items(L, v, valued):
    it = C.c_void_p()
    fb.check(L.GxB_Iterator_new(C.byref(it)))
    fb.check(L.GxB_Vector_Iterator_attach(it, v, None))
    out = []
    info = L.GxB_Vector_Iterator_seek(it, 0)
    while info != 7089:                                   # GxB_EXHAUSTED: the loop of vector.rs:553-594
        i = L.GxB_Vector_Iterator_getIndex(it)
        out.append((i, L.GxB_Iterator_get_UINT64(it)) if valued else i)
        info = L.GxB_Vector_Iterator_next(it)
    L.GxB_Iterator_free(C.byref(it))
    return out


def test_vector_wrapper_calls_like_vector_rs():
    """Vector<bool> / Vector<u64> as vector.rs drives them: new, set (BOOL / UINT64), wait, iterate in ascending index
    order, remove, resize (shrinking drops entries), clear (vector.rs:98-134, 422-520, 553-594)."""
    L = lib()
    v = C.c_void_p()
    fb.check(L.GrB_Vector_new(C.byref(v), obj("GrB_BOOL"), 100))
    for i in (7, 3, 99, 3, 50):
        fb.check(L.GrB_Vector_setElement_BOOL(v, True, i))
    fb.check(L.GrB_Vector_wait(v, 1))
    assert _vec_items(L, v, False) == [3, 7, 50, 99]
    assert L.GrB_Vector_setElement_BOOL(v, True, 100) == -4            # GrB_INVALID_INDEX
    fb.check(L.GrB_Vector_removeElement(v, 7))
    fb.check(L.GrB_Vector_removeElement(v, 8))                           # absent: not an error
    assert _vec_items(L, v, False) == [3, 50, 99]
    fb.check(L.GrB_Vector_resize(v, 60))
    n = C.c_uint64()
    fb.check(L.GrB_Vector_size(C.byref(n), v))
    assert n.value == 60 and _vec_items(L, v, False) == [3, 50]
    fb.check(L.GrB_Vector_resize(v, 1 << 40))
    fb.check(L.GrB_Vector_setElement_BOOL(v, True, (1 << 40) - 1))
    assert _vec_items(L, v, False) == [3, 50, (1 << 40) - 1]
    fb.check(L.GrB_Vector_clear(v))
    assert _vec_items(L, v, False) == []
    fb.check(L.GrB_Vector_nvals(C.byref(n), v))
    assert n.value == 0
    fb.check(L.GrB_Vector_free(C.byref(v)))
    u = C.c_void_p()
    fb.check(L.GrB_Vector_new(C.byref(u), obj("GrB_UINT64"), 10))
    for i, x in ((4, 40), (1, 2 ** 63 + 5), (4, 41), (9, 0)):
        fb.check(L.GrB_Vector_setElement_UINT64(u, x, i))
    assert _vec_items(L, u, True) == [(1, 2 ** 63 + 5), (4, 41), (9, 0)]
    it = C.c_void_p()
    fb.check(L.GxB_Iterator_new(C.byref(it)))
    fb.check(L.GxB_Vector_Iterator_attach(it, u, None))
    assert L.GxB_Vector_Iterator_getpmax(it) == 3
    assert L.GxB_Vector_Iterator_seek(it, 2) == 0 and L.GxB_Vector_Iterator_getIndex(it) == 9 and L.GxB_Vector_Iterator_getp(it) == 2
    assert L.GxB_Vector_Iterator_next(it) == 7089 and L.GxB_Vector_Iterator_seek(it, 3) == 7089
    L.GxB_Iterator_free(C.byref(it))
    fb.check(L.GrB_Vector_free(C.byref(u)))


def test_gxb_init_allocators_see_the_host_footprint(tmp_path):
    """GxB_init's allocators (Redis' in the reference, matrix.rs:123-131) must serve the library's host memory: handles,
    tuple stores, pending lists, vector payloads, container structs, blobs.  Run in a fresh process because the hooks have
    to be installed before anything is allocated."""
    import subprocess
    import sys
    code = r"""
import ctypes as C, sys
sys.path.insert(0, %r)
from falkordb_b200._lib import lib, obj, check
L = lib()
libc = C.CDLL(None)
libc.malloc.restype = C.c_void_p; libc.malloc.argtypes = [C.c_size_t]
libc.calloc.restype = C.c_void_p; libc.calloc.argtypes = [C.c_size_t, C.c_size_t]
libc.realloc.restype = C.c_void_p; libc.realloc.argtypes = [C.c_void_p, C.c_size_t]
libc.free.argtypes = [C.c_void_p]
live, calls = {}, {"malloc": 0, "calloc": 0, "free": 0}
MAL = C.CFUNCTYPE(C.c_void_p, C.c_size_t); CAL = C.CFUNCTYPE(C.c_void_p, C.c_size_t, C.c_size_t)
REA = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_size_t); FRE = C.CFUNCTYPE(None, C.c_void_p)
def m(n):
    p = libc.malloc(n); live[p] = n; calls["malloc"] += 1; return p
def c(a, b):
    p = libc.calloc(a, b); live[p] = a * b; calls["calloc"] += 1; return p
def r(p, n):
    live.pop(p, None); q = libc.realloc(p, n); live[q] = n; return q
def f(p):
    if p: assert p in live, "free of a block the hooks never handed out"; live.pop(p); calls["free"] += 1; libc.free(p)
cb = (MAL(m), CAL(c), REA(r), FRE(f))
L.GxB_init.argtypes = [C.c_int, MAL, CAL, REA, FRE]
check(L.GxB_init(1, *cb))
A = C.c_void_p(); check(L.GrB_Matrix_new(C.byref(A), obj("GrB_UINT64"), 1000, 1000))
for k in range(500): check(L.GrB_Matrix_setElement_UINT64(A, k, k, (k * 7) %% 1000))
check(L.GrB_Matrix_wait(A, 1))
held = sum(live.values())
assert calls["malloc"] >= 4 and held >= 500 * 8 * 2, (calls, held)
assert L.B200_get_stat(b"host_bytes") <= held and L.B200_get_stat(b"host_bytes") >= 500 * 8 * 2
v = C.c_void_p(); check(L.GrB_Vector_new(C.byref(v), obj("GrB_BOOL"), 64))
for k in range(0, 64, 3): check(L.GrB_Vector_setElement_BOOL(v, True, k))
blob = C.c_void_p(); size = C.c_uint64()
L.GxB_Vector_serialize.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p]
check(L.GxB_Vector_serialize(C.byref(blob), C.byref(size), v, None))
assert blob.value in live                      # the caller frees the blob with ITS allocator (vector.rs:171-172)
f(blob.value)
cont = C.c_void_p(); L.GxB_Container_new.argtypes = [C.POINTER(C.c_void_p)]; L.GxB_Container_free.argtypes = [C.POINTER(C.c_void_p)]
check(L.GxB_Container_new(C.byref(cont))); assert calls["calloc"] >= 1
check(L.GxB_Container_free(C.byref(cont)))
check(L.GrB_Vector_free(C.byref(v))); check(L.GrB_Matrix_free(C.byref(A)))
assert not live, "leaked through the hooks: %%r" %% live
assert L.B200_get_stat(b"host_bytes") == 0
print("hooks ok", calls)
""" % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "hooks ok" in out.stdout, out.stdout + out.stderr
