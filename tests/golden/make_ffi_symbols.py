#!/usr/bin/env python
"""Regenerates tests/golden/reference_ffi_symbols.json: every GraphBLAS / LAGraph C symbol the reference's wrapper layer
links against.  A symbol counts when (a) graph/src/graph/graphblas/mod.rs (bindgen) or lagraph*_bindings.rs declares it as an
`extern "C"` function or static and (b) one of the wrapper files below names it outside a comment.  Needs a checkout of the
reference: python tests/golden/make_ffi_symbols.py <reference checkout>.  The JSON is what tests/test_abi.py checks
`nm -D libb200grb.so` against."""
import json
import os
import re
import sys

REF = None                  # the reference checkout, from the command line
GB = "graph/src/graph/graphblas"
WRAPPERS = [f"{GB}/matrix.rs", f"{GB}/vector.rs", f"{GB}/tensor.rs", f"{GB}/versioned_matrix.rs"]
# the traversal operators and the BFS procedure reach the C API through the wrappers plus these direct call sites
CALLERS = ["graph/src/runtime/ops/cond_traverse.rs", "graph/src/runtime/ops/expand_into.rs", "src/module_init.rs"]
# algo_procedures.rs: the shared helpers (create_lagraph_graph .. build_compact_adj_symmetric_from_tensors) and the four procedures
# this backend serves -- algo.pageRank, algo.WCC, algo.BFS, algo.labelPropagation -- by line range of the frozen reference;
# betweenness (:884-1020) and everything from MSF on (:1274-) call LAGraph kernels that stay with LAGraph (SURVEY 8 f4)
ALGO_RANGES = [(360, 673), (689, 883), (1021, 1273)]
ALGO_ALWAYS = {"LAGraph_Init", "LAGraph_Finalize"}


def declared():
    fn, st = {}, {}
    for rel in (f"{GB}/mod.rs", f"{GB}/lagraph_bindings.rs", f"{GB}/lagraphx_bindings.rs"):
        path = os.path.join(REF, rel)
        if not os.path.exists(path):
            continue
        for ln, line in enumerate(open(path, encoding="utf-8", errors="replace"), 1):
            m = re.match(r"\s*pub fn ([A-Za-z_][A-Za-z0-9_]*)\s*\(", line)
            if m and re.match(r"(GrB|GxB|LAGr|LAGraph)_", m.group(1)):
                fn.setdefault(m.group(1), f"{rel}:{ln}")
            m = re.match(r"\s*pub static (?:mut )?([A-Za-z_][A-Za-z0-9_]*)\s*:", line)
            if m and re.match(r"(GrB|GxB|LAGr|LAGraph)_", m.group(1)):
                st.setdefault(m.group(1), f"{rel}:{ln}")
    return fn, st


def used(rel):
    out = {}
    for ln, line in enumerate(open(os.path.join(REF, rel), encoding="utf-8", errors="replace"), 1):
        code = line.split("//")[0]
        for m in re.finditer(r"\b((?:GrB|GxB|LAGr|LAGraph)_[A-Za-z0-9_]+)\b", code):
            out.setdefault(m.group(1), f"{rel}:{ln}")
    return out


def main():
    global REF
    if len(sys.argv) != 2:
        return "usage: python tests/golden/make_ffi_symbols.py <reference checkout>"
    REF = sys.argv[1]
    fn, st = declared()
    functions, statics = {}, {}
    for rel in WRAPPERS + CALLERS:
        if not os.path.exists(os.path.join(REF, rel)):
            continue
        for name, where in used(rel).items():
            if name in fn:
                functions.setdefault(name, {"declared": fn[name], "first_use": where})
            elif name in st:
                statics.setdefault(name, {"declared": st[name], "first_use": where})
    ap = "graph/src/runtime/functions/algo_procedures.rs"
    for ln, line in enumerate(open(os.path.join(REF, ap), encoding="utf-8", errors="replace"), 1):
        if not any(lo <= ln <= hi for lo, hi in ALGO_RANGES):
            continue
        for m in re.finditer(r"\b((?:GrB|GxB|LAGr|LAGraph)_[A-Za-z0-9_]+)\b", line.split("//")[0]):
            name, where = m.group(1), f"{ap}:{ln}"
            if name in fn:
                functions.setdefault(name, {"declared": fn[name], "first_use": where})
            elif name in st:
                statics.setdefault(name, {"declared": st[name], "first_use": where})
    for name in ALGO_ALWAYS:
        if name in fn:
            functions.setdefault(name, {"declared": fn[name], "first_use": ap})
    doc = {"generated_by": "tests/golden/make_ffi_symbols.py",
           "wrappers": WRAPPERS + CALLERS + [ap + " (helpers, pageRank, WCC, BFS, labelPropagation: lines %s)" % ALGO_RANGES],
           "functions": dict(sorted(functions.items())), "statics": dict(sorted(statics.items()))}
    dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_ffi_symbols.json")
    with open(dst, "w") as f:
        json.dump(doc, f, indent=1)
    print(f"{len(functions)} functions, {len(statics)} statics -> {dst}")


if __name__ == "__main__":
    sys.exit(main())
