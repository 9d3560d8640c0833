"""The reference-side artefacts under rust/ are not compiled by the build (it needs no cargo), so they are checked
structurally: the generated `-sys` bindings against the ctypes mirror and the compiled library."""
import ctypes as C
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_nrrt_sys as G  # noqa: E402
from nr_ray_tracer_b200 import api  # noqa: E402

LIB_RS = os.path.join(ROOT, "rust", "nrrt-sys", "src", "lib.rs")
HEADER = os.path.join(ROOT, "include", "nrrt.h")


def test_committed_bindings_are_what_the_generator_produces():
    assert open(LIB_RS).read() == G.generate(), "rust/nrrt-sys/src/lib.rs is stale: python tools/gen_nrrt_sys.py"


def _rust_structs(text):
    out = {}
    for m in re.finditer(r"#\[repr\(C\)\]\s*(?:#\[derive\([^)]*\)\]\s*)*pub struct (\w+) \{(.*?)\n\}", text, re.S):
        fields = re.findall(r"pub (\w+): ([^,\n]+),", m.group(2))
        out[m.group(1)] = fields
    return out


def _rust_size_align(ty, structs):
    """(size, alignment) of a Rust type under #[repr(C)] on x86-64."""
    ty = ty.strip()
    prim = {"u8": 1, "u32": 4, "u64": 8, "f32": 4, "f64": 8, "c_int": 4, "usize": 8}
    if ty in prim:
        return prim[ty], prim[ty]
    if ty.startswith("*const") or ty.startswith("*mut"):
        return 8, 8
    m = re.fullmatch(r"\[(.+); (\d+)\]", ty)
    if m:
        s, a = _rust_size_align(m.group(1), structs)
        return s * int(m.group(2)), a
    off, align = 0, 1
    for _n, t in structs[ty]:
        s, a = _rust_size_align(t, structs)
        off = (off + a - 1) // a * a + s
        align = max(align, a)
    return (off + align - 1) // align * align, align


def test_every_repr_c_struct_matches_the_ctypes_mirror_and_the_library():
    structs = _rust_structs(open(LIB_RS).read())
    assert set(structs) == {n for n, _ in G.STRUCTS}
    for name, cls in G.STRUCTS:
        want = [(f, G.rust_type(t, f)) for f, t in cls._fields_]
        assert structs[name] == want, name
        assert _rust_size_align(name, structs)[0] == C.sizeof(cls), name          # #[repr(C)] layout == C layout
    L = api.lib()
    for which, name in enumerate(G.SIZEOF_ORDER):                                   # ... == what the .so was compiled with
        assert L.nrrt_abi_sizeof(which) == _rust_size_align(name, structs)[0], name
    assert L.nrrt_abi_sizeof(len(G.SIZEOF_ORDER)) == 0
    stats = dict(structs["nrrt_render_stats"])                                      # round-1 defect: two fields were missing
    assert "inst_entries" in stats and "inst_misses" in stats and "mode" in stats


def test_extern_functions_are_the_header_s_and_are_exported():
    rust = set(re.findall(r"pub fn (nrrt_\w+)\(", open(LIB_RS).read()))
    header = set(re.findall(r"\b(nrrt_\w+)\s*\(", re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)))
    header = {h for h in header if not h.endswith("_fn")}
    assert rust == header, (sorted(rust - header), sorted(header - rust))
    L = api.lib()
    for fn in sorted(rust):
        assert hasattr(L, fn), f"{fn} is declared but not exported by libnrrt_b200.so"
    consts = dict(re.findall(r"pub const (NRRT_\w+): \w+ = (-?\d+);", open(LIB_RS).read()))
    hdr = open(HEADER).read()
    for name, val in consts.items():                                                # every constant has the header's value
        m = re.search(rf"\b{name}\s*=\s*(-?\d+)", hdr) or re.search(rf"#define {name} (\d+)", hdr)
        if m is None and name in ("NRRT_OBJ_ROTATE_Y", "NRRT_OBJ_ROTATE_Z", "NRRT_BUILD_SAH"):
            continue                                                               # implicit enum successors
        assert m is not None and int(m.group(1)) == int(val), name

