"""The Rust binding ships as source (ffi/sweepga-cuda-sys) because this image has no cargo.  What can be checked without
compiling it is checked here: every #[repr(C)] struct of src/lib.rs has the header's field order, sizes and offsets (the C
layout rules applied to the Rust field types, compared with gcc's sizeof / offsetof of include/sweepga_b200.h), every
function the header declares is bound with the same number of arguments, and nothing is bound that the header lacks."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_RS = os.path.join(ROOT, "ffi", "sweepga-cuda-sys", "src", "lib.rs")
HEADER = os.path.join(ROOT, "include", "sweepga_b200.h")

RUST_TYPES = {"u8": (1, 1), "u16": (2, 2), "u32": (4, 4), "u64": (8, 8), "i64": (8, 8), "f64": (8, 8), "usize": (8, 8)}


def rust_structs():
    src = open(LIB_RS).read()
    out = {}
    for m in re.finditer(r"#\[repr\(C\)\](?:\s*#\[derive\([^)]*\)\])?\s*pub struct (\w+)\s*\{(.*?)\n\}", src, re.S):
        fields = []
        for f in re.finditer(r"pub (\w+):\s*([^,\n]+),", m.group(2)):
            fields.append((f.group(1), f.group(2).strip()))
        out[m.group(1)] = fields
    return out


def c_layout(fields):
    """C layout rules on the Rust field types -> ({field: offset}, sizeof)"""
    off, align_max, offsets = 0, 1, {}
    for name, ty in fields:
        if ty.startswith("*"):
            size, align = 8, 8
        else:
            a = re.match(r"\[(\w+);\s*(\d+)\]", ty)
            if a:
                es, ea = RUST_TYPES[a.group(1)]
                size, align = es * int(a.group(2)), ea
            else:
                size, align = RUST_TYPES[ty]
        off = (off + align - 1) // align * align
        offsets[name] = off
        off += size
        align_max = max(align_max, align)
    return offsets, (off + align_max - 1) // align_max * align_max


def test_rust_structs_match_header_layout():
    from test_host import _header_layout
    structs = {k: v for k, v in rust_structs().items() if v}  # opaque handles have no public fields
    assert set(structs) == {"swg_config", "swg_mappings", "swg_result", "swg_stats"}
    want = _header_layout({name: [f for f, _ in fields] for name, fields in structs.items()})
    for name, fields in structs.items():
        offsets, size = c_layout(fields)
        assert size == want[name], (name, size, want[name])
        for f, _ in fields:
            assert offsets[f] == want[f"{name}.{f}"], (name, f)


def _split_args(s):
    s = s.strip()
    return [] if s in ("", "void") else [a for a in s.split(",") if a.strip()]


def test_rust_functions_match_header_declarations():
    header = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    decl = {m.group(1): len(_split_args(m.group(2))) for m in re.finditer(r"\b(swg_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header, re.S)}
    src = open(LIB_RS).read()
    ext = src[src.index('extern "C" {'):]
    bound = {m.group(1): len(_split_args(m.group(2))) for m in re.finditer(r"pub fn (swg_\w+)\(([^)]*)\)", ext)}
    assert set(decl) == set(bound), (sorted(set(decl) - set(bound)), sorted(set(bound) - set(decl)))
    for name, n in decl.items():
        assert bound[name] == n, (name, n, bound[name])


def test_build_rs_compiles_the_same_sources_with_the_same_flags():
    import __graft_entry__ as ge
    text = open(os.path.join(ROOT, "ffi", "sweepga-cuda-sys", "build.rs")).read()
    for src in ge.SOURCES:
        assert f'"{src}"' in text, src
    for flag in ("arch=compute_100a,code=sm_100a", "-fmad=false", "--extended-lambda", "-cudart"):
        assert flag in text, flag
    assert "sm_90" not in text and "compute_90" not in text  # one architecture, no fallback


def _hunks(patch):
    """-> [(file, old_start, old_len, new_start, new_len, [body lines])] of a unified diff"""
    out, path = [], None
    lines = patch.split("\n")
    for i, line in enumerate(lines):
        if line.startswith("+++ "):
            path = line[4:].split("/", 1)[1]
        m = re.match(r"@@ -(\d+)(?:,(\d+))? \+(\d+)(?:,(\d+))? @@", line)
        if m:
            old, old_n, new, new_n = (int(g) if g is not None else 1 for g in m.groups())
            body, j = [], i + 1
            while j < len(lines) and lines[j][:1] in (" ", "-", "+") and not lines[j].startswith(("--- ", "+++ ")):
                body.append(lines[j])
                j += 1
            out.append((path, old, old_n, new, new_n, body))
    return out


def test_patch_applies_to_the_cited_lines():
    """patches/apply_filters.patch replaces the body of PafFilter::apply_filters; its hunk header cites the reference lines it
    was written against (src/paf_filter.rs:379-382).  Every hunk's line counts agree with its header, its new start follows
    from the hunks before it in the same file, and the function head sits at the cited lines of the paf_filter.rs hunk.
    When SWEEPGA_SRC names a sweepga v0.1.1 checkout, every context and removed line of every hunk must also quote that
    checkout verbatim at the line its header cites (no offset, no fuzz)."""
    patch = open(os.path.join(ROOT, "patches", "apply_filters.patch")).read()
    assert "--- a/src/paf_filter.rs" in patch and "+++ b/src/paf_filter.rs" in patch
    assert "sweepga_cuda_sys" in patch and "swg_filter" in patch
    hunks = _hunks(patch)
    assert [h[0] for h in hunks] == ["Cargo.toml", "Cargo.toml", "src/lib.rs", "src/main.rs", "src/paf_filter.rs", "src/cuda_filter.rs"]
    delta = {}
    for path, old, old_n, new, new_n, body in hunks:
        assert sum(l[0] in " -" for l in body) == old_n, (path, old)
        assert sum(l[0] in " +" for l in body) == new_n, (path, old)
        assert new == (1 if old_n == 0 and old == 0 else old + delta.get(path, 0)), (path, old, new)
        delta[path] = delta.get(path, 0) + new_n - old_n
    # the pre-image lines of the paf_filter.rs hunk, at the reference's line numbers: the function head is lines 379-382
    _, old, _, _, _, body = hunks[4]
    pre = {old + k: l[1:] for k, l in enumerate(l for l in body if l[0] in " -")}
    assert pre[379].strip() == "pub fn apply_filters(" and pre[382].strip() == ") -> Result<HashMap<usize, RecordMeta>> {"
    ref = os.environ.get("SWEEPGA_SRC")
    if ref:  # the reference sources are not part of this repository: compared where a checkout of them is at hand
        assert re.search(r'^version\s*=\s*"0\.1\.1"', open(os.path.join(ref, "Cargo.toml")).read(), re.M), "not sweepga v0.1.1"
        for path, old, old_n, _, _, body in hunks:
            if old_n:
                src = open(os.path.join(ref, path)).read().split("\n")
                want = [l[1:] for l in body if l[0] in " -"]
                assert src[old - 1:old - 1 + old_n] == want, (path, old)
