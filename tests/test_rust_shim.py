"""The reference-side binding (racer_tracer_b200/rust_shim): what can be checked without a Rust toolchain.

* reference.diff — the patch a maintainer applies to the reference crate — carries the two new source files kept
  here and every edit tools/make_rust_patch.py makes, and nothing else;
* with a checkout of the reference crate (RACER_TRACER_REFERENCE = its racer-tracer/ directory; the repository
  keeps nothing of the reference but the patch's context lines): the patch APPLIES to it (`patch --dry-run`), is
  exactly what tools/make_rust_patch.py generates from it, and every trait method the patch adds is implemented
  for every type of the reference that implements the trait;
* racer-cuda-sys binds every function include/racer_cuda.h declares, and its #[repr(C)] structs list the
  header's fields in the header's order;
* the Rust sources are at least lexically sound (balanced delimiters outside strings and comments).
Nothing here compiles Rust.
"""
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "racer_tracer_b200", "rust_shim")
REF = os.environ.get("RACER_TRACER_REFERENCE", "")
HEADER = open(os.path.join(ROOT, "include", "racer_cuda.h")).read()
SYS = open(os.path.join(SHIM, "racer-cuda-sys", "src", "lib.rs")).read()
DIFF = os.path.join(SHIM, "patch", "reference.diff")

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_rust_patch  # noqa: E402

needs_reference = pytest.mark.skipif(not os.path.isdir(REF) or shutil.which("patch") is None,
                                     reason="needs RACER_TRACER_REFERENCE (a checkout of the reference crate) and patch(1)")


def strip_rust(src):
    """Source without comments, string and char literals (lifetimes survive)."""
    src = re.sub(r"//[^\n]*", "", src)
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r'"(?:\\.|[^"\\])*"', '""', src)
    src = re.sub(r"'(?:\\.|[^'\\])'", "' '", src)
    return src


@needs_reference
def test_patch_applies_to_the_reference():
    r = subprocess.run(["patch", "--dry-run", "-p1", "-i", DIFF], cwd=REF, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "FAILED" not in r.stdout and "fuzz" not in r.stdout, r.stdout[-2000:]
    touched = re.findall(r"^checking file (\S+)", r.stdout, flags=re.M)
    for f in ("src/renderer.rs", "src/config.rs", "src/scene.rs", "src/bvh_node.rs", "src/camera.rs", "src/error.rs",
              "src/renderer/cuda.rs", "src/flatten.rs", "Cargo.toml"):
        assert f in touched, f


def diff_hunks(text):
    """{file: [(old lines, new lines, added lines)]} of a `diff -ruN a b`; every hunk's line counts are checked
    against its header, so that patch(1) can read it."""
    files, hunks, hunk = {}, None, None
    for ln in text.splitlines(keepends=True):
        m = re.match(r"diff -ruN a/(\S+) b/\S+$", ln)
        if m:
            hunks = files.setdefault(m.group(1), [])
            continue
        if ln.startswith(("--- a/", "+++ b/")):
            continue
        m = re.match(r"@@ -\d+(?:,(\d+))? \+\d+(?:,(\d+))? @@", ln)
        if m:
            hunk = (int(m.group(1) or 1), int(m.group(2) or 1), [], [], [])
            hunks.append(hunk)
            continue
        tag, body = ln[0], ln[1:]
        assert tag in " -+", ln
        if tag in " -":
            hunk[2].append(body)
        if tag in " +":
            hunk[3].append(body)
        if tag == "+":
            hunk[4].append(body)
    for f, hs in files.items():
        for n_old, n_new, old, new, _ in hs:
            assert (len(old), len(new)) == (n_old, n_new), f"{f}: hunk line counts differ from its header"
    return {f: [h[2:] for h in hs] for f, hs in files.items()}


def test_committed_patch_carries_the_generators_edits_and_new_files():
    """What tools/make_rust_patch.py writes, as far as it can be checked without the reference: the new files
    exactly as kept under rust_shim/, every edit's text where its anchor puts it, no line added by anything else."""
    files = diff_hunks(open(DIFF).read())
    edits = make_rust_patch.EDITS
    assert sorted(files) == sorted(set(make_rust_patch.NEW_FILES) | {e[0] for e in edits})
    for rel in make_rust_patch.NEW_FILES:
        assert [old for old, _, _ in files[rel]] == [[]], rel
        assert "".join(files[rel][0][1]) == open(os.path.join(SHIM, "racer-tracer", rel)).read(), \
            f"{rel} differs from the patch: run tools/make_rust_patch.py"
    for rel, anchor, text, where in edits:
        fragment = {"after": anchor + text, "before": text + anchor, "replace": text}[where]
        assert any(fragment in "".join(new) for _, new, _ in files[rel]), (rel, text[:80])
        if where == "replace":
            assert any(anchor in "".join(old) for old, _, _ in files[rel]), (rel, anchor[:80])
    for rel, hunks in files.items():
        if rel not in make_rust_patch.NEW_FILES:
            allowed = set("".join(e[2] for e in edits if e[0] == rel).splitlines(keepends=True))
            extra = [ln for _, _, added in hunks for ln in added if ln not in allowed]
            assert not extra, f"{rel}: lines no edit adds: {extra[:3]}"


@needs_reference
def test_committed_patch_is_what_the_generator_writes(tmp_path):
    out = make_rust_patch.build(REF, str(tmp_path / "reference.diff"))
    assert open(out).read() == open(DIFF).read(), "run tools/make_rust_patch.py"


@needs_reference
def test_every_implementor_gets_the_new_trait_method(tmp_path):
    """Apply the patch to a scratch copy; every `impl <Trait> for X` of the four extended traits must then
    contain `fn flatten`, otherwise the crate could not compile."""
    work = tmp_path / "crate"
    shutil.copytree(REF, work, ignore=lambda d, n: [x for x in n if x in ("target", ".git")])
    subprocess.run(["patch", "-p1", "-s", "-i", DIFF], cwd=work, check=True)
    n = 0
    for dirpath, _, files in os.walk(work / "src"):
        for f in files:
            src = strip_rust(open(os.path.join(dirpath, f)).read())
            for m in re.finditer(r"impl\s+(HittableSceneObject|Material|Texture|BackgroundColor)\s+for\s+(\w+)\s*\{", src):
                depth, i = 1, m.end()
                while depth and i < len(src):
                    depth += {"{": 1, "}": -1}.get(src[i], 0)
                    i += 1
                assert "fn flatten" in src[m.end():i], f"{m.group(2)}: impl {m.group(1)} lacks flatten ({f})"
                n += 1
            for name in ("{", "(", "["):
                close = {"{": "}", "(": ")", "[": "]"}[name]
                assert src.count(name) == src.count(close), f"{f}: unbalanced {name}{close}"
    assert n == 8 + 4 + 4 + 2      # geometries, materials, textures, backgrounds
    patched = open(work / "src" / "renderer.rs").read()
    assert "RendererConfig::Cuda => Box::new(cuda::CudaRenderer::new" in patched
    assert "CudaBackend(_, _) => 23" in open(work / "src" / "error.rs").read()


def test_sys_crate_binds_every_function_of_the_header():
    declared = re.findall(r"^(?:int|int64_t|const char\*)\s+(rc_\w+)\s*\(", HEADER, flags=re.M)
    assert len(declared) >= 27
    bound = set(re.findall(r"pub fn (rc_\w+)\s*\(", SYS))
    assert sorted(set(declared) - bound) == []
    assert sorted(bound - set(declared)) == []


@pytest.mark.parametrize("name", ["rc_material", "rc_texture", "rc_image", "rc_perlin", "rc_instance", "rc_bvh_node", "rc_scene",
                                  "rc_camera", "rc_params", "rc_tone_map", "rc_stats"])
def test_sys_crate_structs_follow_the_header(name):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), HEADER, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    c_fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        for part in decl.split(","):
            ident = re.findall(r"(\w+)\s*(?:\[[^\]]*\])*\s*$", part.strip())
            c_fields.append(ident[0])
    rust = re.search(r"pub struct %s \{(.*?)\n?\}" % name, SYS, flags=re.S).group(1)
    rust = re.sub(r"//[^\n]*", "", rust)
    r_fields = [f.rstrip("_") for f in re.findall(r"pub (\w+)\s*:", rust)]
    assert r_fields == c_fields, (name, c_fields, r_fields)


@pytest.mark.parametrize("rel", ["racer-tracer/src/flatten.rs", "racer-tracer/src/renderer/cuda.rs", "racer-cuda-sys/src/lib.rs",
                                 "racer-cuda-sys/build.rs"])
def test_rust_sources_are_lexically_balanced(rel):
    src = strip_rust(open(os.path.join(SHIM, rel)).read())
    for o, c in ("{}", "()", "[]"):
        assert src.count(o) == src.count(c), f"{rel}: unbalanced {o}{c}"
    assert "todo!" not in src and "unimplemented!" not in src
