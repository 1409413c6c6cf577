"""CPU: the committed fixtures under tests/golden/ are exactly what their generator writes (tests/golden/make_fixtures.py: hand
transcriptions of the inputs and assertions of the reference's own tests, each citing file and lines), and every line range a fixture
or a source cites exists in the reference checkout (its files' line counts: tests/golden/reference/line_counts.json)."""
import json
import os
import re
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")


def reference_line_counts():
    """{path inside the reference checkout: number of lines} of its .rs / .cu files"""
    with open(os.path.join(GOLDEN, "reference", "line_counts.json")) as f:
        return json.load(f)["files"]


def test_fixtures_are_what_the_generator_writes(tmp_path):
    shutil.copy(os.path.join(GOLDEN, "make_fixtures.py"), tmp_path / "make_fixtures.py")
    r = subprocess.run([sys.executable, str(tmp_path / "make_fixtures.py")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    made = sorted(f for f in os.listdir(tmp_path) if f.endswith(".json"))
    assert made == sorted(f for f in os.listdir(GOLDEN) if f.endswith(".json")), made
    for f in made:
        assert json.load(open(tmp_path / f)) == json.load(open(os.path.join(GOLDEN, f))), f"{f}: committed fixture differs from the generator's output"


def test_cited_reference_lines_exist():
    ref_lines = reference_line_counts()
    cited = 0
    for f in sorted(os.listdir(GOLDEN)):
        if not f.endswith(".json"):
            continue
        src = json.load(open(os.path.join(GOLDEN, f))).get("source", "")
        for path, spans in re.findall(r"([\w/\.\-]+\.rs):([\d\-,: ]+)", src):
            n_lines = [n for p, n in ref_lines.items() if ("/" + path).endswith("/" + p)]
            assert len(n_lines) == 1, (f, path)
            for a in re.findall(r"\d+", spans):
                assert 1 <= int(a) <= n_lines[0], (f, path, a, n_lines[0])
                cited += 1
    assert cited >= 10


def source_files(root):
    """the files of the working tree, relative to `root` (hidden directories and bytecode caches left out)"""
    out = []
    for d, dirs, fs in os.walk(root):
        dirs[:] = sorted(x for x in dirs if not x.startswith(".") and x != "__pycache__")
        out += sorted(os.path.relpath(os.path.join(d, f), root) for f in fs)
    return out


def test_source_citations_resolve():
    """every `file.rs:line[-line]` / `file.cu:line` citation in the repository's sources and documents names a file of the reference
    checkout (by path suffix) that has that many lines — a mistyped or stale citation fails here"""
    root = os.path.dirname(HERE)
    ref_files = {"/" + f: n for f, n in reference_line_counts().items()}
    ours = {"lib.rs", "ffi.rs", "planner.rs", "reasoner.rs", "r2r.rs"}  # rust_shim's own files
    skip = ("SURVEY", "BASELINE", "PAPERS", "SNIPPETS", "VERDICT", "ADVICE")
    total, bad = 0, []
    for s in source_files(root):
        if not s.endswith((".py", ".cu", ".cuh", ".hpp", ".h", ".md", ".cpp", ".rs", ".sh")) or s.startswith(skip):
            continue
        text = open(os.path.join(root, s), errors="replace").read()
        for m in re.finditer(r"([A-Za-z_][\w/\.\-]*\.(?:rs|cu)):(\d+)(?:-(\d+))?", text):
            path, last = m.group(1), int(m.group(3) or m.group(2))
            if path.startswith(("kb_", "rust_shim", "tests/", "kolibrie_b200/")) or (path in ours and "rust_shim" in s):
                continue
            cands = [n for f, n in ref_files.items() if f.endswith("/" + path) or ("/" + path).endswith(f)]  # or cited by its absolute path
            total += 1
            if not cands or max(cands) < last:
                bad.append((s, m.group(0)))
    assert total >= 300 and not bad, bad[:20]
