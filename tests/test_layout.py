"""The product never touches the oracle, the reference tree or a CPU fallback."""
import ast
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "visual-odometry-pipeline_b200")
# a command word naming a profiler or sanitizer, bare or as a path
PROFILER = re.compile(r"(?:^|/)(?:ncu|nsys|compute-sanitizer|nv-nsight-cu-cli)$")


def _sources():
    for base, _, files in os.walk(PKG):
        if "build" in base.split(os.sep):
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".sh")):
                yield os.path.join(base, f)


def test_product_does_not_import_oracle_or_reference():
    pat = re.compile(r"(from\s+oracle|import\s+oracle|/root/reference|oracle/)")
    bad = [p for p in _sources() if pat.search(open(p).read())]
    assert not bad, bad


def test_no_compat_layers_in_product():
    pat = re.compile(r"\b(import triton|torch\.compile|tilelang)\b")
    bad = [p for p in _sources() if pat.search(open(p).read())]
    assert not bad, bad


def _command_words(path):
    """Words that can name a program to run: in a shell script every word outside comments; in Python the first word of
    every string literal that is not a docstring (an argv[0], a command line, a path).  Prose stays out of both."""
    src = open(path).read()
    if path.endswith(".sh"):
        return [w for line in src.splitlines() for w in re.split(r"[\s;&|()<>=`'\"]+", re.sub(r"(^|\s)#.*", "", line))]
    tree = ast.parse(src)
    docs = {id(n.body[0].value) for n in ast.walk(tree)
            if isinstance(n, (ast.Module, ast.ClassDef, ast.FunctionDef, ast.AsyncFunctionDef)) and n.body
            and isinstance(n.body[0], ast.Expr) and isinstance(n.body[0].value, ast.Constant)}
    return [n.value.split()[0] for n in ast.walk(tree)
            if isinstance(n, ast.Constant) and isinstance(n.value, str) and n.value.split() and id(n) not in docs]


def test_no_script_runs_a_profiler_or_sanitizer():
    # Nsight Compute / Systems and compute-sanitizer are not part of the GPU environment the project is run in (and
    # compute-sanitizer runs have left GPUs needing a reset); kernel time comes from CUDA events and torch.profiler
    bad = []
    for top in ("tools", "tests", os.path.basename(PKG)):
        for base, dirs, files in os.walk(os.path.join(ROOT, top)):
            dirs[:] = [d for d in dirs if d not in ("build", "__pycache__")]
            for f in files:
                p = os.path.join(base, f)
                if f.endswith((".sh", ".py")) and any(PROFILER.search(w) for w in _command_words(p)):
                    bad.append(os.path.relpath(p, ROOT))
    assert not bad, bad


def test_required_files_exist():
    for rel in ("include/vo_b200.h", "oracle/vo_oracle.c", "oracle/oracle.py", "bench.py", "__graft_entry__.py",
                "DESIGN.md", "INTEGRATION.md", "tests/golden/make_golden.py", "oracle/orb_frontend.py", "oracle/sift_frontend.py",
                "tests/golden/make_orb_golden.py", "tests/golden/make_sift_golden.py", "tests/golden/orb_pattern.npy"):
        assert os.path.exists(os.path.join(ROOT, rel)), rel
