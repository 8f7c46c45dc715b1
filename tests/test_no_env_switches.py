"""The library has no environment or compile-time switches that pick a code path: every kernel variant is chosen from
shape, alignment or availability. The only environment reads are MOCHA_LIB (which shared library _lib.py loads) and
NVCC (which compiler build.py runs); the only MOCHA_ macro tested by the preprocessor is MOCHA_TRACE (the trace build)."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "mocha_sigasia2023_b200")

ALLOWED_ENV = {("_lib.py", "MOCHA_LIB"), ("build.py", "NVCC")}
ALLOWED_MACROS = {"MOCHA_TRACE"}

# getenv("X") / os.getenv("X") / os.environ.get("X") / os.environ["X"]; a read whose name is not a literal is reported as "?"
ENV_READ = re.compile(r"""(?:getenv\s*\(|os\.environ\b)(?:\s*\.\s*get\s*\(|\s*\[)?\s*(?:["']([A-Za-z0-9_]+)["'])?""")
PP_COND = re.compile(r"^\s*#\s*(?:if|ifdef|ifndef|elif)\b(.*)$")


def _sources():
    files = glob.glob(os.path.join(PKG, "csrc", "*.cu*")) + glob.glob(os.path.join(PKG, "*.py"))
    assert any(f.endswith("gemm_tc.cu") for f in files) and any(f.endswith("_lib.py") for f in files)
    return sorted(files)


def test_no_environment_reads_besides_library_and_compiler():
    found = []
    for path in _sources():
        name = os.path.basename(path)
        with open(path) as f:
            for lineno, line in enumerate(f, 1):
                for m in ENV_READ.finditer(line):
                    var = m.group(1) or "?"
                    if (name, var) not in ALLOWED_ENV:
                        found.append(f"{name}:{lineno}: {var}")
    assert not found, "environment reads that select behaviour:\n" + "\n".join(found)


def test_no_preprocessor_switches_besides_trace_build():
    found = []
    for path in _sources():
        name = os.path.basename(path)
        with open(path) as f:
            lines = f.read().split("\n")
        for i, line in enumerate(lines):
            m = PP_COND.match(line)
            if not m:
                continue
            for macro in re.findall(r"\bMOCHA_[A-Za-z0-9_]*", m.group(1)):
                guard = (re.match(r"^\s*#\s*ifndef\b", line) and i + 1 < len(lines) and
                         re.match(rf"^\s*#\s*define\s+{macro}\s*$", lines[i + 1]))
                if macro not in ALLOWED_MACROS and not guard:
                    found.append(f"{name}:{i + 1}: {macro}")
    assert not found, "MOCHA_ macros that select a code path at compile time:\n" + "\n".join(found)
