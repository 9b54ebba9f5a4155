"""Every CUDA resource a context acquires is owned by a member whose destructor releases it (csrc/common.cuh: DevBuf, HostBuf and the
Owned types with their acquire helpers).  So the raw acquire and release calls of the CUDA runtime appear in those types only: a call site
elsewhere would be a resource that some hand-kept list has to free, on every error path too.  Checked on the sources, comments and string
literals stripped."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "liorf_b200", "csrc")
OWNERS = "common.cuh"

ACQUIRE = ["cudaMalloc(", "cudaMallocHost(", "cudaHostAlloc(", "cudaStreamCreate", "cudaEventCreate", "cudaGraphInstantiate(",
           "cudaStreamEndCapture(", "cudaIpcOpenMemHandle("]
RELEASE = ["cudaFree(", "cudaFreeHost(", "cudaStreamDestroy(", "cudaEventDestroy(", "cudaGraphDestroy(", "cudaGraphExecDestroy(",
           "cudaIpcCloseMemHandle("]

_TOKEN = re.compile(r'//[^\n]*|/\*.*?\*/|"(?:\\.|[^"\\\n])*"|\'(?:\\.|[^\'\\\n])*\'', re.S)


def _code(path):
    with open(path) as f:
        src = f.read()
    return _TOKEN.sub(lambda m: "\n" * m.group(0).count("\n"), src)


def _sources():
    paths = sorted(glob.glob(os.path.join(CSRC, "*.cu*")))
    assert any(p.endswith("capi.cu") for p in paths) and any(p.endswith(OWNERS) for p in paths)
    return paths


def test_strip_keeps_code_and_drops_comments_and_strings():
    import tempfile
    with tempfile.NamedTemporaryFile("w", suffix=".cu", delete=False) as f:
        f.write('a(); // cudaFree(p)\n/* cudaMalloc(\n */ b("cudaFree(x) // y"); c(\'"\');\ncudaFree(q);\n')
    try:
        code = _code(f.name)
    finally:
        os.unlink(f.name)
    assert code.count("cudaFree(") == 1 and "cudaMalloc(" not in code and code.count("\n") == 4


def test_raw_acquire_and_release_calls_only_in_the_owning_types():
    found = []
    for path in _sources():
        if os.path.basename(path) == OWNERS:
            continue
        for ln, line in enumerate(_code(path).splitlines(), 1):
            found += [f"{os.path.basename(path)}:{ln}: {name}" for name in ACQUIRE + RELEASE if name in line]
    assert not found, "raw CUDA acquire / release outside " + OWNERS + ":\n" + "\n".join(found)


def test_context_is_deleted_in_one_place():
    """liorf_create builds into a std::unique_ptr: no early return deletes the context by hand, liorf_destroy deletes it once"""
    code = _code(os.path.join(CSRC, "capi.cu"))
    assert len(re.findall(r"\bdelete\b", code)) == 1
    body = code[code.index("void liorf_destroy("):]
    body = body[:body.index("\n}\n")]
    assert "delete c;" in body
