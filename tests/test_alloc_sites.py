"""CPU: every device allocation and pinned host buffer of a context comes from ewk::Pool (ewk_ctx.hpp), so poison mode
(EWK_POISON, tests/test_gpu_poison.py) covers every buffer the library owns, including future ones."""
import os
import re

from conftest import REPO

CSRC = os.path.join(REPO, "easywakeword_b200", "csrc")
ALLOC = re.compile(r"\b(cudaMalloc\w*|cudaHostAlloc|cudaMallocHost|cuMemAlloc\w*)\s*\(")
# the only places allowed to allocate: the pool itself, and ewk_host_alloc, which allocates for the caller
ALLOWED = ("cudaError_t Pool::alloc(", "cudaError_t Pool::alloc_host(", 'extern "C" int ewk_host_alloc(')


def _function_of(src, pos):
    """the line that opens the top-level function around pos"""
    start = src.rfind("\n}", 0, pos)
    head = src[start + 2 if start >= 0 else 0:pos]
    for line in head.splitlines():
        if line and not line[0].isspace() and not line.startswith(("//", "#")):
            return line
    return ""


def test_every_allocation_goes_through_the_pool():
    bad = []
    for f in sorted(os.listdir(CSRC)):
        src = open(os.path.join(CSRC, f)).read()
        for m in ALLOC.finditer(src):
            fn = _function_of(src, m.start())
            if not fn.startswith(ALLOWED):
                bad.append(f"{f}:{src.count(chr(10), 0, m.start()) + 1}: {m.group(1)} in {fn[:60]!r}")
    assert not bad, "allocations outside ewk::Pool:\n" + "\n".join(bad)


def test_devbuf_has_no_default_constructor():
    """a DevBuf must be given its pool and name, so no buffer can be declared that bypasses poison mode"""
    hpp = open(os.path.join(CSRC, "ewk_ctx.hpp")).read()
    body = hpp[hpp.index("struct DevBuf {"):hpp.index("};", hpp.index("struct DevBuf {"))]
    assert "DevBuf(Pool* pool_, const char* name_, bool scratch_)" in body
    assert "DevBuf()" not in body
