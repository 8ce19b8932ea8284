"""The PTX of the asynchronous hardware (mbarriers, TMA / bulk copies, tensor memory, tcgen05, cluster barriers) and the
driver lookup of cuTensorMapEncodeTiled live in csrc/ptx.cuh only.  Their encoding rules (phase parity, expect_tx byte
counts, TMEM alloc / relinquish, wait::ld after tcgen05.ld) hang or corrupt a kernel when wrong instead of failing a test, so
a kernel file must call the header rather than write its own copy."""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gencomm_b200", "csrc")
HEADER = "ptx.cuh"
PATTERNS = ("mbarrier.", "mbarrier_init", "mbarrier::", "tcgen05.", "cp.async.bulk", "barrier.cluster", "fence.proxy.async",
            "%%cluster_ctarank", "cudaGetDriverEntryPoint")
# string and character literals are kept (inline PTX is a string), comments are dropped
_TOKEN = re.compile(r'"(?:\\.|[^"\\\n])*"|\'(?:\\.|[^\'\\\n])*\'|//[^\n]*|/\*.*?\*/', re.S)


def strip_comments(src):
    return _TOKEN.sub(lambda m: m.group(0) if m.group(0)[0] in "\"'" else " ", src)


def test_strip_comments():
    src = 'a(); // mbarrier.init\n/* tcgen05.alloc\n */ asm("tcgen05.ld // x"); c = \'/\';'
    assert strip_comments(src) == 'a();  \n  asm("tcgen05.ld // x"); c = \'/\';'


def test_async_ptx_only_in_header():
    sources = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh")))
    assert HEADER in sources
    hits = {}
    for f in sources:
        with open(os.path.join(CSRC, f)) as fh:
            code = strip_comments(fh.read())
        found = [p for p in PATTERNS if p in code]
        if f != HEADER and found:
            hits[f] = found
    assert not hits, f"async-hardware PTX outside {HEADER}: {hits}"
