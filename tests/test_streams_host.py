"""CPU suite: the library keeps no per-device state a second context could overwrite, and issues no work on the legacy
default stream.  A caller who binds a context to a non-blocking stream (daisy_ctx_set_stream) gets no ordering from the
legacy stream: a pageable cudaMemcpy can return while its DMA is still in flight, and a kernel on the caller's stream then
reads stale data.  Both properties are checked on the built library and the sources, so a race that a GPU run happens to
win still fails here."""
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT
from daisyriot_b200 import _lib

CSRC = os.path.join(ROOT, "daisyriot_b200", "csrc")


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh")))


def _code(path):
    # comments removed, line breaks kept (so that reported line numbers are the file's)
    txt = open(path).read()
    txt = re.sub(r"/\*.*?\*/", lambda m: "\n" * m.group(0).count("\n"), txt, flags=re.S)
    return re.sub(r"//[^\n]*", "", txt)


def _user_device_variables(elf_dump):
    """(cubin, symbol, section) of every object symbol in .nv.constant3 (__constant__) or .nv.global (__device__) in the
    text of `cuobjdump -elf`.  Section symbols (type 3) are the sections themselves, not variables."""
    found = []
    for n, cubin in enumerate(re.split(r"\n(?=Fatbin elf code:)", elf_dump)):
        sections = {}
        for m in re.finditer(r"^\s+([0-9a-f]+)\s+[0-9a-f]+\s+[0-9a-f]+\s+[0-9a-f]+\s+[0-9a-f]+\s+[A-Z_]+\s+[0-9a-f]+\s+[0-9a-f]+\s+[0-9a-f]+\s+(\S+)\s*$",
                             cubin, flags=re.M):
            sections[int(m.group(1), 16)] = m.group(2)
        for line in cubin.splitlines():
            f = line.split()
            # index value size info other shndx name
            if len(f) != 7 or not f[0].startswith("0x") or not f[5].startswith("0x"):
                continue
            info, shndx = int(f[3], 16), int(f[5], 16)
            sec = sections.get(shndx, "")
            if (info & 0xF) != 3 and (sec.startswith(".nv.constant3") or sec.startswith(".nv.global")):
                found.append((n, f[6], sec))
    return found


def test_library_holds_no_user_device_variables():
    """A __constant__ or __device__ variable is one per device, shared by every context on it: two contexts driven from two
    host threads would overwrite each other's copy between the upload and the launch that reads it.  The sample pattern
    travels in k_ff_tiles' parameters instead.  (The DAISY_FF_STATS A/B build keeps its counters in a __device__ array; it
    is a diagnostic build and not checked here.)"""
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not on PATH")
    assert os.path.exists(_lib.SO_PATH), "build the CUDA library first"
    out = subprocess.run(["cuobjdump", "-elf", _lib.SO_PATH], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert ".nv.constant0" in out.stdout, "no cubin in the cuobjdump output: the parser would pass vacuously"
    assert _user_device_variables(out.stdout) == []


def test_device_variable_parser_finds_constant_and_global():
    # the parser above must see what it is looking for: a minimal dump with one __constant__ and one __device__ array
    dump = """Fatbin elf code:
================
Sections:
Index Offset   Size ES Align        Type   Flags Link     Info Name
    1     40    2c1  0  1            STRTAB       0    0        0 .shstrtab
   23 1040f8    300  0  4          PROGBITS       2    0        0 .nv.constant3
   24 104400    180  0  8            NOBITS       3    0        0 .nv.global

.section .symtab
 index           value           size      info    other  shndx    name
   0               0               0        0        0      0     (null)
 0x4               0               0      0x3        0   0x23     .nv.constant3
 0x5               0           0x200      0x1        0   0x23     c_uv
 0x6               0           0x180      0x1        0   0x24     g_counts
 0x7           0x400             0x4     0x21        0      0     .nv.reservedSmem.cap
"""
    assert _user_device_variables(dump) == [(0, "c_uv", ".nv.constant3"), (0, "g_counts", ".nv.global")]


LEGACY_CALLS = ("cudaMemcpy", "cudaMemcpy2D", "cudaMemset", "cudaMemcpyToSymbol", "cudaMemcpyFromSymbol")


def _launch_configs(code):
    """(offset, argument list) of every <<<...>>> launch configuration, split at top-level commas."""
    out = []
    for m in re.finditer(r"<<<(.*?)>>>", code, flags=re.S):
        args, depth, cur = [], 0, ""
        for ch in m.group(1):
            if ch in "([{":
                depth += 1
            elif ch in ")]}":
                depth -= 1
            if ch == "," and depth == 0:
                args.append(cur.strip()); cur = ""
            else:
                cur += ch
        args.append(cur.strip())
        out.append((m.start(), args))
    return out


def test_sources_issue_no_legacy_stream_work():
    """Every copy, memset and launch names the context's stream: no synchronous cudaMemcpy / cudaMemcpy2D / cudaMemset /
    symbol copy, and no launch without a stream argument.  (Allocation and cudaFree are not stream work.)"""
    bad = []
    nlaunch = 0
    for path in _sources():
        code = _code(path)
        name = os.path.basename(path)
        for call in LEGACY_CALLS:
            for m in re.finditer(r"\b%s\s*\(" % call, code):
                bad.append("%s:%d: %s(" % (name, code.count("\n", 0, m.start()) + 1, call))
        for at, args in _launch_configs(code):
            nlaunch += 1
            if len(args) < 4 or args[3] in ("", "0", "nullptr", "NULL", "cudaStreamLegacy"):
                bad.append("%s:%d: launch <<<%s>>> without a stream" % (name, code.count("\n", 0, at) + 1, ", ".join(args)))
    assert nlaunch > 20, "found only %d launches: the scan is broken" % nlaunch
    assert not bad, "\n".join(bad)


def test_launch_parser_splits_at_top_level_commas():
    code = "k<<<dim3((N + 1) / 2, nrb), 256, 0, c->stream>>>(a); k2<<<grid, block>>>(b); f<K, R><<<std::max(a, b), 128>>>(c);"
    assert [a for _, a in _launch_configs(code)] == [["dim3((N + 1) / 2, nrb)", "256", "0", "c->stream"], ["grid", "block"], ["std::max(a, b)", "128"]]
