"""CPU tests of the drop-in boundary: the C-ABI library loads here (no GPU), exports every symbol
include/ngmlr_b200.h declares plus the plugin factory, fails loudly without a device, and the
ABI-compat C++ header has the reference's record layout."""
import ctypes as C
import os
import re
import subprocess

import pytest

from ngmlr_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "ngmlr_b200.h")).read()
    declared = set(re.findall(r"\b(ngmlr_b200_[a-z_0-9]+)\s*\(", header))
    assert declared == set(_lib.C_API_SYMBOLS), declared ^ set(_lib.C_API_SYMBOLS)
    for s in list(declared) + list(_lib.PLUGIN_SYMBOLS):
        assert hasattr(lib, s), s
    assert lib.ngmlr_b200_abi_version() == 3
    assert lib.ngmlr_b200_plugin_cookie() == 0x10201130  # cCookie, src/IAlignment.h:193


def test_result_struct_layout_matches_header():
    # compile a tiny C program against the public header and compare sizeof/offsetof with ctypes
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "ngmlr_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu ", sizeof(ngmlr_b200_align_result), offsetof(ngmlr_b200_align_result, cigar),
         offsetof(ngmlr_b200_align_result, cells), sizeof(ngmlr_b200_batch_stats),
         offsetof(ngmlr_b200_batch_stats, fill_ms), sizeof(ngmlr_b200_scoring));
  printf("%zu %zu %zu %zu %zu %zu %zu\n", offsetof(ngmlr_b200_align_result, sv_regions),
         offsetof(ngmlr_b200_batch_stats, text_bytes), sizeof(ngmlr_b200_interval),
         offsetof(ngmlr_b200_interval, on_ref_stop), offsetof(ngmlr_b200_interval, read_seq),
         sizeof(ngmlr_b200_anchor), offsetof(ngmlr_b200_anchor, on_ref));
  printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(ngmlr_b200_sam_aln), offsetof(ngmlr_b200_sam_aln, cigar),
         offsetof(ngmlr_b200_sam_aln, identity), sizeof(ngmlr_b200_sam_read), offsetof(ngmlr_b200_sam_read, first_aln),
         offsetof(ngmlr_b200_sam_read, empty), sizeof(ngmlr_b200_sam_options), offsetof(ngmlr_b200_sam_options, rg_id));
  return 0;
}'''
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.run(["gcc", "-std=c99", "-pedantic-errors", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "t"),
                        os.path.join(d, "t.c")], check=True)
        out = subprocess.run([os.path.join(d, "t")], capture_output=True, text=True, check=True).stdout.split()
    got = [C.sizeof(_lib.AlignResult), _lib.AlignResult.cigar.offset, _lib.AlignResult.cells.offset,
           C.sizeof(_lib.BatchStats), _lib.BatchStats.fill_ms.offset, C.sizeof(_lib.Scoring),
           _lib.AlignResult.sv_regions.offset, _lib.BatchStats.text_bytes.offset, C.sizeof(_lib.Interval),
           _lib.Interval.on_ref_stop.offset, _lib.Interval.read_seq.offset, C.sizeof(_lib.Anchor),
           _lib.Anchor.on_ref.offset]
    from ngmlr_b200 import samtext as st
    got += [C.sizeof(st.SamAln), st.SamAln.cigar.offset, st.SamAln.identity.offset, C.sizeof(st.SamRead),
            st.SamRead.first_aln.offset, st.SamRead.empty.offset, C.sizeof(st.SamOptions), st.SamOptions.rg_id.offset]
    assert [int(x) for x in out] == got


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from ngmlr_b200 import B200Aligner
    with pytest.raises(RuntimeError, match="no CUDA device"):
        B200Aligner(0)
    lib = _lib.load()
    lib.CreateAlignment.restype = C.c_void_p
    assert lib.CreateAlignment(0) is None  # plugin factory fails loudly too


# sizeof/offsetof of Align, CorridorLine, PositionNM, Interval and the vtable slot order of IAlignment
PROBE = r'''
#include <stdio.h>
#include <stddef.h>
#include HEADER
#pragma GCC diagnostic ignored "-Winvalid-offsetof"
struct Probe : public IAlignment {
  int GetScoreBatchSize() const { return 11; }
  int GetAlignBatchSize() const { return 12; }
  int BatchScore(int const, int const, char const* const* const, char const* const* const, float* const, void*) { return 13; }
  int SingleAlign(int const, int const, char const* const, char const* const, Align&, void*) { return 14; }
  int SingleAlign(int const, CorridorLine*, int const, char const* const, char const* const, Align&, int const, int const, void*) { return 15; }
  int SingleScore(int const, int const, char const* const, char const* const, float&, void*) { return 16; }
  int BatchAlign(int const, int const, char const* const* const, char const* const* const, Align* const, void*) { return 17; }
};
int main() {
  printf("%zu %zu %zu %zu ", sizeof(Align), sizeof(CorridorLine), sizeof(PositionNM), sizeof(Interval));
  printf("%zu %zu %zu %zu %zu %zu %zu %zu ", offsetof(Align, pBuffer1), offsetof(Align, nmPerPosition),
         offsetof(Align, firstPosition), offsetof(Align, Score), offsetof(Align, svType),
         offsetof(Align, maxMdBufferLength), offsetof(CorridorLine, offsetInMatrix), offsetof(Interval, score));
  Probe p; IAlignment* a = &p; Align al; float f; 
  typedef int (*fn)(void*);
  void** vt = *(void***)a;
  for (int i = 0; i < 2; ++i) printf("%d ", ((fn)vt[i])(a));
  printf("\n");
  return 0;
}'''


def test_compat_header_layout_equals_reference_header():
    """The PROBE numbers of include/ngmlr_b200_ialignment.h == those of the reference's src/IAlignment.h
    (tests/golden/compiled_ref_golden.json, written by tests/golden/make_ref_golden.py)."""
    import tempfile
    import golden_util as gu
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "p.cpp")
        open(path, "w").write(PROBE.replace("HEADER", '"ngmlr_b200_ialignment.h"'))
        subprocess.run(["g++", "-std=c++11", "-w", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "p"), path,
                        "-Wl,--unresolved-symbols=ignore-all"], check=True)
        got = subprocess.run([os.path.join(d, "p")], capture_output=True, text=True, check=True).stdout
    assert got == gu.load("compiled_ref_golden.json")["abi_layout"]
