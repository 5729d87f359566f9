"""CPU checks of the streamed tensor-core variant (R1_VARIANT_MEGAKERNEL_TENSOR_STREAM): the interface agrees on its value, the
unknown values around it are still refused before any device is looked up, and the sphere operand splits into the contiguous
16 KB chunks the kernel's one-dimensional bulk copies bring in.  The kernels themselves are tested on the GPU by
tests/test_tensor_stream_gpu.py."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from test_tensor_gpu import grid_scene

CHUNK_ROWS, ROW_BYTES = 128, 128


def test_header_python_and_executable_agree_on_the_value(r1):
    header = open(os.path.join(ROOT, "include", "rays1_b200.h")).read()
    values = {m.group(1): int(m.group(2)) for m in re.finditer(r"\b(R1_VARIANT_\w+)\s*=\s*(\d+)", header)}
    assert values["R1_VARIANT_MEGAKERNEL_TENSOR_STREAM"] == 9
    assert 8 not in values.values(), "8 stays unassigned"
    assert r1.VARIANT_MEGAKERNEL_TENSOR_STREAM == 9 and r1.VARIANTS["tensor_stream"] == 9
    assert sorted(values.values()) == sorted(set(r1.VARIANTS.values()))
    main = open(os.path.join(ROOT, "rays1bench_b200", "csrc", "rays1_main.cpp")).read()
    usage = [l for l in main.splitlines() if "--variant" in l and l.startswith("//")]
    assert len(usage) == 1 and "|tensor-stream|" in usage[0]
    assert re.search(r'!strcmp\(v, "tensor-stream"\)\) cfg\.variant = R1_VARIANT_MEGAKERNEL_TENSOR_STREAM;', main)


def test_unknown_variants_are_refused_and_9_reaches_the_device_check(r1):
    lib = r1.lib
    sc = lib.r1_scene_create(8)
    assert lib.r1_scene_add_sphere(sc, 0, 0, 0, 1, r1.MAT_LAMBERT, 0.5, 0.5, 0.5, 0) == 0
    p = r1.RenderParams(16, 9, 1, 4, 0, 0, 0, 1, 1, 0, 0, -1)
    res = r1.Result()
    rgb = np.zeros(16 * 9 * 3, np.uint8)
    for v in (8, 10, -1):
        p.variant = v
        assert lib.r1_render(sc, C.byref(p), rgb, C.byref(res)) == -1 and b"unknown variant" in lib.r1_last_error()
        assert lib.r1_render_device(sc, C.byref(p), None, None, None, C.byref(res)) == -1
    p.variant = r1.VARIANT_MEGAKERNEL_TENSOR_STREAM
    assert lib.r1_render(sc, C.byref(p), rgb, C.byref(res)) in (-2, -3)      # not committed (R1_ERR_STATE) / no device (R1_ERR_CUDA)
    assert lib.r1_render_device(sc, C.byref(p), None, None, None, C.byref(res)) in (-2, -3)
    lib.r1_scene_destroy(sc)


def operand_bytes(n32, c):
    """the operand bytes r1::tcs_fill copies for chunk c: the rows that exist (the last chunk may be short)"""
    return min(CHUNK_ROWS, n32 - CHUNK_ROWS * c) * ROW_BYTES


@pytest.mark.parametrize("grid", ((21, 16), (28, 24), (28, 27)), ids=("n32_352", "n32_704", "n32_768"))
def test_operand_chunks_are_contiguous_16k_slices(r1, grid, tmp_path):
    """chunk c (spheres 128 c .. 128 c + 127) of the K-major no-swizzle operand is bytes 16 384 c .. + rows x 128 of
    r1_tensor_operand, laid out as a 128-row operand of its own; the last chunk is short where n32 mod 128 != 0"""
    s = grid_scene(r1, tmp_path, *grid, commit=False)
    n32 = C.c_uint32(0)
    n = (s.count() + 31) // 32 * 32
    raw = np.zeros(n * ROW_BYTES, np.uint8)
    assert r1.lib.r1_tensor_operand(s.handle, raw, raw.size, C.byref(n32)) == 0 and n32.value == n
    op = s.tensor_operand()
    r, k = np.meshgrid(np.arange(CHUNK_ROWS), np.arange(32), indexing="ij")
    local = (r // 8) * 1024 + (k // 4) * 128 + (r % 8) * 16 + (k % 4) * 4   # byte offset inside one chunk
    chunks = (n + CHUNK_ROWS - 1) // CHUNK_ROWS
    covered = 0
    for c in range(chunks):
        op_bytes = operand_bytes(n, c)
        rows = op_bytes // ROW_BYTES
        piece = raw[c * 16384:c * 16384 + op_bytes]
        assert len(piece) == op_bytes and op_bytes == min(16384, n * ROW_BYTES - c * 16384)
        got = piece.view(np.float32)[local[:rows] // 4]
        assert np.array_equal(got.view(np.uint32), op[c * CHUNK_ROWS:c * CHUNK_ROWS + rows].view(np.uint32))
        covered += op_bytes
    assert covered == raw.size
    if n % CHUNK_ROWS:
        assert operand_bytes(n, chunks - 1) == (n % CHUNK_ROWS) * ROW_BYTES
    s.close()
