"""CPU checks of the tensor-core filter's HOST side and of its formulation (rays1bench_b200/csrc/r1_tensor.cuh):
the sphere operand the library builds (layout, TF32 split, padding rows) and a numpy emulation of the split-TF32 dot product
against the float64 polynomial and against the oracle's Hitable::hit.  The hardware side (tcgen05.mma accumulation) is measured
on the GPU by tests/test_gpu_parity.py::test_tensor_filter_is_conservative."""
import numpy as np
import pytest

from test_gpu_parity import tensor_filter_far_rays, tensor_filter_rays, tensor_filter_truth   # ray generators and float64 truth shared with the GPU tests
from test_tensor_gpu import GRIDS, TENSOR, grid_scene                # the sphere-count sweep of the tensor path

MARGIN = 2.0 ** -16


def tf32_rna(x):
    """cvt.rna.tf32.f32: round to nearest (ties away), 10 explicit mantissa bits, low 13 bits zero"""
    b = np.ascontiguousarray(x, np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def sphere_features(soa):
    """float64 lifted sphere vectors [n, 11] (r1_tensor.cuh): nx^2 ny^2 nz^2 nxny nxnz nynz nx ny nz kk 1"""
    nx, ny, nz = (-soa[k].astype(np.float64) for k in ("cx", "cy", "cz"))
    c2 = nx * nx + ny * ny + nz * nz
    kk = c2 - soa["radius_sq"].astype(np.float64) - c2 * MARGIN
    return np.stack([nx * nx, ny * ny, nz * nz, nx * ny, nx * nz, ny * nz, nx, ny, nz, kk, np.ones_like(nx)], 1)


def ray_rows(org, d):
    """numpy mirror of tc::ray_row: the 32 TF32 words {hi x 11 | lo x 11 | hi x 10} of each ray, float32 arithmetic"""
    f32 = np.float32
    o, dd = org.astype(f32), d.astype(f32)
    od = (o[:, 0] * dd[:, 0] + o[:, 1] * dd[:, 1] + o[:, 2] * dd[:, 2]).astype(f32)
    oo = (o[:, 0] * o[:, 0] + o[:, 1] * o[:, 1] + o[:, 2] * o[:, 2]).astype(f32)
    f = np.stack([dd[:, 0] * dd[:, 0], dd[:, 1] * dd[:, 1], dd[:, 2] * dd[:, 2],
                  (dd[:, 0] + dd[:, 0]) * dd[:, 1], (dd[:, 0] + dd[:, 0]) * dd[:, 2], (dd[:, 1] + dd[:, 1]) * dd[:, 2],
                  f32(2) * (od * dd[:, 0] - o[:, 0]), f32(2) * (od * dd[:, 1] - o[:, 1]), f32(2) * (od * dd[:, 2] - o[:, 2]),
                  np.full(len(o), -1, f32), od * od - oo * f32(1.0 - MARGIN)], 1).astype(f32)
    hi = tf32_rna(f)
    lo = tf32_rna((f - hi).astype(f32))
    return np.concatenate([hi, lo, hi[:, :10]], 1)


def cpu_scene(r1, name, tmp_path):
    """a built-in scene, or a sweep scene "WxH" of tests/test_tensor_gpu.py, host side only"""
    if "x" in name:
        return grid_scene(r1, tmp_path, *map(int, name.split("x")), commit=False)
    return r1.create_scene(name, commit=False)


@pytest.mark.parametrize("name", ("small", "medium", "large", "21x16", "28x27"))
def test_tensor_operand_layout_split_and_padding(r1, name, tmp_path):
    """incl. a 96-row last chunk (n32 = 352) and the largest operand the filter takes (760 spheres, n32 = 768: 96 KB)"""
    s = cpu_scene(r1, name, tmp_path)
    soa = s.soa()
    op = s.tensor_operand()
    n, n32 = len(soa["cx"]), op.shape[0]
    assert n32 == (n + 31) // 32 * 32 and op.shape[1] == 32
    assert (op.view(np.uint32) & 0x1FFF == 0).all(), "every word is a TF32 value"
    real = soa["inv_radius"] > 0
    assert np.array_equal(op[:, 0:11], op[:, 11:22]), "hi words are stored twice (x ray hi, x ray lo)"
    f = sphere_features(soa)[real]
    hi, lo = op[:n][real][:, 0:11].astype(np.float64), op[:n][real][:, 22:32].astype(np.float64)
    assert np.array_equal(hi[:, 10], np.ones(real.sum())), "the constant feature is exact and has no low part"
    rebuilt = hi.copy()
    rebuilt[:, :10] += lo
    assert (np.abs(rebuilt - f) <= 2.0 ** -21 * np.abs(f)).all(), "hi + lo carries the feature to 2^-21"
    assert (np.abs(hi - f) <= 2.0 ** -11 * np.abs(f) + 1e-300).all()
    pad = np.ones(n32, bool)
    pad[:n] = ~real
    assert pad.sum() >= n32 - n
    rows = op[pad]
    assert (rows[:, [9, 20]] > 9e29).all(), "rows no ray can flag: kk = 1e30"
    assert (np.delete(rows, [9, 20, 31], 1) == 0).all()
    s.close()


def test_tensor_operand_limits(r1, tmp_path):
    import ctypes as C
    s = r1.create_scene("synth4096", commit=False)
    n32 = C.c_uint32(0)
    assert r1.lib.r1_tensor_operand(s.handle, np.zeros(16, np.uint8), 16, C.byref(n32)) == -4 and n32.value == 4096   # R1_ERR_LIMIT
    assert b"768" in r1.lib.r1_last_error()
    s.close()
    for grid, (count, want_n32) in GRIDS.items():             # the sweep: 768 is the last accepted, 800 the first refused
        s = grid_scene(r1, tmp_path, *grid, commit=False)
        rc = r1.lib.r1_tensor_operand(s.handle, np.zeros(16, np.uint8), 16, C.byref(n32))
        assert s.count() == count and n32.value == want_n32
        if want_n32 <= 768:
            assert rc == -1, "accepted: only the 16-byte buffer is too small"
            assert r1.lib.r1_tensor_operand(s.handle, np.zeros(want_n32 * 128, np.uint8), want_n32 * 128, C.byref(n32)) == 0
        else:
            assert rc == -4 and b"768" in r1.lib.r1_last_error() and b"800" in r1.lib.r1_last_error()
        s.close()
    s = r1.create_scene("small", commit=False)
    assert r1.lib.r1_tensor_operand(s.handle, np.zeros(16, np.uint8), 16, C.byref(n32)) == -1 and n32.value == 32       # buffer too small
    s.close()


@pytest.mark.parametrize("name", ("medium", "large") + tuple("%dx%d" % g for g in TENSOR))
def test_tensor_filter_formulation_is_conservative(r1, oracle, name, tmp_path):
    """A[ray] . B[sphere] with the split operands exactly as the device and the host build them (products and sum in float64):
    within 2^-20 S of the float64 polynomial, and every sphere the oracle's Hitable::hit returns is flagged.  On the sweep scenes
    the rays include ones grazing spheres from 2 000 and 20 000 units."""
    s = cpu_scene(r1, name, tmp_path)
    soa = s.soa()
    n = len(soa["cx"])
    org, d = tensor_filter_rays(soa, n=1024) if "x" not in name else tensor_filter_far_rays(soa, n=512)
    a = ray_rows(org, d).astype(np.float64)
    op = s.tensor_operand().astype(np.float64)
    b = np.concatenate([op[:, 0:11], op[:, 11:22], op[:, 22:32]], 1)      # sphere words in K order: hi | hi | lo
    e = a @ b.T
    want, discr, big_s = tensor_filter_truth(soa, org, d)
    real = soa["inv_radius"] > 0
    err = (np.abs(e[:, :n] - want) / big_s)[:, real]
    assert err.max() < 2.0 ** -20, err.max()
    must = (discr >= -4.0e-6 * big_s) & real[None, :]
    assert must.sum() > 500 and (e[:, :n][must] >= 0).all()
    assert (e[:, n:] < 0).all() and (e[:, :n][:, ~real] < 0).all()
    so = oracle.scene_create_from_soa(soa)
    idx = oracle.hit(so, org, d)[0]
    oracle.scene_destroy(so)
    hit = idx >= 0
    assert hit.sum() > 300
    assert (e[np.arange(len(idx))[hit], idx[hit]] > 0).all(), "a sphere Hitable::hit returns must pass the filter"
    s.close()
