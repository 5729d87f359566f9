"""CPU-side checks of the C-ABI library and the host logic: the library loads and exports every symbol the header
declares, the scene builders produce the reference's SoA arrays bit for bit, the row-tile partition is a partition,
compute entry points fail loudly without a GPU, TGA / log files have the reference's format, and the two-collective
exchange works at world_size 2 over gloo.  No kernels run here."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, SCENES


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_library_exports_every_declared_symbol(r1):
    header = open(os.path.join(ROOT, "include", "rays1_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(r1_\w+)\s*\(", header))
    assert len(declared) >= 30
    nm = subprocess.run(["nm", "-D", "--defined-only", r1.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\sT\s+(r1_\w+)", nm))
    assert declared <= exported, sorted(declared - exported)
    assert declared == set(r1.EXPORTED), sorted(declared ^ set(r1.EXPORTED))
    assert r1.lib.r1_abi_version() == 2


def test_library_is_built_for_sm100a_only(r1):
    out = subprocess.run(["cuobjdump", "-lelf", r1.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\w+)\.", out))
    assert archs == {"100a"}, archs


def test_product_does_not_link_or_reference_the_oracle(r1):
    """the oracle is test infrastructure: nothing under rays1bench_b200/ may name it"""
    pkg = os.path.join(ROOT, "rays1bench_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "rays1_oracle" not in text and "cpu_checkers" not in text and "oracle/" not in text, f
    ldd = subprocess.run(["ldd", r1.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in ldd and "libref" not in ldd


@pytest.mark.parametrize("name", SCENES + ("synth4096",))
def test_scene_builders_match_oracle_bit_for_bit(r1, oracle, name):
    s = r1.create_scene(name, commit=False)
    so = oracle.scene_create(name)
    a, b = s.soa(), oracle.scene_soa(so)
    assert s.count() == oracle.scene_count(so) == {"small": 8, "medium": 48, "large": 488, "synth4096": 4096}[name]
    for k in a:
        assert np.array_equal(a[k], b[k]) if a[k].dtype != np.float32 else np.array_equal(bits(a[k]), bits(b[k])), k
    assert np.array_equal(bits(s.camera()), bits(oracle.scene_camera(so)))
    oracle.scene_destroy(so)
    s.close()


@pytest.mark.parametrize("name", SCENES + ("synth4096",))
def test_scene_builders_match_reference_golden(r1, golden_rays, name):
    """every SoA array -- centres, radius^2, 1/radius, albedo, fuzz / ior -- has the reference's exact bits (synth4096: the
    MAX_SPHERES = 4096 build of the reference with the 4096-sphere builder on its own classes)"""
    s = r1.create_scene(name, commit=False)
    a, g = s.soa(), golden_rays[name]
    for k in ("cx", "cy", "cz", "radius_sq", "inv_radius", "albedo", "param"):
        assert np.array_equal(bits(a[k]), bits(g["soa_" + k])), k
    assert np.array_equal(a["kind"], g["soa_kind"])
    # the 22 camera constants (gcc folds Camera::init at compile time after its fast-math reassociation; r1_scene_set_camera
    # evaluates it the same way) have the reference's exact bits too
    assert np.array_equal(bits(s.camera()), bits(g["camera"]))
    cam = g["camera"].copy()
    cam[21] = 0.25
    s.set_camera_raw(cam)                                   # constants installed as given
    assert np.array_equal(bits(s.camera()), bits(cam))
    # placeholders: radius 0 at 999999999, no material (rayweek1.cpp:575-576); the hollow shell keeps inv_radius 0
    ph = a["kind"] == r1.MAT_NONE
    assert (a["cx"][ph] == np.float32(999999999)).all() and (a["inv_radius"][ph] == 0).all()
    if name == "small":
        assert a["inv_radius"][4] == 0 and a["radius_sq"][4] == np.float32(-0.45) * np.float32(-0.45)
    s.close()


def test_scene_abi_argument_checking(r1):
    import ctypes as C
    lib = r1.lib
    sc = lib.r1_scene_create(4)
    assert lib.r1_scene_add_sphere(sc, 0, 0, 0, 1.0, 7, 0, 0, 0, 0) == -1      # unknown material
    assert lib.r1_scene_add_sphere(sc, 0, 0, 0, 1.0, r1.MAT_NONE, 0, 0, 0, 0) == -1  # real sphere needs a material
    assert lib.r1_scene_add_sphere(sc, 0, 0, 0, 1.0, r1.MAT_METAL, .5, .5, .5, 3.0) == 0
    assert lib.r1_scene_pad(sc, 8) == 0 and lib.r1_scene_count(sc) == 8
    n = 8
    arr = lambda k=1: np.zeros(n * k, np.float32)  # noqa: E731
    cx, cy, cz, r2, ir, al, pa, kind = arr(), arr(), arr(), arr(), arr(), arr(3), arr(), np.zeros(n, np.int32)
    assert lib.r1_scene_get_soa(sc, cx, cy, cz, r2, ir, kind, al, pa) == 0
    assert pa[0] == 1.0, "Metal fuzz is clamped to <= 1 (rayweek1.cpp:424)"
    assert lib.r1_scene_commit(sc, 0) == -2 and b"camera" in lib.r1_last_error()  # camera not set
    p = r1.RenderParams(16, 9, 1, 50, 0, 0, 0, 1, 8, 0, 0, -1)
    res = r1.Result()
    assert lib.r1_render(sc, C.byref(p), np.zeros(16 * 9 * 3, np.uint8), C.byref(res)) == -2  # not committed
    p.world = 0
    assert lib.r1_render(sc, C.byref(p), np.zeros(16 * 9 * 3, np.uint8), C.byref(res)) == -1
    p.world, p.spp = 1, (1 << 20) + 1                                           # the 64-bit fixed-point pixel sums are sized for 2^20 samples
    assert lib.r1_render(sc, C.byref(p), np.zeros(16 * 9 * 3, np.uint8), C.byref(res)) == -4 and b"2^20" in lib.r1_last_error()
    p.spp, p.variant = 1, 8
    assert lib.r1_render(sc, C.byref(p), np.zeros(16 * 9 * 3, np.uint8), C.byref(res)) == -1  # unknown variant
    assert lib.r1_scene_set_camera_raw(sc, np.zeros(22, np.float32)) == 0
    assert lib.r1_scene_commit(sc, 0) == -3 or lib.r1_device_count() > 0         # camera now set: the next obstacle is the missing GPU
    lib.r1_scene_destroy(sc)


def test_pixel_buffer_sizes_are_checked(r1, tmp_path):
    """benchmark() / tga_write_rgb24() never write past a caller's buffer that is too small for the configured image"""
    r1.configure(width=64, height=36, spp=1, quiet=True)
    try:
        s = r1.create_scene("small", commit=False)
        with pytest.raises(ValueError, match="configured 64x36"):
            r1.benchmark(s, np.zeros((10, 10, 3), np.uint8), False, "small")
        assert s.count() == 8, "a rejected call does not consume the scene"
        # the C entry point itself: too small -> R1_ERR_ARG, scene consumed, nothing written
        import ctypes as C
        ptr, s._ptr = s._ptr, None
        small = np.full(300, 7, np.uint8)
        rc = r1.lib.r1_host_benchmark(ptr, small, small.size, 0, b"small", None, None, None)
        assert rc == -1 and b"needs 6912" in r1.lib.r1_last_error() and (small == 7).all()
        with pytest.raises(ValueError):
            r1.tga_write_rgb24(str(tmp_path / "x.tga"), 8, 8, np.zeros(100, np.uint8))
        buf = np.zeros(100, np.uint8)
        assert r1.lib.r1_host_write_tga(str(tmp_path / "x.tga").encode(), 8, 8, buf, buf.size) == -1
        assert not (tmp_path / "x.tga").exists()
    finally:
        r1.configure(width=1280, height=720, spp=250, quiet=True)


def test_header_declares_what_the_library_exports(r1):
    """every function include/rays1_b200.h declares is exported by the library and bound by the Python module, and vice versa"""
    hdr = open(os.path.join(ROOT, "include", "rays1_b200.h")).read()
    declared = set(re.findall(r"\b(r1_[a-z0-9_]+)\s*\(", hdr)) - {"r1_scene", "r1_result", "r1_render_params"}
    nm = subprocess.run(["nm", "-D", "--defined-only", r1.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (r1_[a-z0-9_]+)$", nm, re.M))
    assert declared <= exported, declared - exported
    assert declared == set(r1.EXPORTED), declared ^ set(r1.EXPORTED)
    assert r1.lib.r1_abi_version() == 2


def test_no_cpu_fallback_without_a_gpu(r1):
    """On a box without a CUDA device every compute entry point must fail loudly (never render on the CPU)."""
    try:
        n = r1.device_count()
    except r1.Rays1Error:
        n = 0
    if n > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(r1.Rays1Error):
        r1.create_large_scene()
    with pytest.raises(r1.Rays1Error):
        r1.fma_peak()
    s = r1.create_scene("small", commit=False)
    with pytest.raises(r1.Rays1Error):
        s.render(16, 9, 1)
    with pytest.raises(r1.Rays1Error):
        s.trace_rays(np.zeros((1, 3)), np.array([[0, 0, 1.0]]))
    with pytest.raises(r1.Rays1Error, match=r"\(-3\)"):
        s.render_sums(16, 9, 1)
    with pytest.raises(r1.Rays1Error, match=r"\(-3\)"):
        r1.sample_points([0], [0], 0, 2)
    # arguments are checked before any device is looked up
    with pytest.raises(r1.Rays1Error, match=r"\(-1\)"):
        s.render_sums(16, 9, 0)
    with pytest.raises(r1.Rays1Error, match=r"\(-1\)"):
        r1.sample_points([0], [0], 0, -1)
    s.close()


@pytest.mark.parametrize("layout", (1, -1, 2))
def test_filter_probe_refuses_layouts_other_than_0(r1, layout):
    """r1_filter_probe reads the operand in the renderer's layout only: any other `layout` is R1_ERR_ARG before the device is
    looked at (this scene is not even committed)"""
    s = r1.create_scene("small", commit=False)
    try:
        with pytest.raises(r1.Rays1Error, match=r"\(-1\).*layout"):
            s.filter_probe(np.zeros((1, 3)), np.array([[0, 0, 1.0]]), 1, layout=layout)
    finally:
        s.close()


@pytest.mark.parametrize("height,row_tile,world", [(720, 8, 1), (720, 8, 2), (720, 8, 8), (2160, 8, 8), (37, 8, 4), (5, 8, 8), (100, 3, 7)])
def test_row_tile_partition_is_a_partition(r1, height, row_tile, world):
    seen = []
    for rank in range(world):
        rows = r1.local_rows(height, row_tile, rank, world)
        ys = [r1.global_row(lr, row_tile, rank, world) for lr in range(rows)]
        assert ys == sorted(ys), "local rows are in ascending global order"
        assert all((y // row_tile) % world == rank for y in ys)
        seen += ys
    assert sorted(seen) == list(range(height))
    counts = [r1.local_rows(height, row_tile, r, world) for r in range(world)]
    assert max(counts) - min(counts) <= row_tile


def test_tga_writer_format(r1, tmp_path):
    """common.h:86-122: 18-byte header, type 2, 24 bpp, descriptor 0, BGR payload, and R/B swapped IN PLACE."""
    w, h = 5, 3
    px = np.arange(w * h * 3, dtype=np.uint8).reshape(h, w, 3)
    orig = px.copy()
    path = str(tmp_path / "out_x.tga")
    r1.tga_write_rgb24(path, w, h, px)
    raw = open(path, "rb").read()
    assert len(raw) == 18 + w * h * 3
    assert list(raw[:18]) == [0, 0, 2, 0, 0, 0, 0, 0, 0, 0, 0, 0, w, 0, h, 0, 24, 0]
    body = np.frombuffer(raw[18:], np.uint8).reshape(h, w, 3)
    assert np.array_equal(body, orig[:, :, ::-1])
    assert np.array_equal(px, orig[:, :, ::-1]), "the caller's buffer is swapped too, as in the reference"


def test_log_results_format(r1, tmp_path, monkeypatch):
    """common.h:47-77 -> 'version|%.3fs|<rays>|%0.3f mrays/s|' (no newline), averaged; parsed by update_readme.py:30-31"""
    monkeypatch.chdir(tmp_path)
    a, b = r1.Result(), r1.Result()
    a.elapsed_seconds, a.num_rays = 2.0, 100_000_000
    b.elapsed_seconds, b.num_rays = 4.0, 300_000_000
    r1.log_results("b200", "large", [a, b])
    txt = open(tmp_path / "out_large.txt").read()
    assert txt == "b200|3.000s|200000000|66.667 mrays/s|"
    tokens = txt.split("|")
    assert float(tokens[3].split()[0]) == pytest.approx(66.667)


def test_flops_model(r1):
    # SURVEY.md 8d: F_ray = 16 N + 70 -> small 150, medium 806, large 7814, synthetic 65606
    assert [r1.flops_per_ray(r1.REAL_SPHERES[k]) for k in ("small", "medium", "large", "synth4096")] == [150, 806, 7814, 65606]


GLOO_WORKER = r"""
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
import rays1bench_b200 as r1
from rays1bench_b200 import dist as r1d
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
W, H, T = 13, 37, 4
rows = r1.local_rows(H, T, rank, world)
mx = r1d.max_local_rows(H, T, world)
local = torch.zeros((mx, W, 3), dtype=torch.uint8)
for lr in range(rows):
    y = r1.global_row(lr, T, rank, world)
    local[lr] = torch.tensor([(y * 7 + x * 3 + c) % 256 for x in range(W) for c in range(3)], dtype=torch.uint8).reshape(W, 3)
gathered = r1d.gather_framebuffer(local, H, T, rank, world)
count = r1d.reduce_ray_count(torch.tensor([1000 + rank], dtype=torch.int64), world)
if rank == 0:
    parts = [gathered[r, : r1.local_rows(H, T, r, world)].numpy() for r in range(world)]
    img = r1.assemble_rows(parts, H, T)
    want = np.array([[[(y * 7 + x * 3 + c) % 256 for c in range(3)] for x in range(W)] for y in range(H)], np.uint8)
    assert np.array_equal(img, want)
    assert int(count) == sum(1000 + r for r in range(world)), int(count)
    print("GLOO_OK")
else:
    assert gathered is None
dist.destroy_process_group()
"""


def test_two_collective_exchange_world2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29641", str(script), ROOT]
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "GLOO_OK" in out.stdout


def test_scene_file_round_trip_matches_builtin_builders(r1, tmp_path):
    """SURVEY 8f rank 3: the text scene format reproduces create_large_scene() / the 4096-sphere scene bit for bit."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_scene
    for name, args in (("large", (30, 16, 0, (3, 8, 15), 10.0)), ("synth4096", (66, 62, 480, (6, 16, 30), 20.0))):
        cam, sph = make_scene.grid_scene(*args)
        path = str(tmp_path / (name + ".r1scene"))
        r1.write_scene_file(path, cam, sph)
        a = r1.create_scene_from_file(path, commit=False)
        b = r1.create_scene(name, commit=False)
        sa, sb = a.soa(), b.soa()
        assert a.count() == b.count()
        for k in sa:
            assert np.array_equal(sa[k].view(np.uint32) if sa[k].dtype == np.float32 else sa[k],
                                  sb[k].view(np.uint32) if sb[k].dtype == np.float32 else sb[k]), (name, k)
        assert np.array_equal(a.camera(), b.camera())
        a.close()
        b.close()
    bad = tmp_path / "bad.r1scene"
    bad.write_text("camera 0 0 5 0 0 0 60 0.1 5\nsphere 0 0 0 1 plastic 1 1 1\n")
    with pytest.raises(r1.Rays1Error):
        r1.create_scene_from_file(str(bad), commit=False)
    with pytest.raises(r1.Rays1Error):
        r1.create_scene_from_file(str(tmp_path / "missing.r1scene"), commit=False)


def test_compare_tga_tool(r1, tmp_path):
    """SURVEY 8f rank 2: TGA reader / RMSE / PNG export agree with the writer (BGR, bottom-up)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import compare_tga
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (9, 16, 3), dtype=np.uint8)      # row 0 = bottom, RGB
    px = img.copy()
    r1.tga_write_rgb24(str(tmp_path / "a.tga"), 16, 9, px)
    got = compare_tga.read_image(str(tmp_path / "a.tga"))
    assert np.array_equal(got, img[::-1])                        # top-down RGB
    other = img.copy()
    other[0, 0, 0] ^= 0x10
    np.savez(tmp_path / "b.npz", rgb=other)
    r = compare_tga.compare(got, compare_tga.read_image(str(tmp_path / "b.npz")))
    assert r["max_abs"] == 16 and not r["identical"] and 0 < r["rmse"] < 1
    compare_tga.write_png(str(tmp_path / "a.png"), got)
    raw = open(tmp_path / "a.png", "rb").read()
    assert raw[:8] == b"\x89PNG\r\n\x1a\n" and b"IDAT" in raw


def test_bench_reference_arm_json_contract():
    """`bench.py --impl reference` (the CPU arm: the reference's own code where oracle/_ref was built, else the oracle port)
    prints ONE JSON line with the benchmark's keys."""
    import json
    import subprocess
    import sys
    from cpu_checkers import RefLib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-budget", "0.3", "--workload", "small"], capture_output=True, text=True, timeout=300, check=True).stdout
    lines = [l for l in out.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True
    assert d["metric"] == "Mrays/s (small scene)" and d["config"]["workload"].startswith("small scene 1280x720 250 spp")
    assert d["value"] > 0 and d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if RefLib.available() else "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "spp" in cb["sample"]
    assert d["gpu_launches"] == 0 and 1.7 < d["rays_per_sample"] < 1.9   # small scene: 1.798 rays per sample (ref_stats.json)


def test_bench_steps_tool_compiles_the_executable(r1):
    """tools/bench_steps.py (the reference's bench.py driver for this build, SURVEY 8f rank 1): --compile-only builds the
    in-tree executable with nvcc and stops, like the reference's --compile-only (bench.py:100-104 there)"""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_steps.py"), "--latest", "--compile-only"],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip().splitlines()[-1] == "compiled " + r1.EXE_PATH
    assert os.access(r1.EXE_PATH, os.X_OK) and "RUN " not in out.stdout


def test_header_is_plain_c_and_links(r1, tmp_path):
    """include/rays1_b200.h is the boundary a C (cgo / FFI) binding would consume: it compiles as strict C99 and a C program
    links against the library with nothing but that header"""
    src = tmp_path / "abi.c"
    src.write_text('#include "rays1_b200.h"\n'
                   'int main(void) {\n'
                   '    r1_render_params p; r1_result r; (void)p; (void)r;\n'
                   '    if (r1_abi_version() != R1_ABI_VERSION) return 1;\n'
                   '    r1_scene *s = r1_scene_create(8);\n'
                   '    if (r1_scene_add_sphere(s, 0, 0, 0, 1.0f, R1_MAT_LAMBERT, .5f, .5f, .5f, 0) != 0) return 2;\n'
                   '    if (r1_scene_pad(s, 8) != R1_OK || r1_scene_count(s) != 8) return 3;\n'
                   '    if (r1_scene_commit(s, 0) != R1_ERR_STATE) return 4;   /* camera not set */\n'
                   '    r1_scene_destroy(s);\n'
                   '    return 0;\n}\n')
    exe = tmp_path / "abi"
    lib_dir = os.path.dirname(r1.LIB_PATH)
    out = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                          "-L", lib_dir, "-lrays1_b200", "-Wl,-rpath," + lib_dir], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert subprocess.run([str(exe)]).returncode == 0
