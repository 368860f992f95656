"""GPU parity: tw_heightgen_2d / tw_heightgen_tiles (CUDA, through the C ABI) vs the CPU oracle - bit-exact for every gen mode."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from cases import convert, height_cases, HM_CFG
from test_oracle_golden import hp_from_args

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _run_case(tw, scene, oracle, ctx, kw, org, size, sp_cache={}):
    cfg = scene.SceneConfig(**kw)
    hp = cfg.height_params()
    key = (cfg.mesh_seed, cfg.mesh_gen_mode)
    if key not in sp_cache:
        sp_cache[key] = cfg.sine_params()
    sp = sp_cache[key]
    x0, y0, dxm = org
    g = tw.Grid2D(x0, y0, float(cfg.dx_val) * dxm, float(cfg.dy_val) * dxm, size[0], size[1])
    ctx.set_sine_params(sp)
    z_gpu, mm = ctx.heightgen_2d(g, hp, enable_glaciate=1, want_minmax=True)
    z_cpu = oracle.heightgen_2d(convert(g, oracle.Grid2D), convert(hp, oracle.HeightParams), sp, 1, 0)
    return z_gpu, z_cpu, mm


@pytest.mark.parametrize("name,kw,org,size", height_cases(), ids=[c[0] for c in height_cases()])
def test_heightgen_bit_exact(tw, scene, oracle, ctx, beq, name, kw, org, size):
    z_gpu, z_cpu, mm = _run_case(tw, scene, oracle, ctx, kw, org, size)
    assert beq(z_gpu, z_cpu) == 0, "max abs diff %g" % np.abs(z_gpu - z_cpu).max()
    assert mm[0] == z_cpu.min() and mm[1] == z_cpu.max()   # fused min/max reduction


def test_sine_min_start_sin_and_no_glaciate(tw, scene, oracle, ctx, beq):
    cfg = scene.SceneConfig(mesh_gen_mode=0, mesh_freq_filter=0, mesh_seed=6, hmap=HM_CFG, zmax_est=1.5)
    hp, sp = cfg.height_params(), cfg.sine_params()
    ctx.set_sine_params(sp)
    for nx, ny, x0 in ((1, 1, -7.0), (3, 200, -7.0), (257, 65, -7.0), (64, 64, -7.0), (96, 40, 4.0e6)):
        # x0 = 4e6: SINF's int(sscale*v) index overflows int; the reference (x86 cvttss2si) then uses INT_MIN & 32767 = 0 - reproduced on the GPU
        g = tw.Grid2D(x0, 11.0, float(cfg.dx_val), float(cfg.dy_val), nx, ny)
        for mss in (0, 50, 20):
            for gl in (0, 1):
                zg = ctx.heightgen_2d(g, hp, enable_glaciate=gl, min_start_sin=mss)
                zc = oracle.heightgen_2d(convert(g, oracle.Grid2D), convert(hp, oracle.HeightParams), sp, gl, mss)
                assert beq(zg, zc) == 0


def test_custom_glaciate_exp_within_tolerance(tw, scene, oracle, ctx):
    # pow(relh, custom) uses CUDA powf vs glibc powf: not bit-exact by construction; north_star tolerance 1e-5 relative per cell
    cfg = scene.SceneConfig(mesh_gen_mode=1, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=8.0, custom_glaciate_exp=2.5)
    hp = cfg.height_params()
    g = tw.Grid2D(-64, -64, float(cfg.dx_val), float(cfg.dy_val), 128, 128)
    zg = ctx.heightgen_2d(g, hp)
    zc = oracle.heightgen_2d(convert(g, oracle.Grid2D), convert(hp, oracle.HeightParams), None, 1, 0)
    assert np.array_equal(np.isnan(zg), np.isnan(zc))      # pow(negative relh, 2.5) is NaN on both sides
    ok = ~np.isnan(zc)
    assert ok.mean() > 0.5
    assert np.all(np.abs(zg - zc)[ok] <= 1e-5 * np.maximum(np.abs(zg), np.abs(zc))[ok] + 1e-5 * cfg.zmax_est)


def test_device_pointer_output_and_async(tw, scene, oracle, ctx, beq):
    import torch
    cfg = scene.SceneConfig(mesh_gen_mode=4, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3)
    hp = cfg.height_params()
    g = cfg.heightmap_grid(96, 80)
    out = torch.empty((80, 96), dtype=torch.float32, device="cuda")
    mm = tw.MinMax()
    ctx.heightgen_2d_launch(g, hp, 1, 0, out, mm)      # mirrors build_arrays(no_wait=1) ...
    while not ctx.heightgen_2d_poll(wait=False):        # ... and the next-frame collection
        pass
    zc = oracle.heightgen_2d(convert(g, oracle.Grid2D), convert(hp, oracle.HeightParams), None, 1, 0)
    assert beq(out.cpu().numpy(), zc) == 0
    assert mm.zmin == zc.min() and mm.zmax == zc.max()


@pytest.mark.parametrize("mode", [0, 1, 4])
def test_tiles_match_per_tile_calls(tw, scene, oracle, ctx, beq, mode):
    # tile_t::create_zvals height fill for a 3x2 block of tiles, zvsize = size+2 (src/tiled_mesh.cpp:302,458-464)
    cfg = scene.SceneConfig(mesh_gen_mode=mode, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3, mesh_size=(64, 64, 1))
    hp, sp = cfg.height_params(), cfg.sine_params()
    ctx.set_sine_params(sp)
    S, zv = 64, 66
    origins = [(tx * S - 7 * S, ty * S + 3 * S) for ty in range(2) for tx in range(3)]
    tiles, mm = ctx.heightgen_tiles(origins, cfg.mesh_size, float(cfg.dx_val), float(cfg.dy_val), zv, hp, want_minmax=True)
    for t, (x1, y1) in enumerate(origins):
        g = oracle.Grid2D(float(x1 - S // 2), float(y1 - S // 2), float(cfg.dx_val), float(cfg.dy_val), zv, zv)
        zc = oracle.heightgen_2d(g, convert(hp, oracle.HeightParams), sp, 1, 0)
        assert beq(tiles[t], zc) == 0
        assert mm[t, 0] == zc.min() and mm[t, 1] == zc.max()
    if mode != 0:
        # neighbouring tiles overlap by 2 cells and agree exactly there: with a power-of-two DX the cell coordinate (x*mdx + mx0) is exact,
        # so the noise modes are pure functions of the global coordinate (the sine tables fold the origin into x_const, which rounds per tile)
        assert np.array_equal(tiles[0][:, S:S + 2], tiles[1][:, 0:2])


def test_full_size_properties(tw, scene, oracle, ctx, beq):
    """BASELINE config 2 at full size (8192^2, 8-octave domain warp): size-independent checks - a row band recomputed as its own grid
    is bit-identical (pure function of global coordinates), an oracle-sized window matches the oracle, min/max equal a separate reduction."""
    import torch
    cfg = scene.SceneConfig(mesh_gen_mode=4, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3)
    hp = cfg.height_params()
    N = 8192
    g = cfg.heightmap_grid(N, N)
    out = torch.empty((N, N), dtype=torch.float32, device="cuda")
    _, mm = ctx.heightgen_2d(g, hp, out=out, want_minmax=True)
    assert torch.isfinite(out).all()
    assert mm == (out.min().item(), out.max().item())
    assert mm == ctx.minmax(out)
    y0, rows = 5000, 64
    gb = tw.Grid2D(g.x0, g.y0 + y0, g.dx, g.dy, N, rows)
    band = ctx.heightgen_2d(gb, hp)
    assert beq(band, out[y0:y0 + rows].cpu().numpy()) == 0
    gw = oracle.Grid2D(g.x0 + 4000, g.y0 + 6000, g.dx, g.dy, 96, 64)
    zc = oracle.heightgen_2d(gw, convert(hp, oracle.HeightParams), None, 1, 0)
    assert beq(out[6000:6064, 4000:4096].cpu().numpy(), zc) == 0


def _bench_kernel_only(steps, dump_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--kernel-only",
                        "--dump-outputs", str(dump_dir)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_bench_dump_outputs(tw, scene, oracle, ctx, beq, tmp_path):
    """bench.py --dump-outputs writes the headline grid's rows (== the oracle, bit for bit) and its min/max, float32, within 64 MB; --steps sets the
    number of timed steps (the launches in the timed region scale with it) and does not change what is written."""
    d2, d3 = tmp_path / "steps2", tmp_path / "steps3"
    r2, r3 = _bench_kernel_only(2, d2), _bench_kernel_only(3, d3)
    assert r2["gpu_launches"] > 0 and 3 * r2["gpu_launches"] == 2 * r3["gpu_launches"], (r2["gpu_launches"], r3["gpu_launches"])
    assert sorted(os.listdir(d2)) == sorted(os.listdir(d3)) == ["height_rows.npy", "minmax.npy"]
    for name in os.listdir(d2):
        assert np.load(d2 / name).tobytes() == np.load(d3 / name).tobytes(), name
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rows, mm = np.load(d2 / "height_rows.npy"), np.load(d2 / "minmax.npy")
    assert sum(f.stat().st_size for f in d2.iterdir()) <= 64 << 20
    assert rows.dtype == mm.dtype == np.float32 and rows.shape == (bench.DUMP_ROWS, bench.N_TILE) and mm.shape == (2,)
    assert mm[0] <= rows.min() and rows.max() <= mm[1]
    cfg = scene.SceneConfig(mesh_gen_mode=4, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3)
    hp = convert(cfg.height_params(), oracle.HeightParams)
    g = cfg.heightmap_grid(bench.N_TILE, bench.N_TILE)
    idx = bench.dump_rows()
    for i in (0, len(idx) // 2, len(idx) - 1):
        zc = oracle.heightgen_2d(oracle.Grid2D(g.x0, g.y0 + int(idx[i]), g.dx, g.dy, bench.N_TILE, 1), hp, None, 1, 0)
        assert beq(rows[i], zc) == 0, int(idx[i])


def test_matches_linked_reference(tw, scene, ctx, beq, request):
    """Directly against the unmodified reference: its linked objects (oracle/_ref) when they are built, otherwise the height grids it produced for
    tests/golden/height.npz (every gen mode and shape, tests/golden/make_golden.py)."""
    import refapi
    if not refapi.available():
        h = np.load(os.path.join(GOLD, "height.npz"))
        for mode in range(5):
            for shape in range(3):
                n = "h_m%d_s%d" % (mode, shape)
                a = h[n + "_args"]
                if mode == 0:
                    ctx.set_sine_params(h[n + "_sp"])
                g = tw.Grid2D(float(a[4]), float(a[5]), 0.0625, 0.0625, int(a[6]), int(a[7]))
                assert beq(ctx.heightgen_2d(g, hp_from_args(tw, a, h[n + "_hmap"])), h[n]) == 0, n
        return
    ref = request.getfixturevalue("ref")
    for mode in (0, 1, 2, 4):
        ref.setup(mode=mode, freq_filter=1, seed=1, zmax_est=2.3, hmap=HM_CFG)
        cfg = scene.SceneConfig(mesh_gen_mode=mode, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3)
        hp = cfg.height_params()
        sp = ref.sine_params()
        ctx.set_sine_params(sp)
        n = 80
        zr = ref.heightgen(-n / 2, -n / 2, float(cfg.dx_val), float(cfg.dy_val), n, n, cache_values=0, glaciate=1)
        zg = ctx.heightgen_2d(tw.Grid2D(-n / 2, -n / 2, float(cfg.dx_val), float(cfg.dy_val), n, n), hp)
        assert beq(zg, zr) == 0
