"""Host-or-device staging of the C ABI's caller buffers (include/tw3d.h: every buffer may be host or device memory). Each entry point runs with
every host/device placement of the buffers it stages; the results must be bit-identical to the all-host run, which the other GPU tests pin to the
oracle and the golden fixtures. Also: an outstanding tw_heightgen_2d_launch completes before the voxel and shadow entry points reuse the scratch."""
import ctypes as C
import itertools
import os

import numpy as np
import pytest

from cases import HM_CFG

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
S, ZV = 32, 34
ORIGINS = [(tx * S - 2 * S, ty * S + S) for ty in range(2) for tx in range(3)]


def _to_device(a):
    import torch
    return torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a).cuda()


def _key(r):
    return [None if x is None else np.asarray(x).tobytes() for x in (r if isinstance(r, tuple) else (r,))]


def _void(_):
    return None


def _placements(call, **bufs):
    """call(**buffers) for every host/device placement of the non-None buffers (fresh copies each run); the final content of every buffer and
    call's return value must equal the all-host run's, bit for bit. Returns the all-host buffers and return value."""
    import torch
    names = [k for k, v in bufs.items() if v is not None]

    def run(on_dev):
        args = {k: (None if v is None else _to_device(v.copy()) if k in on_dev else v.copy()) for k, v in bufs.items()}
        ret = call(**args)
        torch.cuda.synchronize()
        return {k: (args[k].cpu().numpy() if k in on_dev else args[k]) for k in names}, ret

    host, ret0 = run(())
    for r in range(1, len(names) + 1):
        for on_dev in itertools.combinations(names, r):
            got, ret = run(on_dev)
            for k in names:
                assert got[k].tobytes() == host[k].tobytes(), (k, on_dev)
            assert _key(ret) == _key(ret0), on_dev
    return host, ret0


def _cfg(scene, mode=1):
    return scene.SceneConfig(mesh_gen_mode=mode, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3, mesh_size=(S, S, 1))


def _tiles(scene, ctx, mode=1):
    cfg = _cfg(scene, mode)
    return ctx.heightgen_tiles(ORIGINS, cfg.mesh_size, float(cfg.dx_val), float(cfg.dy_val), ZV, cfg.height_params())


def test_heightgen_2d(tw, scene, ctx):
    cfg = _cfg(scene, 4)
    g = cfg.heightmap_grid(200, 150)
    host, mm = _placements(lambda out: ctx.heightgen_2d(g, cfg.height_params(), out=out, want_minmax=True)[1], out=np.empty((150, 200), np.float32))
    assert mm == (float(host["out"].min()), float(host["out"].max()))


@pytest.mark.parametrize("mode", [0, 1])
def test_heightgen_tiles(tw, scene, ctx, mode):
    cfg = _cfg(scene, mode)
    ctx.set_sine_params(cfg.sine_params())
    _placements(lambda out: ctx.heightgen_tiles(ORIGINS, cfg.mesh_size, float(cfg.dx_val), float(cfg.dy_val), ZV, cfg.height_params(), out=out, want_minmax=True)[1],
                out=np.empty((len(ORIGINS), ZV, ZV), np.float32))


def test_tile_weights(tw, scene, ctx):
    from test_weights_host import weight_cases
    cfg = _cfg(scene)
    ctx.set_sine_params(cfg.sine_params())
    dx, dy = float(cfg.dx_val), float(cfg.dy_val)
    tiles = _tiles(scene, ctx)
    tiles = ((tiles - np.float32(tiles.mean())) * np.float32(0.4 / float(tiles.std()))).astype(np.float32)
    rng = np.random.default_rng(3)
    wp = weight_cases(tw.WeightParams, rng, float(tiles.min()), float(tiles.max()), S, dx, dy, n=1)[0]
    hp, P = cfg.height_params(), tw._ptr
    org = np.array(ORIGINS, np.int32)

    def call(zvals, tile_params, weights, has_any_grass):
        ctx._check(tw.lib.tw_tile_weights_batch(ctx._h, P(zvals), P(org), len(ORIGINS), S, S, dx, dy, ZV, C.byref(hp), C.byref(wp), P(tile_params), P(weights), P(has_any_grass)))

    host, _ = _placements(call, zvals=tiles, tile_params=rng.uniform(-0.2, 1.3, (len(ORIGINS), 8)).astype(np.float32),
                          weights=np.zeros((len(ORIGINS), S + 1, S + 1, 4), np.uint8), has_any_grass=np.full(len(ORIGINS), 7, np.uint8))
    assert len(np.unique(host["weights"].reshape(-1, 4), axis=0)) > 10 and host["has_any_grass"].max() <= 1
    _placements(lambda zvals, tile_params, weights: call(zvals, tile_params, weights, None), zvals=tiles, tile_params=host["tile_params"],
                weights=np.zeros_like(host["weights"]))


def test_tile_bounds_normals_ao(tw, scene, ctx):
    cfg = _cfg(scene)
    dx, dy = float(cfg.dx_val), float(cfg.dy_val)
    tiles = _tiles(scene, ctx)
    _placements(lambda zvals: bytes(ctx.tile_bounds(zvals, float(np.median(tiles)), dx, dy, S)), zvals=tiles)
    _placements(lambda zvals, rgba: ctx.tile_normals(zvals, dx, dy, out=rgba)[1], zvals=tiles, rgba=np.zeros((len(ORIGINS), ZV - 1, ZV - 1, 4), np.uint8))
    host, _ = _placements(lambda zvals, ao: _void(ctx.tile_ao(zvals, ORIGINS, cfg.mesh_size, dx, dy, cfg.height_params(), 0.0625, out=ao)),
                          zvals=tiles, ao=np.zeros((len(ORIGINS), ZV - 1, ZV - 1), np.uint8))
    assert host["ao"].min() < 255


@pytest.mark.parametrize("mode", [1, 4])
def test_create_zvals_ao_batch(tw, scene, ctx, mode):
    cfg = _cfg(scene, mode)
    ep = cfg.erosion_params()
    _placements(lambda zvals, ao: ctx.create_zvals_ao_batch(ORIGINS, cfg.mesh_size, float(cfg.dx_val), float(cfg.dy_val), ZV, cfg.height_params(), 100, ep, ep.zmin,
                                                            0.0625, out=zvals, ao=ao, want_minmax=True)[2],
                zvals=np.zeros((len(ORIGINS), ZV, ZV), np.float32), ao=np.zeros((len(ORIGINS), ZV - 1, ZV - 1), np.uint8))


@pytest.mark.parametrize("mode,chunks,reorder", [(0, None, True), (1, None, True), (1, "3", True), (1, "3", False)])
def test_create_zvals_batch(tw, scene, ctx, monkeypatch, mode, chunks, reorder):
    """Sine mode (plain sequence of nested entry calls) and the pipeline: one chunk, and three chunks with and without the heaviest-first order
    (per-chunk device->host copies on the erosion streams, or one copy at the end)."""
    if chunks:
        monkeypatch.setenv("TW_PIPE_CHUNKS", chunks)
    if not reorder:
        monkeypatch.setenv("TW_PIPE_NO_REORDER", "1")
    cfg = _cfg(scene, mode)
    ctx.set_sine_params(cfg.sine_params())
    ep = cfg.erosion_params()
    host, _ = _placements(lambda out: ctx.create_zvals_batch(ORIGINS, cfg.mesh_size, float(cfg.dx_val), float(cfg.dy_val), ZV, cfg.height_params(), 100, ep, ep.zmin,
                                                             out=out, want_minmax=True)[1], out=np.zeros((len(ORIGINS), ZV, ZV), np.float32))
    assert ctx.last_erosion_steps > 0


def test_erosion_and_glaciate(tw, scene, ctx):
    cfg = _cfg(scene)
    tiles = _tiles(scene, ctx)
    zmin, zmax = float(tiles.min()), float(tiles.max())
    ep = tw.ErosionParams(1.0, zmin - 10, 0.0625, zmin - 0.1, zmax + 0.1, 0.0, 0.5)
    host, _ = _placements(lambda maps: (ctx.erode_tiles(maps, 200, ep, min_zvals=tiles.min(axis=(1, 2)), min_zval_all=zmin), ctx.last_erosion_steps)[1], maps=tiles)
    assert (host["maps"] != tiles).any()
    _placements(lambda h: (ctx.erode_parallel(h, zmin, 300, ep, num_threads=1), ctx.last_erosion_steps)[1], h=np.ascontiguousarray(tiles[0]))
    mesh = ctx.heightgen_2d(cfg.heightmap_grid(96, 64), cfg.height_params(), enable_glaciate=0)
    host, _ = _placements(lambda mesh: ctx.glaciate_mesh(mesh, 7, -20, (96, 64), cfg.height_params()), mesh=mesh)
    assert (host["mesh"] != mesh).any()


def test_eval_points_and_voxel_fill(tw, scene, ctx):
    cfg = _cfg(scene)
    xy = np.random.default_rng(5).uniform(-30.0, 30.0, (3000, 2)).astype(np.float32)
    pq = tw.PointQuery(tw.PQ_EXACT_ZVAL, 1.0, 128, 128, 4.0, 4.0, -300, 77, 0)
    _placements(lambda xy, out: _void(ctx.eval_points(xy, cfg.height_params(), pq, out=out)), xy=xy, out=np.zeros(len(xy), np.float32))
    vcfg = scene.SceneConfig(mesh_gen_mode=1, mesh_freq_filter=2, mesh_seed=3, scene_size=(16.0, 16.0, 4.0), mesh_size=(128, 128, 64), zmax_est=1.0)
    vp = scene.voxel_landscape_params(vcfg, 20, 12, 18, normalize_to_1=1)
    _placements(lambda out: _void(ctx.voxel_fill(vp, out=out)), out=np.zeros((12, 20, 18), np.float32))


def test_heightmap_passes(tw, scene, ctx):
    rng = np.random.default_rng(9)
    vals = rng.uniform(-3.0, 5.0, 5000).astype(np.float32)
    mult, add = float(np.float32((float(vals.max()) - float(vals.min())) / 255.0)), float(vals.min())
    _placements(lambda vals, out: _void(ctx.from_floats_u16(vals, mult, add, out=out)), vals=vals, out=np.zeros(2 * len(vals), np.uint8))
    data = rng.integers(0, 256, 2 * 5000, dtype=np.uint8)
    _placements(lambda data, vals: _void(ctx.to_floats_u16(data, mult, add, out=vals)), data=data, vals=np.zeros(5000, np.float32))
    _placements(lambda vals: ctx.minmax(vals), vals=vals)
    img = rng.integers(0, 256, (60, 57, 2), dtype=np.uint8)
    hs = tw.HmapSampler(57, 60, 1, 0.45, 0.0012, 1.7, -0.3, 0.8)
    _placements(lambda data16, out: _void(ctx.heightmap_sample_tiles(data16, hs, ORIGINS, ZV, out=out)), data16=img, out=np.zeros((len(ORIGINS), ZV, ZV), np.float32))
    cfg = _cfg(scene)
    hp, ep = cfg.height_params(), cfg.erosion_params()

    def info(i):
        return (i.min_z, i.max_z, i.val_mult, i.val_add, i.mesh_file_scale, i.mesh_file_tz, i.erosion_moves)
    host, ret = _placements(lambda data16, vals: info(ctx.proc_gen_heightmap(70, 50, float(cfg.dx_val), float(cfg.dy_val), hp, 300, ep, data16=data16, vals=vals)[1]),
                            data16=np.zeros(2 * 70 * 50, np.uint8), vals=np.zeros((50, 70), np.float32))
    host2, ret2 = _placements(lambda data16: info(ctx.proc_gen_heightmap(70, 50, float(cfg.dx_val), float(cfg.dy_val), hp, 300, ep, data16=data16)[1]),
                              data16=np.zeros(2 * 70 * 50, np.uint8))
    assert ret2 == ret and host2["data16"].tobytes() == host["data16"].tobytes() and ret[-1] > 0


def _voxel_case(tw):
    rng = np.random.default_rng(1)
    nx, ny, nz = 24, 20, 18
    f = rng.standard_normal((ny, nx, nz)).astype(np.float32)
    for ax in range(3):
        f = (f + np.roll(f, 1, ax) + np.roll(f, -1, ax)) / 3
    vpp = tw.VoxelPostParams()
    vpp.nx, vpp.ny, vpp.nz = nx, ny, nz
    for d in range(3):
        vpp.lo_pos[d], vpp.vsz[d] = (-1.0, 0.5, 0.25)[d], (0.05, 0.07, 0.04)[d]
    vpp.make_closed_surface, vpp.remove_unconnected, vpp.centre_seed = 1, 3, 0
    zix = rng.integers(0, nz // 2, (ny, nx)).astype(np.uint32)
    g = np.load(os.path.join(GOLD, "voxel_post.npz"))
    return np.ascontiguousarray(f * 3, np.float32), vpp, zix, (g["edge_table"].astype(np.uint32), g["tri_table"].astype(np.int32), g["edge_to_vals"].astype(np.uint32))


def test_voxel_post(tw, ctx):
    vals, vpp, zix, (et, tt, ev) = _voxel_case(tw)
    host, _ = _placements(lambda vals, zix_xy, outside: _void(ctx.voxel_outside(vals, vpp, zix_xy, out=outside)), vals=vals, zix_xy=zix, outside=np.zeros(vals.shape, np.uint8))
    outside = host["outside"]
    host, changed = _placements(lambda vals, outside: ctx.voxel_remove_unconnected(vals, outside, vpp), vals=vals, outside=outside)
    assert changed > 0
    v2, o2 = host["vals"], host["outside"]
    ntris = len(ctx.voxel_triangles(v2, o2, vpp, (et, tt, ev)))
    assert ntris > 100
    P, n = tw._ptr, C.c_uint64()

    def call(vals, outside, edge_table, tri_table, edge_to_vals, tris):
        ctx._check(tw.lib.tw_voxel_triangles(ctx._h, P(vals), P(outside), C.byref(vpp), P(edge_table), P(tri_table), P(edge_to_vals), P(tris), ntris, C.byref(n)))
        return n.value
    _placements(call, vals=v2, outside=o2, edge_table=et, tri_table=tt, edge_to_vals=ev, tris=np.zeros((ntris, 3, 3), np.float32))


def _shadow_case(tw, scene, ctx):
    from test_gpu_shadows import _params
    cfg = scene.SceneConfig(mesh_gen_mode=1, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.0, mesh_size=(17, 17, 1))
    txy = np.array([(tx - 1, ty + 3) for ty in range(3) for tx in range(3)], np.int32)
    tiles = ctx.heightgen_tiles([(tx * 17, ty * 17) for tx, ty in txy], cfg.mesh_size, float(cfg.dx_val), float(cfg.dy_val), 19, cfg.height_params())
    tiles = ((tiles - np.float32(tiles.mean())) * np.float32(3.0)).astype(np.float32)
    return tiles, txy, _params(tw, cfg, 17, float(tiles.min()) - 0.5, float(tiles.max()) + 0.5, (3.0, 2.0, 0.4))


def _shadow_call(tw, ctx, txy, sp):
    P = tw._ptr

    def call(zvals, smask, sh_out_x, sh_out_y):
        ctx._check(tw.lib.tw_tile_shadows_batch(ctx._h, P(zvals), P(txy), len(txy), zvals.shape[1], C.byref(sp), P(smask), P(sh_out_x), P(sh_out_y)))
    return call


def test_tile_shadows(tw, scene, ctx):
    tiles, txy, sp = _shadow_case(tw, scene, ctx)
    nt, zv = tiles.shape[0], tiles.shape[1]
    host, _ = _placements(_shadow_call(tw, ctx, txy, sp), zvals=tiles, smask=np.zeros(tiles.shape, np.uint8),
                          sh_out_x=np.zeros((nt, zv), np.float32), sh_out_y=np.zeros((nt, zv), np.float32))
    assert 0 < (host["smask"] == 2).mean() < 1


def test_pending_launch_completes_before_voxel_and_shadow_calls(tw, scene, ctx):
    """tw_heightgen_2d_launch with a page-locked host output stages the grid in scratch slot 0 and copies it out band by band after the call returns;
    the voxel and shadow entry points stage their host buffers in the same slot, so they must complete the launch first."""
    import torch
    cfg = _cfg(scene, 4)
    g, hp = cfg.heightmap_grid(1536, 1024), cfg.height_params()
    exp, exp_mm = ctx.heightgen_2d(g, hp, want_minmax=True)
    vals, vpp, zix, tables = _voxel_case(tw)
    outside = ctx.voxel_outside(vals, vpp, zix)
    tiles, txy, sp = _shadow_case(tw, scene, ctx)

    def remove_unconnected():
        v, o = vals.copy(), outside.copy()
        return v, o, ctx.voxel_remove_unconnected(v, o, vpp)

    def shadows():
        m, ox, oy = np.zeros(tiles.shape, np.uint8), np.zeros(tiles.shape[:2], np.float32), np.zeros(tiles.shape[:2], np.float32)
        _shadow_call(tw, ctx, txy, sp)(tiles, m, ox, oy)
        return m, ox, oy
    calls = [lambda: (ctx.voxel_outside(vals, vpp, zix),), remove_unconnected, lambda: (ctx.voxel_triangles(vals, outside, vpp, tables),), shadows]
    for call in calls:
        want = call()
        out = torch.empty((g.ny, g.nx), dtype=torch.float32, pin_memory=True)
        mm = tw.MinMax()
        ctx.heightgen_2d_launch(g, hp, 1, 0, out, mm)
        got = call()
        assert ctx.heightgen_2d_poll(wait=True)
        assert out.numpy().tobytes() == exp.tobytes() and (mm.zmin, mm.zmax) == exp_mm
        assert _key(got) == _key(want)
