"""-m gpu parity on textured / alpha / volume scenes, ray-level and BSDF-level checks."""
import numpy as np
import pytest

from conftest import rel_rmse

pytestmark = pytest.mark.gpu


def _attach(scene, env, size, tile=None, **kw):
    from vk_gltf_renderer_b200.renderer import PathTracer, Resources
    res = Resources(scene=scene, hdr_rgb=env, camera=scene.camera, size=size, tile=tile)
    pt = PathTracer(0)
    for k, v in kw.items():
        setattr(pt, k, v)
    pt.onAttach(res)
    return pt, res


def _oracle(oracle_mod, scene, env):
    o = oracle_mod.Oracle()
    o.set_scene(scene)
    o.set_environment(env)
    return o


def _gpu_render(scene, env, w, h, frames, **kw):
    from vk_gltf_renderer_b200.renderer import render_headless, Resources
    res = Resources(scene=scene, hdr_rgb=env, camera=scene.camera, size=(w, h))
    return render_headless(res, frames, **kw)


def test_bsdf_parity(oracle_mod):
    """bsdfEvaluate / bsdfSample: CUDA vs oracle on 200k random materials x directions.
    fp32 tolerance: 2e-4 relative on values; event types and the chosen lobe must agree except on
    measure-zero threshold crossings (<= 0.01 % of records)."""
    import torch
    from vk_gltf_renderer_b200 import bsdf_io
    from vk_gltf_renderer_b200.renderer import PathTracer, Resources
    pt = PathTracer(0)
    pt.onAttach(Resources(size=(8, 8)))
    o = oracle_mod.Oracle()
    rec = bsdf_io.random_records(200000)
    d_in = torch.from_numpy(rec).cuda()
    d_out = torch.empty((len(rec), 8), dtype=torch.float32, device="cuda")
    pt.bsdf_eval(d_in.data_ptr(), len(rec), d_out.data_ptr())
    pt.synchronize()
    got, ref = d_out.cpu().numpy(), o.bsdf_eval(rec)
    assert np.isfinite(got).all() and np.isfinite(ref).all()
    bad = ~np.isclose(got, ref, rtol=2e-4, atol=1e-6).all(axis=1)
    assert bad.mean() <= 1e-4, f"eval mismatches: {bad.sum()}"
    assert (ref[:, 6] > 0).mean() > 0.2
    pt.bsdf_sample(d_in.data_ptr(), len(rec), d_out.data_ptr())
    pt.synchronize()
    got, ref = d_out.cpu().numpy(), o.bsdf_sample(rec)
    ev_ok = got[:, 7] == ref[:, 7]
    assert (~ev_ok).mean() <= 1e-4
    live = ev_ok & (ref[:, 7] != 0)
    bad = ~np.isclose(got[live][:, :7], ref[live][:, :7], rtol=5e-4, atol=2e-6).all(axis=1)
    assert bad.mean() <= 1e-3, f"sample mismatches: {bad.sum()} of {live.sum()}"
    assert len(set(ref[:, 7].astype(int).tolist())) >= 4  # absorb, diffuse/glossy reflection, transmission


def test_trace_parity_soup_and_alpha(std_env, oracle_mod):
    """Closest-hit + shadow parity on a 20k-triangle soup (culling on) and on the alpha-masked atrium
    (stochastic any-hit with per-ray seeds): ids and (t,u,v) bit-exact, seeds advance identically."""
    import torch
    from gpu_util import random_rays, to_dev
    from vk_gltf_renderer_b200 import synth
    for scn, lo, hi in ((synth.triangle_soup(20000), [-1, -1, -1], [1, 1, 1]),
                        (synth.synth_sponza(tex_size=128, detail=0.05), [-15, 0, -6], [15, 12, 6])):
        pt, _ = _attach(scn, std_env, (16, 16))
        o = oracle_mod.Oracle()
        o.set_scene(scn)
        rays = random_rays(60000, lo, hi)
        seeds = ((np.arange(len(rays), dtype=np.uint64) * 2654435761) % (2 ** 32)).astype(np.uint32)
        s_ref = seeds.copy()
        ref = o.trace_closest(rays, s_ref)
        d_rays, d_seeds = to_dev(rays), to_dev(seeds.copy())
        d_hits = torch.empty((len(rays), 6), dtype=torch.float32, device="cuda")
        pt.trace_closest(d_rays.data_ptr(), len(rays), d_hits.data_ptr(), d_seeds.data_ptr())
        pt.synchronize()
        got = d_hits.cpu().numpy()
        assert np.array_equal(got.view(np.uint32)[:, 1:4], ref.view(np.uint32)[:, 1:4])
        assert np.array_equal(got[:, [0, 4, 5]], ref[:, [0, 4, 5]])
        assert np.array_equal(d_seeds.cpu().numpy(), s_ref)
        # shadow rays: bounded segments
        rays_s = rays.copy()
        rays_s[:, 7] = 4.0
        s_ref = seeds.copy()
        ref_t = o.trace_shadow(rays_s, s_ref)
        d_rays, d_seeds = to_dev(rays_s), to_dev(seeds.copy())
        d_t = torch.empty((len(rays), 3), dtype=torch.float32, device="cuda")
        pt.trace_shadow(d_rays.data_ptr(), len(rays), d_t.data_ptr(), d_seeds.data_ptr())
        pt.synchronize()
        assert np.array_equal(d_t.cpu().numpy(), ref_t)
        assert 0.02 < (ref_t[:, 0] > 0).mean() < 0.98


def test_render_parity_synth_sponza_small(std_env, oracle_mod):
    """Textured multi-material atrium with MASK foliage, 25 materials, depth 6, 8 frames:
    rel RMSE <= 1e-3 vs the oracle (hardware bilinear/trilinear weights are 8-bit, the oracle's fp32)."""
    from vk_gltf_renderer_b200 import synth
    scn = synth.synth_sponza(tex_size=256, detail=0.05)
    o = _oracle(oracle_mod, scn, std_env)
    ref = oracle_mod.render(o, scn.camera, 320, 180, 8, max_depth=6)
    pt, img = _gpu_render(scn, std_env, 320, 180, 8, ptMaxDepth=6)
    assert np.isfinite(img).all()
    e = rel_rmse(img, ref)
    print("synth sponza rel RMSE", e)
    assert e <= 1e-3


def test_render_parity_shader_ball(shader_ball_scene, std_env, oracle_mod):
    o = _oracle(oracle_mod, shader_ball_scene, std_env)
    ref = oracle_mod.render(o, shader_ball_scene.camera, 160, 120, 8, max_depth=5)
    pt, img = _gpu_render(shader_ball_scene, std_env, 160, 120, 8, ptMaxDepth=5)
    e = rel_rmse(img, ref)
    print("shader ball rel RMSE", e)
    assert e <= 1e-3


def test_render_parity_glass_volume(std_env, oracle_mod):
    """Transmission + volume absorption (Beer), IOR swap inside, coloured shadow transmission through the
    any-hit tree: stream-replicated parity, rel RMSE <= 1e-3."""
    from vk_gltf_renderer_b200 import synth
    scn = synth.synth_glass(n=48, scatter=False)
    o = _oracle(oracle_mod, scn, std_env)
    ref = oracle_mod.render(o, scn.camera, 128, 128, 8, max_depth=12)
    pt, img = _gpu_render(scn, std_env, 128, 128, 8, ptMaxDepth=12)
    assert np.isfinite(img).all()
    e = rel_rmse(img, ref)
    print("glass rel RMSE", e)
    assert e <= 1e-3


def test_render_parity_glass_volume_scatter_statistical(std_env, oracle_mod):
    """KHR_materials_volume_scatter: in-volume random walks (up to 64+ scatters, NEE inside the medium).
    Paths with ~100 chaotic events amplify 1e-7 libm differences to O(1), so per-pixel stream parity is
    not attainable by ANY two fp32 implementations; SURVEY.md section 8d's fallback protocol applies:
    (1) the two estimators must agree exactly on the early part of every path => the median per-pixel
    relative difference stays tiny, (2) no bias: image-mean radiance within 1 %, 16x16-tile means within
    5 sigma of the sampling error, (3) identical ray budgets within 0.5 %."""
    from vk_gltf_renderer_b200 import synth
    scn = synth.synth_glass(n=48, scatter=True)
    o = _oracle(oracle_mod, scn, std_env)
    frames = 16
    ref = oracle_mod.render(o, scn.camera, 128, 128, frames, max_depth=12)
    pt, img = _gpu_render(scn, std_env, 128, 128, frames, ptMaxDepth=12)
    assert np.isfinite(img).all()
    rel = np.abs(img[..., :3] - ref[..., :3]).sum(-1) / np.maximum(ref[..., :3].sum(-1), 1e-3)
    print("glass scatter: median rel diff", np.median(rel), "mean ratio", img[..., :3].mean() / ref[..., :3].mean())
    assert np.median(rel) <= 1e-4
    assert abs(img[..., :3].mean() / ref[..., :3].mean() - 1.0) <= 1e-2
    lum_g = img[..., :3].mean(-1).reshape(8, 16, 8, 16).mean((1, 3))
    lum_r = ref[..., :3].mean(-1).reshape(8, 16, 8, 16).mean((1, 3))
    sig = ref[..., :3].mean(-1).reshape(8, 16, 8, 16).std((1, 3)) / 16.0 + 1e-4
    assert (np.abs(lum_g - lum_r) <= 5.0 * sig + 1e-2 * lum_r).all()
    st, so = pt.stats(), o.stats()
    assert abs(st["closestRays"] / so["closestRays"] - 1.0) <= 5e-3
    assert abs(st["shadowRays"] / so["shadowRays"] - 1.0) <= 5e-3


def test_multisample_frames_and_tiling(box_scene, std_env, oracle_mod):
    """ptSamples > 1 continues one RNG stream per pixel (path regeneration); a row tile renders the
    same pixels as the full frame (seeds use global coordinates)."""
    o = _oracle(oracle_mod, box_scene, std_env)
    ref = oracle_mod.render(o, box_scene.camera, 96, 64, 3, max_depth=5, num_samples=4)
    pt, img = _gpu_render(box_scene, std_env, 96, 64, 3, ptMaxDepth=5, ptSamples=4)
    assert rel_rmse(img, ref) <= 1e-3
    assert np.array_equal(img[..., 3], ref[..., 3])
    from vk_gltf_renderer_b200.renderer import render_headless, Resources
    res = Resources(scene=box_scene, hdr_rgb=std_env, camera=box_scene.camera, size=(96, 64), tile=(16, 24))
    pt2, tile = render_headless(res, 3, ptMaxDepth=5, ptSamples=4)
    assert tile.shape == (24, 96, 4)
    assert np.array_equal(tile, img[16:40])
    # interleaved bands (multi-GPU load balancing): rank r of 2 owns every other band of 4 rows
    from vk_gltf_renderer_b200 import tiling
    parts = []
    for r in range(2):
        res = Resources(scene=box_scene, hdr_rgb=std_env, camera=box_scene.camera, size=(96, 64), tile=("interleave", 4, 2, r))
        _, t = render_headless(res, 3, ptMaxDepth=5, ptSamples=4)
        assert np.array_equal(t, img[tiling.interleaved_rows(64, 2, r, 4)])
        parts.append(t)
    assert np.array_equal(tiling.deinterleave(np.concatenate(parts), 64, 2, 4), img)
    res = Resources(scene=box_scene, hdr_rgb=std_env, camera=box_scene.camera, size=(96, 64), tile=("interleave", 5, 2, 0))
    with pytest.raises(Exception):
        render_headless(res, 1)


def test_unsupported_paths_fail_loudly(box_scene, std_env):
    from vk_gltf_renderer_b200.renderer import B200PTError, PathTracer, Resources
    res = Resources(scene=box_scene, hdr_rgb=std_env, camera=box_scene.camera, size=(32, 32))
    res.settings.envSystem = 0  # physical sky: not built
    pt = PathTracer(0)
    pt.onAttach(res)
    res.frameCount = 0
    with pytest.raises(B200PTError):
        pt.onRender(None, res)
    res.settings.envSystem, res.settings.hdrBlur = 1, 0.5   # blurred HDR backplate (smoothHDRBlur, nvshaders): not built, not ignored
    with pytest.raises(B200PTError):
        pt.onRender(None, res)
    res.settings.hdrBlur = 0.0
    pt.onRender(None, res)


def test_frames_in_flight_and_async_readback(box_scene, std_env):
    """Overlapping frames (lanes) accumulate in frame order: 1, 2 and 3 frames in flight give the same bits, and
    the pipelined read-back returns the image as of the frame it was issued after."""
    import ctypes as C
    from vk_gltf_renderer_b200.renderer import PathTracer, Resources
    imgs = []
    for lanes in (1, 2, 3):
        res = Resources(scene=box_scene, hdr_rgb=std_env, camera=box_scene.camera, size=(80, 48))
        pt = PathTracer(0)
        pt.ptMaxDepth = 6
        pt.onAttach(res)
        pt.set_frames_in_flight(lanes)
        bufs = [np.zeros((48, 80, 4), np.float32) for _ in range(2)]
        snaps = []
        for f in range(7):
            res.frameCount = f
            pt.onRender(None, res)
            pt.read_accum_async(bufs[f & 1].ctypes.data_as(C.c_void_p), bufs[f & 1].size, f & 1)
            if f > 0:
                pt.wait_read((f - 1) & 1)
                snaps.append(bufs[(f - 1) & 1].copy())
        pt.wait_read(6 & 1)
        snaps.append(bufs[6 & 1].copy())
        final = pt.read_accum()
        assert np.array_equal(final, snaps[-1])
        imgs.append(snaps)
        pt.onDetach(res)
    for k in range(7):
        assert np.array_equal(imgs[0][k], imgs[1][k]) and np.array_equal(imgs[0][k], imgs[2][k])
    assert not np.array_equal(imgs[0][0], imgs[0][6])


@pytest.mark.parametrize("kind", ["mask", "blend", "tinted"])
def test_render_parity_deep_anyhit_layers(std_env, oracle_mod, kind):
    """14 non-opaque layers on every ray: more candidates than one any-hit walk collects, so the continuation
    round and the final in-kernel fallback run for camera rays and for shadow rays (stochastic alpha for MASK /
    BLEND, coloured transmission for the tinted sheets).  Same bits of randomness as the oracle, candidate by
    candidate: rel RMSE <= 1e-3."""
    from vk_gltf_renderer_b200 import synth
    scn = synth.synth_layers(blend=(kind == "blend"), tinted=(kind == "tinted"))
    o = _oracle(oracle_mod, scn, std_env)
    ref = oracle_mod.render(o, scn.camera, 160, 120, 4, max_depth=5)
    pt, img = _gpu_render(scn, std_env, 160, 120, 4, ptMaxDepth=5)
    assert np.isfinite(img).all()
    e = rel_rmse(img, ref)
    print("layers", kind, "rel RMSE", e)
    assert e <= 1e-3


def test_cpp_host_headless_matches_python_host(box_scene, std_env, tmp_path):
    """The C++ host mirror (host/b200pt_host.cpp: SceneData, Resources, PathTracer : BaseRenderer) driven by
    b200pt_headless renders the image the Python mirror renders (camera matrices are computed independently in
    double on both sides, so agreement is to rounding of the 396-byte frame constants, not bit-for-bit) and prints
    the reference's HEADLESS_SUMMARY / BENCHMARK_JSON records."""
    import json
    import os
    import subprocess
    from vk_gltf_renderer_b200 import _lib
    exe = os.path.join(os.path.dirname(_lib.LIB_PATH), "b200pt_headless")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    blob, raw = str(tmp_path / "box.b2sc"), str(tmp_path / "box.raw")
    box_scene.save_blob(blob, std_env)
    out = subprocess.run([exe, "--scene", blob, "--size", "96", "64", "--frames", "4", "--ptMaxDepth", "5", "--ptSamples", "2",
                          "--outRaw", raw, "--out", str(tmp_path / "box.pfm")], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    summary = [l for l in out.stdout.splitlines() if l.startswith("HEADLESS_SUMMARY ")]
    record = [l for l in out.stdout.splitlines() if l.startswith("BENCHMARK_JSON ")]
    assert len(summary) == 1 and "ptSamples=2" in summary[0] and "resolution=96x64" in summary[0] and "effective_spp=8" in summary[0]
    rec = json.loads(record[0][len("BENCHMARK_JSON "):])
    assert rec["type"] == "headless_summary" and rec["frames"] == 4 and rec["measured_frames"] == 3 and rec["closest_rays"] > 0
    img = np.fromfile(raw, np.float32).reshape(64, 96, 4)
    _, ref = _gpu_render(box_scene, std_env, 96, 64, 4, ptMaxDepth=5, ptSamples=2)
    assert np.array_equal(img[..., 3], ref[..., 3])
    assert rel_rmse(img, ref) <= 1e-4
    assert os.path.getsize(tmp_path / "box.pfm") > 96 * 64 * 12


HARNESS_KEYS = ("frames", "maxFrames", "ptSamples", "effective_spp", "measured_effective_spp", "resolution_w", "resolution_h", "wall_ms", "ms_per_frame",
                "total_wall_ms", "total_ms_per_frame", "warmup_frames", "measured_frames", "throughput_MSps", "spp_per_sec")


def test_headless_accepts_the_reference_harness_command_line(box_scene, std_env, tmp_path):
    """The exact argument list utils/benchmark/benchmark_runner.py:164-198 spawns (--headless --size W H --frames N --maxFrames N
    --ptSamples S --ptAdaptiveSampling 0 --renderSystem 0 --envSystem 1 --scenefile X.glb --hdrfile Y.hdr): the .glb and .hdr are
    loaded directly, the first BENCHMARK_JSON record with "schema":1 is the headless_summary carrying every key the reference's
    parser reads (utils/benchmark/benchmark_results.py:147-170), frame 1 is warm-up (src/benchmarking.hpp:128), and the image is
    the one the Python host renders from the same files.  The log is kept under gpurun_out/ for the CPU-side parser test."""
    import json
    import os
    import shutil
    import subprocess
    from vk_gltf_renderer_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(os.path.dirname(_lib.LIB_PATH), "b200pt_headless")
    raw = str(tmp_path / "box.raw")
    cmd = [exe, "--headless", "--size", "96", "64", "--frames", "6", "--maxFrames", "6", "--ptSamples", "2", "--ptAdaptiveSampling", "0", "--renderSystem", "0",
           "--envSystem", "1", "--scenefile", os.path.join(root, "tests", "assets", "Box.glb"), "--hdrfile", os.path.join(root, "tests", "assets", "std_env.hdr"),
           "--ptMaxDepth", "5", "--outRaw", raw]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert out.returncode == 0, out.stdout
    recs = [json.loads(l[l.find("BENCHMARK_JSON ") + 15:]) for l in out.stdout.splitlines() if "BENCHMARK_JSON " in l]
    recs = [r for r in recs if r.get("schema") == 1]
    summary = [r for r in recs if r["type"] == "headless_summary"][0]
    assert all(k in summary for k in HARNESS_KEYS)
    # the same keys as the record of tests/golden/headless_box_harness.log, which the reference's parser was run on
    golden = json.load(open(os.path.join(root, "tests", "golden", "headless_box_harness_parsed.json")))["benchmark_records"][-1]
    assert set(golden) == set(summary)
    assert summary["frames"] == 6 and summary["maxFrames"] == 6 and summary["ptSamples"] == 2 and summary["effective_spp"] == 12
    assert summary["warmup_frames"] == 1 and summary["measured_frames"] == 5 and summary["measured_effective_spp"] == 10
    assert summary["resolution_w"] == 96 and summary["resolution_h"] == 64 and summary["throughput_MSps"] > 0
    assert any(l.startswith("HEADLESS_SUMMARY ") for l in out.stdout.splitlines())
    img = np.fromfile(raw, np.float32).reshape(64, 96, 4)
    _, ref = _gpu_render(box_scene, std_env, 96, 64, 6, ptMaxDepth=5, ptSamples=2)
    assert np.array_equal(img[..., 3], ref[..., 3]) and rel_rmse(img, ref) <= 1e-4
    os.makedirs(os.path.join(root, "gpurun_out"), exist_ok=True)
    with open(os.path.join(root, "gpurun_out", "headless_box_harness.log"), "w") as f:
        f.write(out.stdout)
    # flags of the reference app that mean nothing here are skipped, a different render system is an error
    out = subprocess.run(cmd[:-2] + ["--vsync", "0", "--renderSystem", "1"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert out.returncode != 0 and "renderSystem" in out.stdout


def test_frame_batching_is_bit_identical(std_env):
    """b200pt_set_frame_batch: B consecutive frames of a static camera run as one wavefront and fold into the image in frame
    order -- every image the unbatched renderer produces at a batch boundary (and at an explicit flush inside a batch) comes
    out bit for bit, with textures, MASK foliage (any-hit candidates, continuation rounds) and 2 samples per pixel; the frame-0
    selection / depth outputs come from the first frame only; a camera change mid-batch flushes the pending frames first."""
    from vk_gltf_renderer_b200 import synth
    from vk_gltf_renderer_b200.renderer import PathTracer, Resources
    scn = synth.synth_sponza(tex_size=128, detail=0.05)

    def run(batch, lanes, frames, spp=2):
        res = Resources(scene=scn, hdr_rgb=std_env, camera=scn.camera, size=(160, 96))
        pt = PathTracer(0)
        pt.ptMaxDepth, pt.ptSamples = 6, spp
        pt.onAttach(res)
        pt.set_frames_in_flight(lanes)
        pt.set_frame_batch(batch)
        snaps = {}
        for f in range(frames):
            res.frameCount = f
            pt.onRender(None, res)
            if f in (2, 6, frames - 1):
                snaps[f] = pt.read_accum()  # flushes a partial batch
        ids, depth = pt.read_selection()
        st = pt.stats()
        pt.onDetach(res)
        return snaps, ids, depth, st
    ref, ids0, d0, st0 = run(1, 2, 11)
    for batch, lanes in ((4, 1), (3, 2), (8, 2)):
        got, ids, d, st = run(batch, lanes, 11)
        for f in ref:
            assert np.array_equal(got[f], ref[f]), (batch, lanes, f)
        assert np.array_equal(ids, ids0) and np.array_equal(d, d0)
        assert st["closestRays"] == st0["closestRays"] and st["shadowRays"] == st0["shadowRays"] and st["kernelLaunches"] < st0["kernelLaunches"]
    # a frame that does not continue the pending batch (the accumulation restarts) flushes it and starts a new one
    res = Resources(scene=scn, hdr_rgb=std_env, camera=scn.camera, size=(160, 96))
    pt = PathTracer(0)
    pt.ptMaxDepth = 6
    pt.onAttach(res)
    pt.set_frame_batch(4)
    for f in (0, 1, 0, 1, 2):
        res.frameCount = f
        pt.onRender(None, res)
    a = pt.read_accum()
    pt.onDetach(res)
    res = Resources(scene=scn, hdr_rgb=std_env, camera=scn.camera, size=(160, 96))
    pt2, b = _gpu_render(scn, std_env, 160, 96, 3, ptMaxDepth=6)
    assert np.array_equal(a, b)

