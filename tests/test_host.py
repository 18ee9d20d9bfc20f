"""Host-side mirror of the reference interface: settings, pass plan, cameras, generator."""
import math
import os

import numpy as np

import bevy_gaussian_splatting_b200 as B
from bevy_gaussian_splatting_b200 import abi


def test_cloud_settings_defaults_match_reference():
    """src/gaussian/settings.rs:110-133."""
    s = B.CloudSettings()
    assert (s.aabb, s.global_opacity, s.global_scale, s.opacity_adaptive_radius) == (False, 1.0, 1.0, True)
    assert s.radix_sort_depth_bits == B.RadixSortDepthBits.Bits32
    assert s.gaussian_mode == B.GaussianMode.Gaussian3d and s.rasterize_mode == B.RasterizeMode.Color
    assert s.draw_mode == B.DrawMode.All and s.color_space == B.GaussianColorSpace.SrgbRec709Display
    a = s.to_abi()
    assert (a.gaussian_mode, a.rasterize_mode, a.aabb, a.opacity_adaptive_radius, a.draw_mode,
            a.radix_sort_depth_bits, a.flags) == (1, 0, 0, 1, 0, 32, 0)
    assert B.CloudSettings(sort_all=True).to_abi().flags == abi.BGS_FLAG_SORT_ALL


def test_headless_camera_matrices():
    """examples/headless.rs:177-184 + glam perspective_infinite_reverse_rh (fov pi/4, near 0.1)."""
    v = B.headless_view(1920, 1080)
    f = 1.0 / math.tan(math.pi / 8)
    assert np.isclose(v.clip_from_view[1, 1], f) and np.isclose(v.clip_from_view[0, 0], f / (1920 / 1080))
    assert v.clip_from_view[3, 2] == -1.0 and np.isclose(v.clip_from_view[2, 3], 0.1)
    assert np.allclose(v.view_from_world[:3, :3], np.eye(3)) and np.allclose(v.view_from_world[:3, 3], [0, -1.5, -5])
    # a point 10 units in front of the camera: ndc.z = near / depth (reverse-Z), inside (0, 1)
    p = np.array([0, 1.5, -5, 1], np.float32)
    c = v.clip_from_world @ p
    assert np.isclose(c[2] / c[3], 0.1 / 10.0) and abs(c[0]) < 1e-6
    a = v.to_abi()
    assert list(a.viewport) == [0.0, 0.0, 1920.0, 1080.0]
    assert np.allclose(np.array(list(a.clip_from_world)).reshape(4, 4).T, v.clip_from_world)   # column-major
    assert np.allclose(B.orbit_view(0, 8).view_from_world, v.view_from_world, atol=1e-6)


def test_random_gaussians_distributions_and_determinism():
    """planar_3d.rs:120-168: ranges per field; same (n, seed) -> same cloud; prefix-stable in n."""
    c = B.random_gaussians_3d_seeded(50_000, 0)
    assert c.rotation.min() >= -1 and c.rotation.max() < 1 and abs(c.rotation.mean()) < 0.02
    assert c.position_visibility[:, :3].min() >= -20 and c.position_visibility[:, :3].max() < 20
    assert np.all(c.position_visibility[:, 3] == 1.0)
    assert c.scale_opacity[:, :3].min() >= 0 and c.scale_opacity[:, :3].max() < 1
    assert c.scale_opacity[:, 3].min() >= 0 and c.scale_opacity[:, 3].max() < 0.8
    assert c.spherical_harmonic.shape == (50_000, 48) and c.spherical_harmonic.min() >= -1
    d = B.random_gaussians_3d_seeded(50_000, 0)
    assert np.array_equal(c.spherical_harmonic, d.spherical_harmonic)
    e = B.random_gaussians_3d_seeded(300_000, 0)
    assert np.array_equal(e.rotation[:50_000], c.rotation)
    assert not np.array_equal(B.random_gaussians_3d_seeded(1000, 1).rotation, c.rotation[:1000])


def test_planar_layout_sizes():
    """a1: 240 B/gaussian f32, 128 B/gaussian f16 (position stays f32)."""
    c = B.random_gaussians_3d_seeded(10, 0)
    f32_bytes = sum(a.nbytes for a in (c.position_visibility, c.spherical_harmonic, c.rotation, c.scale_opacity)) // 10
    shp, rso = c.pack_f16()
    f16_bytes = (c.position_visibility.nbytes + shp.nbytes + rso.nbytes) // 10
    assert (f32_bytes, f16_bytes) == (240, 128)


def test_entity_aabb_follows_the_reference_sequence():
    """compute_aabb (interface.rs:22-66) -> Aabb {center, half_extents} (cloud.rs:45-62) -> min()/max() in f32."""
    cloud = B.random_gaussians_3d_seeded(513, 9)
    lo, hi = cloud.compute_aabb()
    p = cloud.position_visibility[:, :3]
    f = np.float32
    mn = np.full(3, np.inf, f); mx = np.full(3, -np.inf, f)
    for row in p:                                  # the non-rayon loop of interface.rs:52-57, literally
        mn = np.minimum(mn, (row - f(0.1)).astype(f)); mx = np.maximum(mx, (row + f(0.1)).astype(f))
    center = ((mn + mx).astype(f) / f(2)).astype(f); half = ((mx - mn).astype(f) / f(2)).astype(f)
    assert np.array_equal(lo, (center - half).astype(f)) and np.array_equal(hi, (center + half).astype(f))
    u = B.GaussianSplattingPlugin.cloud_uniform(B.CloudSettings(), None, (lo, hi))
    assert list(u.aabb_min) == [float(lo[0]), float(lo[1]), float(lo[2]), 1.0] and u.aabb_max[3] == 1.0


def test_settings_flags_and_modes_map_to_the_abi():
    from bevy_gaussian_splatting_b200 import abi
    assert B.CloudSettings().to_abi().flags == 0
    assert B.CloudSettings(sort_all=True).to_abi().flags == abi.BGS_FLAG_SORT_ALL
    assert B.CloudSettings(binning_rounds=True).to_abi().flags == abi.BGS_FLAG_CHUNKS
    assert B.CloudSettings(binning_rounds=False, sort_all=True).to_abi().flags == abi.BGS_FLAG_NO_CHUNKS | abi.BGS_FLAG_SORT_ALL
    s = B.CloudSettings(rasterize_mode=B.RasterizeMode.Position, gaussian_mode=B.GaussianMode.Gaussian2d, aabb=True).to_abi()
    assert (s.rasterize_mode, s.gaussian_mode, s.aabb) == (3, 0, 1)
    hdr = open(os.path.join(os.path.dirname(__file__), "..", "include", "bgs.h")).read()
    for name, val in (("BGS_FLAG_SORT_ALL", 1), ("BGS_FLAG_ASYNC", 2), ("BGS_FLAG_NO_CHUNKS", 4), ("BGS_FLAG_CHUNKS", 8)):
        assert f"{name} = {val}u" in hdr and getattr(abi, name) == val
    assert "BGS_RASTERIZE_POSITION = 3" in hdr


def test_bench_arms_on_a_box_without_a_gpu():
    """The reference arm runs the CPU oracle port and prints the contract's JSON line; the CUDA arm refuses to run
    without a GPU (no CPU fallback)."""
    import json, subprocess, sys, torch
    root = os.path.join(os.path.dirname(__file__), "..")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "3"], cwd=root,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Msplats/s" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["n_gpus"] == 1
    if not torch.cuda.is_available():
        r = subprocess.run([sys.executable, "bench.py", "--steps", "1"], cwd=root, capture_output=True, text=True, timeout=600)
        assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def test_bench_steps_set_the_timed_frames():
    """--steps is the number of timed frames of either arm; a run without any is refused."""
    import json, subprocess, sys
    root = os.path.join(os.path.dirname(__file__), "..")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "2", "--warmup", "3"], cwd=root,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and "best of 2 frames" in line["cpu_baseline"]["sample"]
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, "bench.py", *bad], cwd=root, capture_output=True, text=True, timeout=300)
        assert r.returncode == 2, r.stderr[-2000:]


def test_bench_dump_frames_full_and_sampled(tmp_path, monkeypatch):
    """--dump-outputs writes the frames whole while they fit the size limit, else the same seeded pixel sample of every
    view, identical from run to run; all of it float32 / float64 within the limit."""
    import bench

    frames = np.random.default_rng(1).integers(0, 256, (3, 40, 64, 4), dtype=np.uint8)
    bench.dump_frames(str(tmp_path / "full"), frames)
    assert os.listdir(tmp_path / "full") == ["frames.npy"]
    got = np.load(tmp_path / "full" / "frames.npy")
    assert got.dtype == np.float32 and np.array_equal(got, frames)
    limit = 4096 + 20_000
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", limit)
    for d in ("a", "b"):
        bench.dump_frames(str(tmp_path / d), frames)
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= limit
    sample, pix = np.load(tmp_path / "a" / "frames_sample.npy"), np.load(tmp_path / "a" / "frames_sample_pixel.npy")
    assert sample.dtype == np.float32 and pix.dtype == np.float64 and sample.shape == (3, len(pix), 4) and len(pix) > 100
    assert np.array_equal(sample, frames.reshape(3, -1, 4)[:, pix.astype(np.int64)])
    assert np.array_equal(sample, np.load(tmp_path / "b" / "frames_sample.npy"))
