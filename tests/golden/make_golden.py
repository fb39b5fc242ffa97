"""Generate the committed golden vectors by running the REFERENCE's own code in this container.

    python tests/golden/make_golden.py          (needs /root/reference; writes tests/golden/*.npz)

What is pinned (files under /root/reference executed unmodified through tests/golden/_reference_shim.py):
  rope_*.npz        aether/pipelines/aetherv1_pipeline_cogvideox.py:25-144, :148-163  get_3d_rotary_pos_embed
  compute_scale.npz aether/utils/postprocess_utils.py:847-864                         compute_scale
  sliding_*.npz     evaluation/video_depth/launch_aether.py:81-287                    process_with_sliding_window
                    (tile plan, compute_scale, spatial + temporal blend chain) with a deterministic stand-in
                    for the per-tile pipeline call (tests/helpers.py::fake_tile_outputs)
  pipeline_*.npz    aether/pipelines/aetherv1_pipeline_cogvideox.py:350-965           check/preprocess/prepare_latents/
                    __call__ (reconstruction, prediction with raymap + dynamic CFG, planning) driving the oracle
                    modules with float64 arithmetic and bf16 module I/O (tests/helpers.py::exact_oracle_modules) on
                    CPU with a CPU generator -- portable across hosts (round 1 used bf16 CPU modules whose rounding
                    followed the host ISA); diffusers' VideoProcessor stand-in = oracle/video_processor.py.
The third-party diffusers modules themselves stay "parity unpinned" (see oracle/__init__.py).
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE))
sys.path.insert(0, str(HERE.parent))
sys.path.insert(0, str(HERE.parent.parent))

import _reference_shim as shim  # noqa: E402
from helpers import (TINY, empty_prompt_embeds, fake_tile_outputs, subsample, synthetic_long_clip,  # noqa: E402
                     synthetic_raymap, synthetic_video, exact_oracle_modules)


def make_rope():
    P = shim.reference_pipeline_module()
    cases = {"full_fps12": (60, 90, 11, 12, (30, 45)), "full_fps8": (60, 90, 11, 8, (30, 45)),
             "full_fps24_f5": (60, 90, 5, 24, (30, 45)), "tiny_fps12": (12, 20, 5, 12, (6, 10)),
             "tiny_fps10": (12, 20, 5, 10, (6, 10))}
    out = {}
    for name, (sh, sw, f, fps, grid) in cases.items():
        crops = P.get_resize_crop_region_for_grid(grid, sw // 2, sh // 2)
        cos, sin = P.get_3d_rotary_pos_embed(embed_dim=64, crops_coords=crops, grid_size=grid, temporal_size=f,
                                             fps_factor=12 / fps)
        cos, sin = cos.numpy(), sin.numpy()
        step = 1 if cos.shape[0] <= 600 else 53
        out[f"{name}__cos"] = cos[::step]
        out[f"{name}__sin"] = sin[::step]
        out[f"{name}__meta"] = np.array([sh, sw, f, fps, grid[0], grid[1], step, cos.shape[0]], dtype=np.int64)
        out[f"{name}__sums"] = np.array([cos.astype(np.float64).sum(), sin.astype(np.float64).sum(),
                                         np.abs(cos).astype(np.float64).sum()])
        out[f"{name}__crops"] = np.array(crops, dtype=np.int64)
    np.savez_compressed(HERE / "rope.npz", **out)
    print("rope.npz", len(out))


def make_compute_scale():
    POST = shim.reference_postprocess_module()
    g = np.random.default_rng(0)
    out = {}
    for i, (shape, gain, f64) in enumerate([((1, 200, 37), 1.7, False), ((1, 41 * 48, 58), 0.83, True),
                                            ((1, 33, 720), 1.0, False), ((1, 5, 5), 0.0, False)]):
        pred = g.uniform(0.05, 2.0, size=shape).astype(np.float32)
        tgt = (pred * gain + 0.01 * g.standard_normal(shape)).astype(np.float64 if f64 else np.float32)
        if gain == 0.0:
            pred = np.zeros(shape, np.float32)
        s = POST.compute_scale(pred, tgt, np.ones_like(tgt))
        out[f"c{i}__pred"], out[f"c{i}__target"], out[f"c{i}__scale"] = pred, tgt, np.float64(s)
    np.savez_compressed(HERE / "compute_scale.npz", **out)
    print("compute_scale.npz")


def make_sliding():
    EVD = shim.reference_sliding_window_module()

    class FakePipeline:
        """Stands in for the per-tile pipeline call (launch_aether.py:151-158): records the crops it is handed."""

        def __init__(self, obs):
            self.obs = obs
            self.calls = []

        def __call__(self, video, num_inference_steps, num_frames, generator, return_dict, fps):
            # locate the crop inside the clip to recover (t_start, h_start, w_start) exactly like a tile plan would
            self.calls.append(video.shape)
            t0, h0, w0 = self._locate(video)
            rgb, disp = fake_tile_outputs(video, t0, h0, w0)
            return rgb[None], disp[None], None

        def _locate(self, video):
            return self._next

    import math

    def run(t, h, w, name):
        obs = synthetic_long_clip(t, h, w)
        fp = FakePipeline(obs)
        # replay the reference tile enumeration to feed _locate (pure bookkeeping, mirrors :87-149)
        from aether_b200.sliding_window import plan_windows
        plan = plan_windows(t, h, w, t)
        it = iter(plan.tiles)

        def locate(video):
            tl = next(it)
            assert video.shape[:3] == (tl.t_end - tl.t_start, tl.h_end - tl.h_start, tl.w_end - tl.w_start)
            assert np.array_equal(video, obs[0, tl.t_start:tl.t_end, tl.h_start:tl.h_end, tl.w_start:tl.w_end])
            return tl.t_start, tl.h_start, tl.w_start
        fp._locate = locate
        orig = torch.Generator

        class _Gen:   # launch_aether.py:155 builds torch.Generator(device="cuda"); no CUDA here and the stand-in ignores it
            def __init__(self, device=None):
                pass

            def manual_seed(self, s):
                return self
        # the scale of every blend link, in call order (spatial links window by window, then the temporal chain):
        # compute_scale sums fp32 products with torch.sum, whose order follows the host's thread count
        scales, ref_scale = [], EVD.compute_scale

        def recording_scale(*a, **k):
            s = ref_scale(*a, **k)
            scales.append(float(s))
            return s
        torch.Generator = _Gen
        EVD.compute_scale = recording_scale
        try:
            rgb, disp = EVD.process_with_sliding_window(fp, obs, num_inference_step=4, total_frames=t, seed=3407)
        finally:
            torch.Generator = orig
            EVD.compute_scale = ref_scale
        assert len(fp.calls) == len(plan.tiles)
        tiles = np.array([[tl.t_start, tl.t_end, tl.h_start, tl.h_end, tl.w_start, tl.w_end] for tl in plan.tiles],
                         dtype=np.int64)
        np.savez_compressed(HERE / f"sliding_{name}.npz", thw=np.array([t, h, w]), tiles=tiles,
                            disparity_sub=subsample(disp, (3, 16, 16)), disparity_dtype=str(disp.dtype),
                            disparity_shape=np.array(disp.shape), disparity_sum=np.float64(disp.sum()),
                            disparity_abs_sum=np.float64(np.abs(disp).sum()),
                            rgb_sub=subsample(rgb, (8, 32, 32, 1)), rgb_shape=np.array(rgb.shape))
        print(f"sliding_{name}.npz", disp.shape, disp.dtype, len(plan.tiles), "tiles")
        all_scales[name] = np.array(scales, dtype=np.float64)

    all_scales = {}
    run(57, 480, 720, "temporal")        # 3 temporal windows, no spatial tiling (windows stay fp32)
    run(49, 480, 853, "horizontal")      # 2 temporal x 2 horizontal tiles (overlap 587 px, SURVEY.md 8d config 5)
    run(41, 600, 720, "vertical")        # 1 temporal x 2 vertical tiles
    run(129, 480, 853, "long")           # 12 temporal x 2 horizontal = 24 tiles: the chain of BASELINE configs[4]
    #                                      (512 frames -> 60 x 2 tiles) at a quarter of its length, incl. the
    #                                      irregular last window at t - 41
    np.savez_compressed(HERE / "sliding_scales.npz", **all_scales)
    print("sliding_scales.npz", {k: len(v) for k, v in all_scales.items()})


def make_pipeline():
    P = shim.reference_pipeline_module()
    dit, vae, sched = exact_oracle_modules()
    emb = empty_prompt_embeds()
    pipe = P.AetherV1PipelineCogVideoX(tokenizer=None, text_encoder=lambda prompt: emb, vae=vae, scheduler=sched,
                                       transformer=dit)
    captured = {}
    orig_decode = pipe.decode_latents

    def decode_latents(latents):
        captured.setdefault("latents", []).append(latents.detach().clone())
        return orig_decode(latents)
    pipe.decode_latents = decode_latents

    H, W, F = TINY["height"], TINY["width"], TINY["num_frames"]
    video = synthetic_video(F, H, W)
    raymap = synthetic_raymap(F, H // 8, W // 8)
    cases = {
        "reconstruction": dict(task="reconstruction", video=video, num_inference_steps=3),
        "prediction": dict(task="prediction", image=video[0], raymap=raymap, num_inference_steps=3),
        "planning": dict(task="planning", image=video[0], goal=video[-1], num_inference_steps=2, guidance_scale=2.5),
        "reconstruction_fps8": dict(task="reconstruction", video=video, num_inference_steps=2, fps=8),
    }
    for name, kw in cases.items():
        captured.clear()
        with torch.no_grad():
            out = pipe(height=H, width=W, num_frames=F, generator=torch.Generator().manual_seed(42), **kw)
        lat = torch.cat([captured["latents"][0], captured["latents"][1]], dim=2)     # rgb | disparity latents
        np.savez_compressed(
            HERE / f"pipeline_{name}.npz",
            rgb_sub=subsample(out.rgb, (2, 2, 2, 1)), disparity=out.disparity, raymap=out.raymap,
            rgb_disp_latents=lat.float().numpy(), rgb_shape=np.array(out.rgb.shape))
        print(f"pipeline_{name}.npz rgb {out.rgb.shape} disp {out.disparity.shape} raymap {out.raymap.shape}")
    # error behaviour of check_inputs (:362-449): message strings are part of the drop-in surface
    msgs = {}
    bad = {
        "frames": dict(task="reconstruction", video=video[:9], num_frames=9),
        "fps": dict(task="reconstruction", video=video, num_frames=F, fps=13),
        "both": dict(task="prediction", image=video[0], video=video, num_frames=F),
        "none": dict(task="prediction", num_frames=F),
        "goal_task": dict(task="prediction", image=video[0], goal=video[1], num_frames=F),
        "raymap_shape": dict(task="prediction", image=video[0], raymap=raymap[:5], num_frames=F),
        "task": dict(task="segmentation", video=video, num_frames=F),
        "hw": dict(task="reconstruction", video=video, num_frames=F, height=100),
    }
    for k, kw in bad.items():
        kw.setdefault("height", H)
        kw.setdefault("width", W)
        try:
            pipe(**kw)
            msgs[k] = "NO ERROR"
        except ValueError as e:
            msgs[k] = str(e)
    np.savez_compressed(HERE / "pipeline_errors.npz", **{k: np.array(v) for k, v in msgs.items()})
    print("pipeline_errors.npz", msgs)


def make_prepare_input():
    from helpers import PREPARE_INPUT_SIZES, prepare_input_frames
    """launch_aether.py:388-403 prepare_input (aspect-preserving cv2 resize to the 480 x 720 window, /255) on seeded
    uint8 frames; the file read is replaced by a lookup."""
    EVD = shim.reference_sliding_window_module()
    out = {}
    for h, w in PREPARE_INPUT_SIZES:
        frames = prepare_input_frames(h, w)
        EVD.iio.imread = lambda p, frames=frames: frames[int(p)]
        ref = EVD.prepare_input([str(i) for i in range(len(frames))])
        out[f"{h}x{w}__shape"] = np.array(ref.shape)
        out[f"{h}x{w}__sum"] = np.float64(ref.sum())
        out[f"{h}x{w}__sub"] = subsample(ref, (1, 24, 24, 1))
    np.savez_compressed(HERE / "prepare_input.npz", **out)
    print("prepare_input.npz", len(out))


DEPTH_EVAL_MODES = {
    "median": dict(max_depth=70, post_clip_max=70),
    "scale": dict(max_depth=70, post_clip_max=70, align_with_scale=True),
    "scale_shift_l2": dict(max_depth=70, post_clip_max=70, align_with_lstsq=True),
    "scale_shift_lad": dict(max_depth=70, post_clip_max=70, align_with_lad2=True, max_iters=200, lr=1e-2),
    "metric": dict(max_depth=70, post_clip_max=70, metric_scale=True),
    "median_disp_edge_mask": dict(max_depth=70, disp_input=True, mask_edge=True, pre_clip_min=0.1, use_mask=True),
}


def make_depth_eval():
    """evaluation/video_depth/tools.py:179-470 depth_evaluation on a seeded synthetic scene, every alignment the
    evaluation scripts select (eval_depth.py:157-215) + the disparity-space / edge-mask / custom-mask options."""
    from helpers import depth_eval_case
    T = shim.reference_depth_tools_module()
    pred, gt, mask = depth_eval_case()
    out = {}
    for name, kw in DEPTH_EVAL_MODES.items():
        kw = dict(kw)
        cm = mask if kw.pop("use_mask", False) else None
        res, err, full, gt_full = T.depth_evaluation(pred.copy(), gt.copy(), custom_mask=cm, **kw)
        keys = sorted(res)
        out[f"{name}__keys"] = np.array(keys)
        out[f"{name}__vals"] = np.array([float(res[k]) for k in keys], dtype=np.float64)
        out[f"{name}__err_sum"] = np.float64(err.double().sum().item())
        out[f"{name}__full_sum"] = np.float64(full.double().sum().item())
    np.savez_compressed(HERE / "depth_eval.npz", **out)
    print("depth_eval.npz", {k: out[f"{k}__vals"][:2] for k in DEPTH_EVAL_MODES})


def _stats(a):
    a = np.asarray(a, dtype=np.float64)
    return np.array([a.sum(), np.abs(a).sum(), (a * a).sum()])


def make_pose_blend():
    """aether/utils/postprocess_utils.py (raymap_to_poses, postprocess_pointmap, smoothing, alignment, SLERP), the rel-pose
    window blend (evaluation/rel_pose/launch_aether.py:124-250) and the demo merge (scripts/demo.py:235-422), all executed
    from the reference's files on the deterministic inputs of tests/helpers.py (filterpy = oracle/kalman.py stand-in)."""
    from types import SimpleNamespace
    from helpers import fake_pose_window, raymap_from_poses, synthetic_trajectory
    POST = shim.reference_postprocess_module()
    EVP = shim.reference_rel_pose_module()
    DEMO = shim.reference_demo_module()
    out = {}
    # -- raymap -> poses / fov, point map
    traj = synthetic_trajectory(17, seed=3)
    ray = raymap_from_poses(traj, 12, 20, focal_px=150.0, scale=1.0)
    pose, fx, fy = POST.raymap_to_poses(ray.copy())
    out["r2p__pose"], out["r2p__fovx"], out["r2p__fovy"] = pose, fx, fy
    _, disp, _ = fake_pose_window(0, 17, h=12, w=20, seed=1)
    for mode in ("none", "simple", "kalman"):
        pcd = POST.postprocess_pointmap(disp.copy(), ray.copy(), smooth_camera=(mode != "none"), smooth_method=mode)
        out[f"pcd_{mode}__pose"] = pcd["camera_pose"]
        out[f"pcd_{mode}__K"] = pcd["intrinsics"]
        out[f"pcd_{mode}__points"] = _stats(pcd["pointmap"])
        out[f"pcd_{mode}__points_sub"] = subsample(pcd["pointmap"], (4, 16, 16, 1))
    # -- smoothing / alignment / interpolation primitives
    noisy = synthetic_trajectory(41, seed=5)
    out["smooth_gaussian"] = POST.smooth_poses(noisy.copy(), 5, "gaussian")
    out["smooth_savgol"] = POST.smooth_poses(noisy.copy(), 7, "savgol")
    out["smooth_kalman"] = POST.smooth_trajectory(noisy.copy(), 5)
    static = np.repeat(noisy[:1], 12, axis=0) + 1e-4 * np.random.default_rng(0).standard_normal((12, 4, 4)) * (np.arange(16).reshape(4, 4) % 4 == 3)
    st = POST.detect_static_sequence(static)
    out["static__flags"] = np.array([float(st[0]), st[1], st[2]])
    out["static__smoothed"] = POST.adaptive_pose_smoothing(static.copy(), st[1], st[2])
    a, b = synthetic_trajectory(33, seed=7)[:, :3, :4], synthetic_trajectory(33, seed=8)[:, :3, :4]
    R, T, sc = POST.align_camera_extrinsics(torch.from_numpy(a), torch.from_numpy(b))
    out["align__R"], out["align__T"], out["align__s"] = R.numpy(), T.numpy(), np.float64(sc)
    out["align__applied"] = POST.apply_transformation(torch.from_numpy(a), R, T, sc).numpy()
    out["interp"] = np.stack([POST.interpolate_poses(noisy[3], noisy[30], wgt) for wgt in (0.0, 0.25, 0.5, 1.0)])
    out["interp_close"] = POST.interpolate_poses(noisy[3], noisy[4], 0.3)
    # -- rank 1: rel-pose windows (105 frames -> starts 0, 32, 64), fake pipeline
    class FakePipe:
        def __call__(self, video, num_inference_steps, num_frames, generator, return_dict, fps):
            t0 = int(video[0, 0, 0, 0])
            rgb, d, r = fake_pose_window(t0, num_frames, seed=2)
            return rgb[None], d[None], r[None]
    frames = np.zeros((1, 105, 24, 40, 3))
    frames[0, :, 0, 0, 0] = np.arange(105)                  # the fake pipeline reads the window start from the clip
    orig = torch.Generator

    class _Gen:
        def __init__(self, device=None):
            pass

        def manual_seed(self, s):
            return self
    torch.Generator = _Gen
    try:
        res = EVP.process_video_with_sliding_window(FakePipe(), frames, 4, 42)
    finally:
        torch.Generator = orig
    for k in ("rgb", "disparity", "focals"):
        out[f"relpose__{k}"] = _stats(res[k])
    out["relpose__poses"] = res["poses"]
    out["relpose__range"] = np.array(res["range"])
    out["relpose__disparity_sub"] = subsample(res["disparity"], (5, 4, 4))
    # -- rank 2: demo merge (89 frames, windows of 41, stride 24 -> starts 0, 24, 48)
    starts = DEMO.get_window_starts(89, 41, 24)
    out["demo__starts"] = np.array(starts)
    for align in (False, True):
        wins = []
        for t0 in starts:
            rgb, d, r = fake_pose_window(t0, 41, seed=4)
            wins.append(SimpleNamespace(rgb=rgb, disparity=d, raymap=r))
        args = SimpleNamespace(width=40, height=24, smooth_camera=True, smooth_method="kalman", align_pointmaps=align)
        m_rgb, m_disp, m_pose, pts = DEMO.blend_and_merge_window_results(wins, starts, args)
        tag = f"demo_align{int(align)}"
        out[f"{tag}__rgb"], out[f"{tag}__disp"], out[f"{tag}__pts"] = _stats(m_rgb), _stats(m_disp), _stats(pts)
        out[f"{tag}__poses"] = m_pose
        out[f"{tag}__pts_sub"] = subsample(np.asarray(pts), (6, 4, 4, 1))
        out[f"{tag}__disp_sub"] = subsample(m_disp, (6, 4, 4))
    np.savez_compressed(HERE / "pose_blend.npz", **out)
    print("pose_blend.npz", len(out), "arrays; relpose range", out["relpose__range"], "demo starts", starts)


if __name__ == "__main__":
    torch.manual_seed(0)
    which = sys.argv[1:] or ["rope", "scale", "sliding", "pipeline", "prepare", "depth_eval", "pose_blend"]
    if "depth_eval" in which:
        make_depth_eval()
    if "pose_blend" in which:
        make_pose_blend()
    if "prepare" in which:
        make_prepare_input()
    if "rope" in which:
        make_rope()
    if "scale" in which:
        make_compute_scale()
    if "sliding" in which:
        make_sliding()
    if "pipeline" in which:
        make_pipeline()
