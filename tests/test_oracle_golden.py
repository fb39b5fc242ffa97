"""CPU: the oracle restatements and the host-side mirrors against the golden vectors produced by the
reference's own code (tests/golden/make_golden.py).  Bit-exact where the arithmetic is the same expression
graph (RoPE table, tile plan, compute_scale, pipeline glue with identical modules/RNG); the blend chain is
compared at fp64 round-off (identical operations, numpy in both cases)."""
import numpy as np
import pytest
import torch

from helpers import (TINY, empty_prompt_embeds, fake_tile_outputs, subsample, synthetic_long_clip, synthetic_raymap,
                     synthetic_video, exact_oracle_modules)


# ------------------------------------------------------------------------------------------------ RoPE
@pytest.mark.parametrize("impl", ["oracle", "product"])
def test_rope_tables_match_reference(golden_dir, impl):
    g = np.load(golden_dir / "rope.npz")
    names = sorted({k.split("__")[0] for k in g.files})
    assert len(names) == 5
    for name in names:
        sh, sw, f, fps, gh, gw, step, n = g[f"{name}__meta"].tolist()
        if impl == "oracle":
            from oracle.rope import prepare_rotary_positional_embeddings as prep
            cos, sin = prep(sh * 8, sw * 8, f, sample_height=sh, sample_width=sw, fps=fps)
        else:
            from aether_b200.rope import prepare_rotary_positional_embeddings as prep
            cos, sin = prep(sh * 8, sw * 8, f, patch_size=2, vae_scale_factor_spatial=8, sample_height=sh,
                            sample_width=sw, attention_head_dim=64, base_fps=12, fps=fps)
        assert cos.shape == (n, 64) and cos.dtype == torch.float32
        assert np.array_equal(cos.numpy()[::step], g[f"{name}__cos"]), name
        assert np.array_equal(sin.numpy()[::step], g[f"{name}__sin"]), name
        sums = g[f"{name}__sums"]
        assert cos.double().sum().item() == pytest.approx(sums[0], rel=1e-12)
        assert sin.double().sum().item() == pytest.approx(sums[1], rel=1e-12, abs=1e-9)


def test_rope_preserves_norm():
    """KAT: a rotation never changes the pairwise norm."""
    from oracle.rope import apply_rotary_emb, prepare_rotary_positional_embeddings
    cos, sin = prepare_rotary_positional_embeddings(96, 160, 5, sample_height=12, sample_width=20, fps=8)
    x = torch.randn(1, 2, cos.shape[0], 64)
    y = apply_rotary_emb(x, cos, sin)
    n0 = x.reshape(1, 2, -1, 32, 2).pow(2).sum(-1)
    n1 = y.reshape(1, 2, -1, 32, 2).pow(2).sum(-1)
    assert torch.allclose(n0, n1, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------------ scheduler
def test_scheduler_known_answers():
    from oracle.scheduler import OracleDPMScheduler
    from aether_b200.scheduler import AetherDPMScheduler
    o, p = OracleDPMScheduler(), AetherDPMScheduler()
    for n in (50, 4, 2):
        o.set_timesteps(n)
        p.set_timesteps(n)
        assert torch.equal(o.timesteps, p.timesteps.cpu())
        ts = o.timesteps.tolist()
        assert ts[0] == 999 and ts[-1] == 1000 // n - 1
        for i, t in enumerate(ts):
            tb = ts[i - 1] if i > 0 else None
            co, cp = o.coefficients(t, tb), p.coefficients(t, tb)
            for k in ("sqrt_a", "sqrt_1ma", "m1", "m2", "m_noise"):
                assert float(co[k]) == pytest.approx(cp[k], rel=1e-12, abs=1e-15), (n, t, k)
            if tb is not None and co["prev_t"] >= 0:
                assert float(co["m3"]) == pytest.approx(cp["m3"], rel=1e-12)
                assert float(co["m4"]) == pytest.approx(cp["m4"], rel=1e-12, abs=1e-15)
        first = o.coefficients(ts[0], None)
        assert float(first["sqrt_a"]) == 0.0 and float(first["m1"]) == 0.0          # zero terminal SNR: alpha_T = 0
        last = o.coefficients(ts[-1], ts[-2])
        assert float(last["m1"]) == 0.0 and float(last["m2"]) == -1.0 and float(last["m_noise"]) == 0.0
    # last step returns x0 exactly
    o.set_timesteps(4)
    x = torch.randn(1, 2, 3, 4).bfloat16()
    v = torch.randn(1, 2, 3, 4)
    prev, x0 = o.step(v, torch.randn(1, 2, 3, 4), 249, 499, x)
    assert torch.equal(prev, x0)
    assert o.alphas_cumprod[999].item() == 0.0 and o.alphas_cumprod.dtype == torch.float64


# ------------------------------------------------------------------------------------------------ blend
def test_compute_scale_matches_reference(golden_dir):
    from oracle.blend import compute_scale
    g = np.load(golden_dir / "compute_scale.npz")
    for i in range(4):
        pred, tgt = g[f"c{i}__pred"], g[f"c{i}__target"]
        assert compute_scale(pred, tgt, np.ones_like(tgt)) == float(g[f"c{i}__scale"])
    assert float(g["c3__scale"]) == 0.0           # zero denominator -> 0 (postprocess_utils.py:858-862)


@pytest.mark.parametrize("name", ["temporal", "horizontal", "vertical", "long"])
def test_tile_plan_and_blend_match_reference(golden_dir, name, monkeypatch):
    """compute_scale sums its fp32 products with torch.sum, whose summation order follows the host's thread count, so a
    link's scale may differ from the reference's by an fp32 rounding.  Each scale the oracle computes is checked against
    the reference's scale of the same link (tests/golden/sliding_scales.npz) at that rounding, and the reference's scale
    is carried on: the fp64 chain itself is then compared at round-off on any host."""
    import oracle.blend as B
    from aether_b200.sliding_window import plan_windows
    g = np.load(golden_dir / f"sliding_{name}.npz")
    t, h, w = g["thw"].tolist()
    plan = plan_windows(t, h, w, t)
    tiles = np.array([[tl.t_start, tl.t_end, tl.h_start, tl.h_end, tl.w_start, tl.w_end] for tl in plan.tiles])
    assert np.array_equal(tiles, g["tiles"])
    obs = synthetic_long_clip(t, h, w)
    disps = []
    for tl in plan.tiles:
        crop = obs[0, tl.t_start:tl.t_end, tl.h_start:tl.h_end, tl.w_start:tl.w_end]
        disps.append(fake_tile_outputs(crop, tl.t_start, tl.h_start, tl.w_start)[1])
    ref_scales = np.load(golden_dir / "sliding_scales.npz")[name].tolist()
    seen, oracle_scale = [], B.compute_scale

    def scale_of_link(prediction, target, mask):
        ref = ref_scales[len(seen)]
        seen.append(oracle_scale(prediction, target, mask))
        assert seen[-1] == pytest.approx(ref, rel=2e-6, abs=0), (len(seen) - 1, seen[-1], ref)
        return ref
    monkeypatch.setattr(B, "compute_scale", scale_of_link)
    final = B.blend_all(disps, tiles, plan.n_spatial, plan.is_horizontal)
    assert len(seen) == len(ref_scales)
    assert final.dtype == np.float64 and list(final.shape) == g["disparity_shape"].tolist()
    np.testing.assert_allclose(subsample(final, (3, 16, 16)), g["disparity_sub"], rtol=1e-12, atol=0)
    assert final.sum() == pytest.approx(float(g["disparity_sum"]), rel=1e-12)


def test_prepare_frames_and_depth_match_reference_launcher(golden_dir):
    """Launcher glue either side of the tile loop: `prepare_input` (launch_aether.py:388-403) against the golden made
    by the reference's own function, and depth = clip(1 / disparity, 0, 100) (:347)."""
    pytest.importorskip("cv2")
    from aether_b200.sliding_window import disparity_to_depth, plan_windows, prepare_frames
    from helpers import PREPARE_INPUT_SIZES, prepare_input_frames
    g = np.load(golden_dir / "prepare_input.npz")
    for h, w in PREPARE_INPUT_SIZES:
        got = prepare_frames(prepare_input_frames(h, w))
        assert got.dtype == np.float64 and list(got.shape) == g[f"{h}x{w}__shape"].tolist()
        assert got.sum() == float(g[f"{h}x{w}__sum"])
        assert np.array_equal(subsample(got, (1, 24, 24, 1)), g[f"{h}x{w}__sub"])
        plan_windows(got.shape[0], got.shape[1], got.shape[2])          # always a single tiling direction
    d = np.array([[0.0, 1e-3, 0.5, 4.0]])
    with np.errstate(divide="ignore"):
        assert np.array_equal(disparity_to_depth(d), np.array([[100.0, 100.0, 2.0, 0.25]]))


def test_plan_config5_geometry():
    """SURVEY.md 8(d) config 5: 512 frames of 480x853 -> 60 temporal x 2 spatial = 120 tiles, overlap 587 px."""
    from aether_b200.sliding_window import partition_tiles, plan_windows
    plan = plan_windows(512, 480, 853)
    assert plan.n_temporal == 60 and plan.n_spatial == 2 and len(plan.tiles) == 120 and plan.is_horizontal
    assert plan.tiles[0].w_end - plan.tiles[1].w_start == 587
    assert plan.tiles[-1].t_start == 471 and plan.tiles[-1].t_end == 512
    parts = [partition_tiles(120, r, 8) for r in range(8)]
    assert sorted(sum(parts, [])) == list(range(120)) and all(len(p) == 15 for p in parts)
    # the 9-frame fallback of launch_aether.py:87-89 shrinks the window (and the pipeline then rejects it)
    assert plan_windows(9, 480, 720).frames_per_window == 9


# ------------------------------------------------------------------------------------------------ pipeline glue
def _product_pipeline_with_oracle_modules():
    from aether_b200.pipeline import AetherV1PipelineCogVideoX
    dit, vae, sched = exact_oracle_modules()
    return AetherV1PipelineCogVideoX(vae=vae, scheduler=sched, transformer=dit,
                                     empty_prompt_embeds=empty_prompt_embeds())


@pytest.mark.parametrize("name,kw", [
    ("reconstruction", dict(task="reconstruction", num_inference_steps=3)),
    ("prediction", dict(task="prediction", num_inference_steps=3)),
    ("planning", dict(task="planning", num_inference_steps=2, guidance_scale=2.5)),
    ("reconstruction_fps8", dict(task="reconstruction", num_inference_steps=2, fps=8)),
])
def test_pipeline_glue_matches_reference(golden_dir, name, kw):
    """aether_b200.pipeline (host mirror) driving the SAME oracle modules with the SAME CPU generator must
    reproduce the reference pipeline's outputs: this pins input preprocessing, latent assembly, raymap
    fold/unfold, RoPE, dynamic CFG, the loop and the output post-processing to the reference.

    The modules compute in float64 with bf16 I/O (helpers.exact_oracle_modules) so the fixture does not depend on
    the host's bf16/fp32 GEMM kernels; on the generating host the comparison is bit-exact.  Across hosts the only
    residue is a last-bit difference of a float64/float32 transcendental (exp/tanh/cos differ by <= 1 ulp between
    SIMD back ends) that can, rarely, flip one bf16 rounding at a module boundary; the following DiT steps and the
    random-weight VAE decoder then spread that single ulp (measured with a deliberately perturbed time embedding:
    4.6 % of the disparity elements differ, rel-RMS 2e-3).  Bound: rel-RMS <= 5e-3 and <= 10 % differing elements
    (a glue error -- wrong channel order, wrong frame padding, a missed CFG branch -- moves these by O(1)).
    Verified bit-exact here under MKL_ENABLE_INSTRUCTIONS=AVX2 / ATEN_CPU_CAPABILITY=avx2 / 3 threads as well."""
    g = np.load(golden_dir / f"pipeline_{name}.npz")
    H, W, F = TINY["height"], TINY["width"], TINY["num_frames"]
    video = synthetic_video(F, H, W)
    kw = dict(kw)
    if kw["task"] == "reconstruction":
        kw["video"] = video
    else:
        kw["image"] = video[0]
        if kw["task"] == "planning":
            kw["goal"] = video[-1]
        else:
            kw["raymap"] = synthetic_raymap(F, H // 8, W // 8)
    pipe = _product_pipeline_with_oracle_modules()
    out = pipe(height=H, width=W, num_frames=F, generator=torch.Generator().manual_seed(42), **kw)
    for got, want, what in ((out.disparity, g["disparity"], "disparity"), (out.raymap, g["raymap"], "raymap"),
                            (subsample(out.rgb, (2, 2, 2, 1)), g["rgb_sub"], "rgb")):
        assert got.shape == want.shape, what
        mism = float((got != want).mean())
        rel = float(np.sqrt(((got.astype(np.float64) - want) ** 2).mean()) / np.sqrt((want.astype(np.float64) ** 2).mean()))
        print(f"{name} {what}: mismatching elements {mism:.2e}, rel-rms {rel:.2e}")
        assert mism <= 0.1 and rel <= 5e-3, (what, mism, rel)
    assert out.rgb.dtype == np.float32 and out.disparity.dtype == np.float32 and out.raymap.dtype == np.float32


def test_pipeline_error_messages_match_reference(golden_dir):
    g = np.load(golden_dir / "pipeline_errors.npz")
    H, W, F = TINY["height"], TINY["width"], TINY["num_frames"]
    video = synthetic_video(F, H, W)
    raymap = synthetic_raymap(F, H // 8, W // 8)
    pipe = _product_pipeline_with_oracle_modules()
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
        with pytest.raises(ValueError) as ei:
            pipe(**kw)
        assert str(ei.value) == str(g[k]), k


# ------------------------------------------------------------------------------------------------ depth metrics (8f rank 4)
def test_depth_evaluation_matches_reference(golden_dir, tmp_path):
    """aether_b200.depth_eval.depth_evaluation against evaluation/video_depth/tools.py:179-470 run by the reference
    itself (tests/golden/make_golden.py::make_depth_eval): every alignment eval_depth.py selects, the disparity-space /
    edge-mask / custom-mask options, and the `frame_%04d.npy` round trip of launch_aether.py:364-365."""
    import sys
    sys.path.insert(0, str(golden_dir))
    from make_golden import DEPTH_EVAL_MODES
    from aether_b200.depth_eval import depth_evaluation, evaluate_depth_sequence, save_depth_frames
    from helpers import depth_eval_case
    g = np.load(golden_dir / "depth_eval.npz")
    pred, gt, mask = depth_eval_case()
    for name, kw in DEPTH_EVAL_MODES.items():
        kw = dict(kw)
        cm = mask if kw.pop("use_mask", False) else None
        res, err, full, gt_full = depth_evaluation(pred.copy(), gt.copy(), custom_mask=cm, **kw)
        keys = sorted(res)
        assert keys == [str(k) for k in g[f"{name}__keys"]]
        # identical torch / numpy operations on identical inputs; the Adam-fitted mode goes through 200 float64 updates
        tol = 1e-9 if name != "scale_shift_lad" else 1e-6
        np.testing.assert_allclose([float(res[k]) for k in keys], g[f"{name}__vals"], rtol=tol, atol=1e-12, err_msg=name)
        assert err.double().sum().item() == pytest.approx(float(g[f"{name}__err_sum"]), rel=tol)
        assert full.double().sum().item() == pytest.approx(float(g[f"{name}__full_sum"]), rel=tol)
        assert err.shape == gt_full.shape == (pred.shape[0] * pred.shape[1], pred.shape[2])
    # writer -> reader round trip: np.save per frame, evaluated with the `--align scale&shiftl2` selection
    depth = np.clip(1.0 / np.maximum(pred, 1e-3), 0, 1e2)
    assert save_depth_frames(str(tmp_path / "seq"), depth) == pred.shape[0]
    assert sorted(p.name for p in (tmp_path / "seq").iterdir()) == [f"frame_{i:04d}.npy" for i in range(pred.shape[0])]
    back = evaluate_depth_sequence(str(tmp_path / "seq"), list(gt), align="scale&shiftl2")
    direct = depth_evaluation(depth, gt, max_depth=70, post_clip_max=70, align_with_lstsq=True)[0]
    assert back == direct
