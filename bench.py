#!/usr/bin/env python
"""bench.py -- headline metric of BASELINE.json: latent-frames/sec for a 41x480x720 50-step generation at 1/2/4/8 B200,
measured on the path `north_star` shards: the tile-parallel sliding-window evaluation.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR

--dump-outputs DIR: after the K timed rounds the blend rank writes what the last timed round computed as DIR/<name>.npy
(see `dump_outputs`), so that two builds of the project can be compared output for output on identical seeded inputs.

Workload.  A synthetic clip in the geometry of BASELINE.json configs[4] (480 x 853 frames -> two 480 x 720 spatial
tiles per 41-frame temporal window, stride 8; reference evaluation/video_depth/launch_aether.py:81-287) is evaluated by
`aether_b200.sliding_window.TileParallelRun`.  Its tiles are dealt round-robin over the N ranks and processed in
ROUNDS; one bench "step" = one round:

    every rank runs ONE tile = one configs[1] generation (reconstruction, 41 frames 480x720 -> 11x60x90 latents,
    S = 15076 tokens, 50 DPM steps, batch 1, bf16) through the full AetherV1PipelineCogVideoX.__call__ (VAE encode,
    50 x (DiT forward + fused CFG/DPM step), rgb + disparity VAE decodes), the round's N - 1 remote disparity tiles
    travel peer to peer (NCCL over NVLink) to the blend rank, and the blend chain there (spatial cross-fade + temporal
    chain with the masked-LSQ scale, K10 kernels) advances by the windows that became complete.

At N = 1 a step is therefore exactly one configs[1] generation (plus its share of the blend); the clip grows with N
(one tile per rank per round) => "scaling": "weak"; value = N * 11 latent frames * K / seconds.
  value : tile crops already resident in HBM, CUDA events around exactly K rounds, max over ranks.
  e2e   : the same round with HOST buffers: the tile's frames are host numpy uint8 (a decoded video), uploaded inside the
          timed region (the reference's prepare_input would turn them into float64 on the host first,
          launch_aether.py:388-403; same values, 8x the bytes), and the frames of the blended disparity that became
          final in the round are copied back to host numpy.
  collective_ms / blend_ms : device-timed inside the timed rounds (blend rank), reported per round.
  config5_4step : the reference's own evaluation setting (4 denoise steps per tile, launch_aether.py:67-70) on a
          FIXED 8-tile clip at every N (strong scaling): seconds for the whole evaluate (tiles + exchange + blend +
          D2H), with the exchange / blend / D2H parts separated -- the regime where the VAE and the blend matter.
  roofline : the attention kernel (dominant), duration from CUDA events recorded around every attention launch on
          the launching stream inside the timed region; algorithmic flop = 4*B*H*S^2*64 per launch.
  gpu_library_baseline (N = 1): the same DiT forward through stock PyTorch (bf16 oracle modules on the GPU: cuDNN /
          flash SDPA + cuBLAS + eager elementwise kernels) -- what the reference's diffusers path would execute on this
          B200; outside the timed region, for context.
  cpu_baseline / --impl reference : the reference's CPU path = the fp32 torch restatement of the diffusers modules
          (oracle/), timed on the host cores on a bounded sample (two transformer blocks of one forward at full S plus
          embed/tail, median of three samples) and extrapolated x42 layers x50 steps.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True      # the benchmark may run from a read-only tree: no __pycache__ there

LATENT_FRAMES, LAT_H, LAT_W = 11, 60, 90
TEXT_LEN, TEXT_DIM = 226, 4096
HEADS, LAYERS = 48, 42
S_TOKENS = TEXT_LEN + LATENT_FRAMES * (LAT_H // 2) * (LAT_W // 2)
DENOISE_STEPS = 50
CLIP_H, CLIP_W, WINDOW, STRIDE_T = 480, 853, 41, 8
METRIC = "latent-frames/sec, 41x480x720 50-step generation (tile-parallel sliding-window evaluation)"
WORKLOAD = ("sliding-window evaluation rounds (configs[4] geometry: 480x853 clip, 2 spatial tiles x 41-frame windows, "
            "stride 8); per round every rank runs one configs[1] tile (reconstruction, 41 frames 480x720 -> 11x60x90 "
            "latents, S=15076, 50 steps, batch 1) through the full pipeline, NCCL p2p exchange to the blend rank, "
            "blend chain advance")


def bench_config(world: int, tile_steps: int, steps: int, warmup: int, attention_mode: int = 5) -> dict:
    """The `config` object of the JSON line -- identical for the product arm and the `--impl reference` arm."""
    n_e2e = 1 + ((warmup + steps + 1) * world) % 2
    cfg = {"workload": WORKLOAD,
           "model": "AetherV1 DiT geometry (42 layers, 48x64, in 96 / out 56) + CogVideoX-5b VAE geometry, seeded synthetic "
                    "weights",
           "denoise_steps": tile_steps, "tokens": S_TOKENS, "attention_mode": attention_mode, "tiles_per_round": world,
           "clip_frames": clip_frames_for_tiles((warmup + steps + n_e2e) * world),
           "parallelism": f"tile-parallel x{world}: round-robin tiles, NCCL p2p of the disparity tiles to the blend rank "
                          f"each round, streaming blend chain on rank 0",
           "l2": "per-step working set (11.1 GB weights + ~1.4 GB activations) >> 126 MB L2; no explicit flush"}
    if tile_steps != DENOISE_STEPS:
        cfg["INVALID_FOR_HEADLINE"] = f"--tile-steps {tile_steps} (development run; the metric needs 50)"
    return cfg


def clip_frames_for_tiles(n_tiles: int) -> int:
    n_windows = (n_tiles + 1) // 2
    return WINDOW + STRIDE_T * (n_windows - 1)


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1400.0, "fallback (B200_PROFILING.md sustained 1.4 PFLOP/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for n, v in zip(names, r[5:9]):
                if "Active" in v and "Not" not in v:
                    reasons.add(n)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------ CPU reference
def _physical_cores() -> int:
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return os.cpu_count() or 1


def cpu_reference_sample(n_samples: int = 3, k_layers: int = 2):
    """k transformer blocks (+ embed and tail) of one forward at full S on the host cores, fp32 oracle.  One thread per
    PHYSICAL core (SMT siblings only add noise to an fp32 GEMM), affinity left to the OS, median over the samples."""
    import torch
    from oracle.dit import DiTConfig, OracleDiT
    from oracle.rope import prepare_rotary_positional_embeddings
    threads = _physical_cores()
    torch.set_num_threads(threads)
    cfg = DiTConfig(num_layers=k_layers)
    torch.manual_seed(0)
    model = OracleDiT(cfg).eval()
    x = torch.randn(1, LATENT_FRAMES, 96, LAT_H, LAT_W)
    e = torch.randn(1, TEXT_LEN, TEXT_DIM) * 0.2
    cos, sin = prepare_rotary_positional_embeddings(480, 720, LATENT_FRAMES)
    ts = torch.tensor([999])
    full, rest = [], []
    with torch.no_grad():
        model(x, e, ts, image_rotary_emb=(cos, sin), n_layers=0)          # page in / thread-pool warm-up, untimed
        for _ in range(n_samples):
            t0 = time.perf_counter()
            model(x, e, ts, image_rotary_emb=(cos, sin))
            full.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            model(x, e, ts, image_rotary_emb=(cos, sin), n_layers=0)
            rest.append(time.perf_counter() - t0)
    t_full, t_rest = statistics.median(full), statistics.median(rest)
    t_layer = max(t_full - t_rest, 1e-9) / k_layers
    t_forward = LAYERS * t_layer + t_rest
    value = LATENT_FRAMES / (DENOISE_STEPS * t_forward)
    return dict(value=value, t_layer_s=t_layer, t_embed_tail_s=t_rest, t_forward_extrapolated_s=t_forward,
                threads=threads, samples_s=[round(v, 3) for v in full], k_layers=k_layers,
                cpu_work_s=sum(full) + sum(rest))


def cpu_baseline_dict(r, kind="port"):
    return {"value": r["value"], "unit": "latent-frames/s", "cores": r["threads"], "kind": kind,
            "sample": (f"{r['k_layers']} of {LAYERS} transformer blocks + embed/tail of ONE forward at full S={S_TOKENS} "
                       f"(fp32 torch restatement of the diffusers modules; {len(r['samples_s'])} samples {r['samples_s']} s, "
                       f"median -> {r['t_layer_s']:.2f} s/block on {r['threads']} threads = physical cores), extrapolated "
                       f"x{LAYERS} layers x{DENOISE_STEPS} steps; VAE and blend of the round NOT included (favours the CPU "
                       f"arm); diffusers itself is not installable here")}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_sample(n_samples=3, k_layers=2)
    ms_per_step = r["t_forward_extrapolated_s"] * DENOISE_STEPS * 1000.0          # one round = one 50-step generation
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "latent-frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args.gpus, args.tile_steps, args.steps, max(args.warmup, 3),
                                   int(os.environ.get("AETHER_ATTENTION_MODE", "5"))),
            "reference_detail": {"device": "host CPU", "samples_timed": len(r["samples_s"]), "extrapolated": True},
            "cpu_baseline": cpu_baseline_dict(r),
            "e2e": {"value": r["value"], "unit": "latent-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ product arm
class SyntheticClip:
    """Stands in for the [1, T, H, W, 3] float64 array of launch_aether.prepare_input without holding T x 9.8 MB of
    host memory: crops are generated per tile, seeded by the tile position, either resident on the device (float32,
    `value` rounds) or as host numpy uint8 frames in page-locked memory (`e2e` rounds)."""

    def __init__(self, t, h, w, device):
        self.shape = (1, t, h, w, 3)
        self.device = device
        self.host_mode = False
        self._cache = {}

    def __getitem__(self, idx):
        import numpy as np
        import torch
        _, ts, hs, ws, _ = idx
        n, hh, ww = ts.stop - ts.start, hs.stop - hs.start, ws.stop - ws.start
        seed = ts.start * 1000 + ws.start
        key = (n, hh, ww)
        if self.host_mode:              # one host crop per shape, generated OUTSIDE the timed region (prepare_host)
            if ("host",) + key not in self._cache:
                pinned = torch.empty((n, hh, ww, 3), dtype=torch.uint8).pin_memory()      # numpy view of pinned memory
                arr = pinned.numpy()
                arr[...] = np.random.default_rng(seed).integers(0, 256, (n, hh, ww, 3), dtype=np.uint8)
                self._cache[("host",) + key] = (arr, pinned)
            return self._cache[("host",) + key][0]
        if key not in self._cache:      # one resident crop per shape: "inputs already resident in HBM"
            g = torch.Generator(device=self.device).manual_seed(seed)
            self._cache[key] = torch.rand((n, hh, ww, 3), device=self.device, generator=g, dtype=torch.float32)
        return self._cache[key]


DUMP_SAMPLE = 1 << 21          # elements kept of a larger output: the four outputs stay well under 64 MB together
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays: dict) -> None:
    """Write every array of `arrays` (name -> numpy array or torch tensor) as <out_dir>/<name>.npy: float64 stays float64,
    everything else becomes float32.  An array of more than DUMP_SAMPLE elements is replaced by the DUMP_SAMPLE elements
    of its flattened form at a fixed seeded set of indices (ascending order, seed 0: the same positions in every run and
    every build)."""
    import numpy as np
    import torch
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        if isinstance(a, np.ndarray):
            a = a.astype(np.float64 if a.dtype == np.float64 else np.float32, copy=False)
        else:
            a = a.detach().to(a.dtype if a.dtype == torch.float64 else torch.float32).cpu().numpy()
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        total += a.nbytes
        if total > DUMP_MAX_BYTES:
            raise ValueError(f"--dump-outputs: more than {DUMP_MAX_BYTES} bytes of outputs")
        np.save(out_dir / f"{name}.npy", a)


def gpu_library_forward_ms(dev, reps: int = 3):
    """One DiT forward at the bench shape through stock PyTorch (oracle modules in bf16 on the GPU)."""
    import torch
    from oracle.dit import DiTConfig, OracleDiT
    from oracle.rope import prepare_rotary_positional_embeddings
    with torch.device(dev):
        model = OracleDiT(DiTConfig()).to(torch.bfloat16).eval()
    g = torch.Generator(device=dev).manual_seed(0)
    with torch.no_grad():
        for p in model.parameters():
            p.copy_(torch.randn(p.shape, device=dev, generator=g, dtype=torch.float32) * 0.02)
    x = torch.randn(1, LATENT_FRAMES, 96, LAT_H, LAT_W, device=dev, generator=g).bfloat16()
    e = (torch.randn(1, TEXT_LEN, TEXT_DIM, device=dev, generator=g) * 0.2).bfloat16()
    cos, sin = prepare_rotary_positional_embeddings(480, 720, LATENT_FRAMES)
    cos, sin = cos.to(dev), sin.to(dev)
    ts = torch.tensor([999], device=dev)
    times = []
    with torch.no_grad():
        for i in range(reps + 1):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            model(x, e, ts, image_rotary_emb=(cos, sin))
            b.record()
            torch.cuda.synchronize()
            if i:
                times.append(a.elapsed_time(b))
    del model
    torch.cuda.empty_cache()
    return statistics.median(times)


def gpu_library_leg(dev, model, pipe, text):
    """One DiT forward (B=1, S=15076, 42 layers): stock PyTorch bf16 vs this library, CUDA events, median of 3."""
    import torch
    out = {"dit_forward_ms": gpu_library_forward_ms(dev), "ours_dit_forward_ms": None,
           "what": "one CogVideoX DiT forward (B=1, S=15076, 42 layers) through stock PyTorch bf16 on this GPU "
                   "(F.scaled_dot_product_attention + cuBLAS + eager elementwise): the device work the reference's "
                   "diffusers path would launch; outside the timed region, not power-capped like the timed rounds"}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g = torch.Generator(device=dev).manual_seed(5)
    lat = torch.randn(1, LATENT_FRAMES, 96, LAT_H, LAT_W, device=dev, generator=g).bfloat16()
    rope = pipe._prepare_rotary_positional_embeddings(480, 720, LATENT_FRAMES, dev, fps=12)
    tt = torch.tensor([999], device=dev)
    txt = text.to(dev).bfloat16()
    ours = []
    for i in range(4):
        a.record()
        model(lat, txt, tt, image_rotary_emb=rope)
        b.record()
        torch.cuda.synchronize()
        if i:
            ours.append(a.elapsed_time(b))
    out["ours_dit_forward_ms"] = statistics.median(ours)
    return out


def run_product(args):
    import numpy as np
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # stdout carries exactly one JSON line: NCCL's own banner / debug lines (NCCL_DEBUG=VERSION|WARN|INFO) go to stderr
        if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
            os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as ge
    from aether_b200 import _lib
    if not _lib.lib_path().exists():
        ge.build()
    from aether_b200.pipeline import AetherV1PipelineCogVideoX
    from aether_b200.scheduler import AetherDPMScheduler
    from aether_b200.sliding_window import TileParallelRun, process_with_sliding_window
    from aether_b200.transformer import AetherTransformer3D
    from aether_b200.vae import AetherVAE

    model = AetherTransformer3D(device=dev)
    model.init_synthetic_(seed=0)
    model.pack(release_unpacked=True)
    vae = AetherVAE(device=dev)
    vae.init_synthetic_(seed=1)
    vae.enable_slicing()
    vae.enable_tiling()
    text = torch.randn(1, TEXT_LEN, TEXT_DIM, generator=torch.Generator().manual_seed(3)) * 0.2
    pipe = AetherV1PipelineCogVideoX(vae=vae, scheduler=AetherDPMScheduler(), transformer=model,
                                     empty_prompt_embeds=text).to(dev)
    tile_steps = args.tile_steps
    warmup = max(args.warmup, 3)
    n_e2e = 1 + ((warmup + args.steps + 1) * world) % 2         # keeps the tile count even (two tiles per window)
    rounds = warmup + args.steps + n_e2e
    clip = SyntheticClip(clip_frames_for_tiles(rounds * world), CLIP_H, CLIP_W, dev)
    stats = {}
    last_tile = []          # --dump-outputs: what the pipeline call of this rank's latest tile returned

    def tile_pipe(*a, **kw):
        last_tile[:] = [pipe(*a, **kw)]
        return last_tile[0]

    # the evaluation decodes rgb for every tile like the reference (skip_unused_rgb=False): a round is a complete
    # configs[1] generation, nothing of it is skipped
    run = TileParallelRun(tile_pipe if args.dump_outputs else pipe, clip, tile_steps, clip.shape[1], seed=3407,
                          rank=rank, world_size=world, device=dev, skip_unused_rgb=False, stats=stats)
    assert run.n_rounds == rounds, (run.n_rounds, rounds)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    calls0 = _lib.CALLS[0]
    for j in range(warmup):
        run.run_round(j)
    torch.cuda.synchronize()
    calls_per_round = (_lib.CALLS[0] - calls0) / warmup
    run.finish_stats_reset()

    # ---- timed region: exactly K rounds
    model.enable_timing(True)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    attn_ms = attn_n = 0
    ev0.record()
    for j in range(warmup, warmup + args.steps):
        run.run_round(j)
        if j == warmup + args.steps - 1:
            ev1.record()
        torch.cuda.current_stream().synchronize()         # the host loop of the evaluation is synchronous per tile
        ms, n = model.read_attention_timing()             # attention launches of the round's last denoise step
        attn_ms, attn_n = attn_ms + ms, attn_n + n
    barrier()
    elapsed_ms = max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop() if sampler else None
    model.enable_timing(False)
    run.collect_stats()
    timed_stats = dict(stats)
    run.finish_stats_reset()
    value = world * LATENT_FRAMES * args.steps * (tile_steps / DENOISE_STEPS) / (elapsed_ms / 1000.0)
    if args.dump_outputs and rank == 0:
        # the last timed round: the pipeline outputs of its tile on this rank, and the blended disparity frames that
        # no later window changes any more (what fetch_finalized hands a caller; the e2e rounds push more windows)
        rgb, disp, ray = last_tile[0]
        upto = run.plan.tiles[run.blend.windows_done * run.plan.n_spatial].t_start
        dump_outputs(args.dump_outputs, {"tile_rgb": rgb, "tile_disparity": disp, "tile_raymap": ray,
                                         "blended_disparity": run.blend.final[:upto]})

    # ---- e2e: the same round with host buffers (host uint8 frames in pinned memory in, finalised blended frames out)
    clip.host_mode = True
    clip[0, 0:WINDOW, 0:480, 0:720, :]                      # generate the synthetic host crop before the timed region
    pinned = (torch.empty((WINDOW + STRIDE_T * world, CLIP_H, CLIP_W), dtype=torch.float64).pin_memory()
              if rank == 0 else None)
    run.fetch_finalized(discard=True)                      # frames finalised before the e2e rounds are not counted
    h2d = WINDOW * 480 * 720 * 3              # uint8 frames of the tile
    d2h = 0
    barrier()
    t0 = time.perf_counter()
    for j in range(warmup + args.steps, rounds):
        run.run_round(j)
        got = run.fetch_finalized(pinned)
        if got is not None:
            d2h += got[1].nbytes
    torch.cuda.synchronize()
    e2e_s = max_over_ranks((time.perf_counter() - t0) * 1000.0) / 1000.0
    e2e = {"value": world * LATENT_FRAMES * n_e2e * (tile_steps / DENOISE_STEPS) / e2e_s, "unit": "latent-frames/s",
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(d2h / n_e2e), "seconds_per_round": e2e_s / n_e2e,
           "rounds": n_e2e,
           "scope": "one round through the public API with HOST buffers: host numpy uint8 frames [41,480,720,3] -> "
                    "AetherV1PipelineCogVideoX.__call__ (upload, /255 + layout + 2x-1 + bf16 in one kernel, VAE encode, "
                    "50 x (DiT + DPM step), rgb + disparity VAE decode) -> NCCL p2p exchange -> blend chain -> D2H of the "
                    "frames finalised by the round (bytes per round, blend rank)"}
    run.finish()                                           # complete the chain (last window already pushed)
    clip.host_mode = False

    # ---- configs[4] at its own setting (4 denoise steps per tile), fixed 8-tile clip at every N: strong scaling
    strong = None
    if not args.no_strong_leg:
        sclip = SyntheticClip(clip_frames_for_tiles(8), CLIP_H, CLIP_W, dev)
        sclip.host_mode = True
        sclip[0, 0:WINDOW, 0:480, 0:720, :]
        sstats = {}
        barrier()
        t0 = time.perf_counter()
        _, disp = process_with_sliding_window(pipe, sclip, 4, sclip.shape[1], 3407, rank=rank, world_size=world,
                                              device=dev, stats=sstats)
        torch.cuda.synchronize()
        s_s = max_over_ranks((time.perf_counter() - t0) * 1000.0) / 1000.0
        strong = {"tiles": 8, "frames": sclip.shape[1], "denoise_steps_per_tile": 4, "seconds": s_s,
                  "value": 8 * LATENT_FRAMES / s_s, "unit": "latent-frames/s (4-step tiles)", "scaling": "strong",
                  "blend_rank_ms": {k: round(v, 3) for k, v in sstats.items() if k.endswith("_ms")},
                  "scope": "evaluate one 65-frame 480x853 clip end to end (host uint8 frames in, blended fp64 disparity out "
                           "on the blend rank): 8 tiles over N ranks, rgb decode skipped for tiles whose rgb the reference "
                           "discards"}

    # ---- correctness of the exchange + blend at THIS world size: the reference's 24-tile golden chain (129 frames of
    # 480 x 853, tests/golden/sliding_long.npz, produced by the reference's process_with_sliding_window) through the same
    # tile-parallel engine with the golden's deterministic stand-in tiles; checked on the blend rank.
    xcheck = None
    gpath = ROOT / "tests" / "golden" / "sliding_long.npz"
    if not args.no_exchange_check and gpath.exists():
        sys.path.insert(0, str(ROOT / "tests"))
        from helpers import fake_tile_outputs, subsample, synthetic_long_clip
        gold = np.load(gpath)
        t_, h_, w_ = gold["thw"].tolist()
        obs = synthetic_long_clip(t_, h_, w_)
        _, disp = process_with_sliding_window(
            None, obs, 4, t_, 3407, rank=rank, world_size=world, device=dev,
            tile_fn=lambda tl, crop: fake_tile_outputs(crop, tl.t_start, tl.h_start, tl.w_start))
        if rank == 0:
            ok = bool(np.allclose(subsample(disp, (3, 16, 16)), gold["disparity_sub"], rtol=2e-6, atol=0)
                      and abs(disp.sum() - float(gold["disparity_sum"])) <= 2e-6 * abs(float(gold["disparity_sum"])))
            xcheck = {"golden": "tests/golden/sliding_long.npz (24 tiles, reference-generated)", "world_size": world,
                      "matches_rtol_2e-6": ok}

    if rank == 0:
        try:          # launches inside the native VAE calls (each counted once in _lib.CALLS): 1 encode + 2 decodes per tile
            vae_extra = 0 if vae.per_op else ((vae.launches(0, WINDOW, 480, 720) - 1) + 2 * (vae.launches(1, LATENT_FRAMES, LAT_H, LAT_W) - 1))
        except Exception:
            vae_extra = 0
        peak, peak_src = _peaks()
        flop = 4.0 * 1 * HEADS * float(S_TOKENS) ** 2 * 64
        avg_ms = attn_ms / max(attn_n, 1)
        achieved = flop / (avg_ms / 1000.0) / 1e12 if attn_n else None
        traffic = None
        prof = ROOT / "profiles" / "attention_traffic.json"
        if prof.exists():
            traffic = json.loads(prof.read_text()).get("dram_bytes_per_launch")
        ms_per_step = elapsed_ms / args.steps
        per_round = lambda k: round(timed_stats.get(k, 0.0) / args.steps, 3)
        line = {
            "metric": METRIC, "value": value, "unit": "latent-frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": bench_config(world, tile_steps, args.steps, warmup, int(model.attention_fp16_pv)),
            "e2e": e2e,
            "collective_ms": per_round("collective_ms"), "blend_ms": per_round("blend_ms"),
            "tile_ms": per_round("tile_ms"),
            "collective_note": "per round on the blend rank; includes waiting for the slowest rank's tile of the round",
            "gpu_launches": int(round(calls_per_round + tile_steps * (model.launches_per_forward(1) - 1) + vae_extra)) * args.steps,
            "gpu_launches_note": "per round: C-ABI calls counted live + (kernels per DiT forward - 1) x denoise steps + the kernels "
                                 "and device copies the three native VAE calls enqueue beyond their own call (dry-run count of "
                                 "aether_vae_encode / aether_vae_decode); x timed rounds",
            "clocks": clocks,
            "roofline": {"kernel": f"aether_attention_bf16 mode {int(model.attention_fp16_pv)} (tcgen05)",
                         "bound": "tensor", "achieved": achieved, "peak": peak,
                         "unit": "TFLOP/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                         "peak_source": peak_src, "launches_timed": attn_n, "avg_launch_ms": avg_ms,
                         "share_of_step": (avg_ms * LAYERS * tile_steps / ms_per_step) if attn_n else None},
        }
        if strong is not None:
            line["config5_4step"] = strong
        if xcheck is not None:
            line["exchange_blend_check"] = xcheck
        if world == 1 and not args.no_gpu_library_baseline:
            try:                                      # context only: never lose the measured line over it
                line["gpu_library_baseline"] = gpu_library_leg(dev, model, pipe, text)
            except Exception as e:
                line["gpu_library_baseline"] = {"error": f"{type(e).__name__}: {e}"}
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_baseline_dict(cpu_reference_sample(3, 2))
            except Exception as e:
                line["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="product", choices=["product", "reference"])
    ap.add_argument("--tile-steps", type=int, default=DENOISE_STEPS,
                    help="denoise steps per tile (development only; the headline metric is defined at 50)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-library-baseline", action="store_true")
    ap.add_argument("--no-strong-leg", action="store_true", help="skip the fixed-clip 4-step strong-scaling leg")
    ap.add_argument("--no-exchange-check", action="store_true", help="skip the golden check of the exchange + blend")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed round as DIR/<name>.npy (float32/float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1 (the number of timed rounds)")
    if args.dump_outputs and args.impl != "product":
        ap.error("--dump-outputs needs --impl product (the reference arm computes no outputs)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
