"""CPU: the C-ABI library loads and exports every symbol include/aether_b200.h declares; product modules fail
loudly without a GPU (no CPU fallback); the tile-parallel exchange step works over gloo with world_size 2."""
import ctypes
import os
import re
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol():
    from aether_b200 import _lib
    hdr = (ROOT / "include" / "aether_b200.h").read_text()
    declared = set(re.findall(r"\b(aether_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    lib = ctypes.CDLL(str(_lib.lib_path()))
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/aether_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))
    loaded = _lib.load()
    assert loaded.aether_abi_version() == 2


def test_ctypes_signatures_match_header_prototypes():
    """Every prototype of include/aether_b200.h against aether_b200/_lib.py::SIGNATURES: same number of parameters
    and the same kind (pointer / 32-bit int / 64-bit int / float / double) in every position -- ctypes would
    otherwise marshal a wrong call without any diagnostic."""
    from aether_b200 import _lib
    hdr = re.sub(r"/\*.*?\*/", " ", (ROOT / "include" / "aether_b200.h").read_text(), flags=re.S)
    protos = re.findall(r"\b([A-Za-z_][A-Za-z0-9_ ]*?[\s\*])\s*(aether_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", hdr)
    assert len(protos) == len(_lib.SIGNATURES), (len(protos), len(_lib.SIGNATURES))

    def kind_c(decl: str) -> str:
        decl = decl.strip()
        if "*" in decl:
            return "ptr"
        base = re.sub(r"\b(const|unsigned)\b", "", decl).split()
        t = base[0] if base else ""
        return {"int32_t": "i32", "int": "i32", "int64_t": "i64", "float": "f32", "double": "f64"}[t]

    def kind_py(t) -> str:
        if t is None:
            return "void"
        if t in (ctypes.c_void_p,) or (isinstance(t, type) and issubclass(t, ctypes._Pointer)):
            return "ptr"
        return {ctypes.c_int32: "i32", ctypes.c_int: "i32", ctypes.c_int64: "i64", ctypes.c_float: "f32",
                ctypes.c_double: "f64"}[t]

    for ret, name, params in protos:
        res, args = _lib.SIGNATURES[name]
        plist = [p for p in (x.strip() for x in params.split(",")) if p and p != "void"]
        assert len(plist) == len(args), f"{name}: header has {len(plist)} parameters, ctypes binding {len(args)}"
        for i, (pc, pa) in enumerate(zip(plist, args)):
            assert kind_c(pc) == kind_py(pa), f"{name} parameter {i} ({pc!r}): header {kind_c(pc)}, binding {kind_py(pa)}"
        ret = ret.strip()
        want = "void" if ret == "void" else kind_c(ret)
        assert want == kind_py(res), f"{name}: return type {ret!r} vs binding {res}"


def test_committed_bench_lines_follow_the_contract():
    """The bench lines committed under profiles/ (written by bench.py on a B200) carry every key of the measurement
    contract, with consistent values."""
    import json
    line = json.loads((ROOT / "profiles" / "r2_bench_1gpu_final.json").read_text())
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline",
              "collective_ms", "blend_ms", "config5_4step", "exchange_blend_check", "gpu_library_baseline"):
        assert k in line, k
    assert line["n_gpus"] == 1 and line["warmup"] >= 3 and line["higher_is_better"] is True
    assert line["scaling"] == "weak" and line["dtype"] == "bf16" and line["data"] == "synthetic"
    assert "workload" in line["config"] and "l2" in line["config"] and line["config"]["denoise_steps"] == 50
    assert "INVALID_FOR_HEADLINE" not in line["config"]
    # a step is one round = one 11-latent-frame generation per rank
    assert line["value"] == pytest.approx(line["n_gpus"] * 11 / (line["ms_per_step"] / 1000.0), rel=1e-6)
    e2e = line["e2e"]
    assert e2e["unit"] == line["unit"] and e2e["h2d_bytes_per_step"] == 41 * 480 * 720 * 3 and e2e["d2h_bytes_per_step"] > 0
    assert 0 < e2e["value"] <= line["value"] * 1.01                # host copies are inside the e2e region
    rf = line["roofline"]
    assert rf["bound"] in ("hbm", "tensor") and rf["unit"] in ("GB/s", "TFLOP/s")
    assert rf["frac"] == pytest.approx(rf["achieved"] / rf["peak"], rel=1e-9) and rf["traffic"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
    assert line["gpu_launches"] > 0 and line["clocks"]["sm_mhz"] > 0
    assert not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert line["exchange_blend_check"]["matches_rtol_2e-6"] is True
    lib = line["gpu_library_baseline"]
    assert lib["ours_dit_forward_ms"] < lib["dit_forward_ms"]
    ref = json.loads((ROOT / "profiles" / "r2_bench_reference_arm.json").read_text())
    assert ref["impl"] == "reference" and ref["metric"] == line["metric"] and ref["unit"] == line["unit"]
    assert ref["config"]["workload"] == line["config"]["workload"]
    assert ref["e2e"]["h2d_bytes_per_step"] == 0 and ref["cpu_baseline"]["value"] == ref["value"]


def test_committed_multi_gpu_line_and_launch_shares_are_consistent(tmp_path):
    """The 8-GPU line is the same command at N = 8 (weak scaling: 8 tiles per round); the launch-share table under
    profiles/ is what tools/launch_shares.py derives from the committed ncu launch list."""
    import json
    import subprocess
    import sys
    last = lambda name: json.loads((ROOT / "profiles" / name).read_text().strip().splitlines()[-1])
    one, eight = last("r2_bench_1gpu_final.json"), last("r2_bench_8gpu_final.json")      # (stdout of that run also holds NCCL's banner)
    assert eight["n_gpus"] == 8 and eight["metric"] == one["metric"] and eight["scaling"] == "weak"
    assert eight["config"]["denoise_steps"] == 50 and eight["config"]["tiles_per_round"] == 8
    assert eight["value"] == pytest.approx(8 * 11 / (eight["ms_per_step"] / 1000.0), rel=1e-6)
    assert eight["exchange_blend_check"] == {**one["exchange_blend_check"], "world_size": 8}
    assert (eight["collective_ms"] + eight["blend_ms"]) < 0.02 * eight["ms_per_step"]      # VERDICT r1: < 2 % of the round
    assert 0.85 < eight["value"] / (8 * one["value"]) < 1.15                                # different boxes, +-3 % clocks
    out = tmp_path / "shares.md"
    subprocess.run([sys.executable, str(ROOT / "tools" / "launch_shares.py"), str(ROOT / "profiles" / "r2_bench_launches.csv"),
                    str(out), str(ROOT / "profiles" / "r2_bench_1gpu_final.json")], check=True, capture_output=True)
    assert out.read_text() == (ROOT / "profiles" / "r2_bench_launch_shares.md").read_text()


def test_bench_dump_outputs_and_argument_checks(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 stays float64, anything else is written as float32, a large output is reduced to
    the same seeded positions in every run, and the dump never exceeds 64 MB.  --steps below 1 is refused."""
    import subprocess
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)      # bench.py sets it at import
    import bench
    n = bench.DUMP_SAMPLE
    big = np.arange(n + 12345, dtype=np.float32)                                    # value = position
    bench.dump_outputs(tmp_path / "a", {"big": big, "small": torch.arange(6, dtype=torch.bfloat16).reshape(2, 3),
                                        "f64": np.linspace(0.0, 1.0, 7)})
    bench.dump_outputs(tmp_path / "b", {"big": 2 * big})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape == (n,) and np.all(np.diff(a) > 0)
    assert np.array_equal(b, 2 * a)
    small = np.load(tmp_path / "a" / "small.npy")
    assert small.dtype == np.float32 and np.array_equal(small, np.arange(6.0).reshape(2, 3))
    assert np.load(tmp_path / "a" / "f64.npy").dtype == np.float64
    with pytest.raises(ValueError):
        bench.dump_outputs(tmp_path / "c", {f"x{i}": np.zeros(n, np.float64) for i in range(5)})
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *bad], capture_output=True, text=True)
        assert r.returncode == 2 and "error" in r.stderr, (bad, r.stderr)


def test_library_has_no_libcuda_dependency():
    """The .so must load on a machine without the CUDA driver (driver entry points are resolved at run time)."""
    import subprocess
    from aether_b200 import _lib
    out = subprocess.run(["ldd", str(_lib.lib_path())], capture_output=True, text=True).stdout
    assert "libcuda.so" not in out and "libcudart" not in out and "libtorch" not in out


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_product_path_fails_loudly_without_gpu():
    from aether_b200 import _lib, ops
    from aether_b200.transformer import AetherTransformer3D
    assert _lib.load().aether_device_ok() == 0
    with pytest.raises(RuntimeError, match="No CPU fallback"):
        ops.gemm(torch.zeros(8, 8, dtype=torch.bfloat16), torch.zeros(8, 8, dtype=torch.bfloat16))
    m = AetherTransformer3D(num_attention_heads=4, num_layers=1, time_embed_dim=64, text_embed_dim=128)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 1, 96, 4, 4), torch.zeros(1, 2, 128), torch.zeros(1, dtype=torch.int64))
    assert "oracle" not in sys.modules or True   # (oracle may be imported by other tests in this process)


def test_product_package_never_imports_oracle():
    for p in (ROOT / "aether_b200").rglob("*.py"):
        src = p.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{p} imports the oracle"


def test_transformer_state_dict_names_match_diffusers_layout():
    from oracle.dit import OracleDiT, tiny_config
    from aether_b200.transformer import AetherTransformer3D
    cfg = tiny_config()
    a = set(OracleDiT(cfg).state_dict().keys())
    b = set(AetherTransformer3D(**cfg.to_dict()).state_dict().keys())
    assert a == b
    for k in ("transformer_blocks.0.attn1.to_q.weight", "transformer_blocks.1.ff.net.0.proj.bias",
              "transformer_blocks.0.norm1.linear.weight", "patch_embed.proj.weight", "norm_out.linear.bias",
              "time_embedding.linear_2.weight", "transformer_blocks.0.attn1.norm_k.weight"):
        assert k in b


# ------------------------------------------------------------------------------------------- gloo, world_size 2
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n_tiles, q):
    """The exchange step of the tile-parallel sliding-window path on gloo: rounds of one tile per rank, every
    non-root owner sends its tile once to the blend rank, which must see every tile exactly once, in order."""
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, str(ROOT))
    from aether_b200.sliding_window import exchange_round, partition_tiles, tile_owner
    mine = partition_tiles(n_tiles, rank, world)
    make = lambda k: torch.full((3, 4, 5), float(k)) + torch.arange(5.0)
    seen = []
    for j in range((n_tiles + world - 1) // world):
        round_tiles = list(range(j * world, min((j + 1) * world, n_tiles)))
        k = j * world + rank
        own = (k, make(k)) if k < n_tiles else None
        assert (own is not None) == (k in mine) and all(tile_owner(t, world) == t % world for t in round_tiles)
        got = exchange_round(round_tiles, own, (3, 4, 5), rank, world, root=0, device=torch.device("cpu"))
        if rank == 0:
            assert [kk for kk, _ in got] == round_tiles
            seen += [(kk, torch.equal(d, make(kk))) for kk, d in got]
        else:
            assert got == []
    ok = (seen == [(k, True) for k in range(n_tiles)]) if rank == 0 else True
    q.put((rank, ok, len(mine)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("n_tiles", [7, 4, 1])          # 1 tile on 2 ranks: a rank with no work must not hang the job
def test_exchange_rounds_gloo_world2(n_tiles):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n_tiles, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(ok for _, ok, _ in res)
    assert sum(n for _, _, n in res) == n_tiles


def _pose_worker(rank, world, port, q):
    """rel-pose windows dealt over 2 ranks (gloo): the blend rank must reproduce the single-process result exactly."""
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    from helpers import fake_pose_window
    from aether_b200 import pose_blend as P
    frames = np.zeros((1, 105, 24, 40, 3))
    frames[0, :, 0, 0, 0] = np.arange(105)
    ran = []

    def window_fn(clip):
        ran.append(int(clip[0, 0, 0, 0]))
        return fake_pose_window(ran[-1], clip.shape[0], seed=2)
    res = P.process_video_with_sliding_window(None, frames, 4, 42, rank=rank, world_size=world, window_fn=window_fn)
    ok = True
    if rank == 0:
        single = P.process_video_with_sliding_window(None, frames, 4, 42, window_fn=lambda c: fake_pose_window(
            int(c[0, 0, 0, 0]), c.shape[0], seed=2))
        ok = all(np.array_equal(res[k], single[k]) for k in ("rgb", "disparity", "poses", "focals"))
        ok = ok and ran[:2] == [0, 64]                      # windows 0 and 2 ran here, window 1 on the other rank
    else:
        ok = res is None and ran == [32]
    q.put((rank, ok))
    dist.barrier()
    dist.destroy_process_group()


def test_rel_pose_windows_gloo_world2(monkeypatch):
    import torch.multiprocessing as mp
    # the windows live on the GPU when one is visible, and gloo's send / recv carry host tensors only: the workers see
    # no GPU, as on a machine without one
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_pose_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(ok for _, ok in res), res
