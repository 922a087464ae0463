"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares; host logic (scheduler,
module tree, error conventions, representation packing, 2-rank gloo broadcast) — no kernel is launched here."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from motionclone_b200 import _lib, dist as mcdist  # noqa: E402
from motionclone_b200.guidance import schedule_set_timesteps  # noqa: E402
from motionclone_b200.pipeline import AnimationPipeline, DDIMScheduler  # noqa: E402
from motionclone_b200.synthetic import NOISE_SCHEDULER_KWARGS, UNET_SD15_CONFIG, UNET_TINY_CONFIG  # noqa: E402
from motionclone_b200.unet3d import UNet3DConditionModel  # noqa: E402
from oracle import mc_oracle as O  # noqa: E402


def test_library_exports_every_header_symbol():
    header = open(os.path.join(ROOT, "include", "motionclone_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(mc_[a-z0-9_]+)\s*\(", header)))
    assert declared, "no declarations parsed"
    lib = _lib.lib()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/motionclone_b200.h but not exported"
    assert sorted(_lib.EXPORTS) == declared
    assert lib.mc_abi_version() == 2


def test_ops_refuse_cpu_tensors():
    from motionclone_b200 import ops
    x = torch.randn(1, 4, 2, 8, 8).half()
    acp = O.alphas_cumprod()
    with pytest.raises(TypeError):
        ops.cfg_ddim_step(x, x, x, None, 7.5, acp[999], acp[987])
    with pytest.raises(TypeError):
        ops.temporal_attention_forward(torch.randn(1, 16, 4, 64).half(), torch.randn(1, 16, 4, 64).half(), None, 8, 0.35,
                                       want_o=False, want_probs=True)


def test_state_dict_keys_match_reference_module_tree():
    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_state_dict_shapes_tiny.json")))
    mine = {k: list(v.shape) for k, v in UNet3DConditionModel(**UNET_TINY_CONFIG).state_dict().items()}
    assert mine == ref
    with torch.device("meta"):
        sd15 = UNet3DConditionModel(**UNET_SD15_CONFIG)
    n = sum(p.numel() for p in sd15.parameters())
    assert abs(n - 1.31e9) < 0.1e9, n  # ~0.86 B SD1.5 UNet + ~0.45 B motion modules
    guided = [k for k, m in sd15.named_modules() if type(m).__name__ == "VersatileAttention" and "up_blocks.1" in k]
    assert guided == [f"up_blocks.1.motion_modules.{i}.temporal_transformer.transformer_blocks.0.attention_blocks.{j}"
                      for i in range(3) for j in range(2)]
    assert sum(type(m).__name__ == "VersatileAttention" for m in sd15.modules()) == 40


def test_scheduler_matches_oracle_and_error_conventions():
    s = DDIMScheduler(**NOISE_SCHEDULER_KWARGS)
    assert torch.equal(s.alphas_cumprod, O.alphas_cumprod())
    s.customized_set_timesteps = schedule_set_timesteps.__get__(s)
    s.customized_set_timesteps(50, 30, 0.4, device="cpu")
    assert list(s.timesteps_host) == list(O.uneven_timesteps(50, 30, 0.4)) == s.timesteps.tolist()
    with pytest.raises(ValueError):
        s.customized_set_timesteps(1001, 30, 0.4)
    with pytest.raises(ValueError):
        s.customized_set_timesteps(50, 30, 0.4, timestep_spacing_type="bogus")
    for kind in ("linspace", "leading", "trailing"):
        s.customized_set_timesteps(50, 0, 0.0, timestep_spacing_type=kind)
        assert len(s.timesteps_host) == 50


def test_pipeline_shell_contract():
    pipe = AnimationPipeline(unet=UNet3DConditionModel(**UNET_TINY_CONFIG), scheduler=DDIMScheduler(**NOISE_SCHEDULER_KWARGS))
    assert pipe.prepare_extra_step_kwargs(None, 0.0) == {"eta": 0.0, "generator": None}
    lat = pipe.prepare_latents(1, 4, 8, 64, 64, torch.float32, torch.device("cpu"), torch.Generator().manual_seed(0))
    assert lat.shape == (1, 4, 8, 8, 8)
    with pytest.raises(ValueError):
        pipe.prepare_latents(1, 4, 8, 64, 64, torch.float32, torch.device("cpu"), None, latents=torch.zeros(1, 4, 8, 4, 4))
    with pytest.raises(NotImplementedError):
        pipe._encode_prompt("x", torch.device("cpu"), 1, True, "")


def test_representation_pack_roundtrip():
    g = torch.Generator().manual_seed(0)
    rep = {f"m{i}": [torch.rand(16, 8, 16, 1, generator=g).half(), torch.randint(0, 16, (16, 8, 16, 1), generator=g).to(torch.uint8)]
           for i in range(6)}
    buf, manifest = mcdist.pack_representation(rep)
    assert buf.dtype == torch.uint8 and buf.numel() == 6 * 16 * 8 * 16 * 3
    back = mcdist.unpack_representation(buf, manifest)
    assert list(back) == list(rep)
    for k in rep:
        assert torch.equal(back[k][0], rep[k][0]) and torch.equal(back[k][1], rep[k][1])
    assert mcdist.shard_samples(8, 1, 4) == [1, 5] and mcdist.shard_samples(3, 2, 4) == [2]


_WORKER = r"""
import os, sys, torch
sys.path.insert(0, sys.argv[1])
from motionclone_b200 import dist as mcdist
rank, world, local = mcdist.init_from_env("gloo")
g = torch.Generator().manual_seed(0)
rep = None
if rank == 0:
    rep = {f"m{i}": [torch.rand(4, 8, 16, 1, generator=g).half(), torch.randint(0, 16, (4, 8, 16, 1), generator=g).to(torch.uint8)] for i in range(6)}
manifest = mcdist.representation_manifest([f"m{i}" for i in range(6)], 4, 8, 16)
assert mcdist.manifest_nbytes(manifest) == 6 * 4 * 8 * 16 * 3
got = mcdist.broadcast_representation(rep, torch.device("cpu"), manifest)
g2 = torch.Generator().manual_seed(0)
for i in range(6):
    v = torch.rand(4, 8, 16, 1, generator=g2).half(); ix = torch.randint(0, 16, (4, 8, 16, 1), generator=g2).to(torch.uint8)
    assert torch.equal(got[f"m{i}"][0], v) and torch.equal(got[f"m{i}"][1], ix)
assert mcdist.shard_samples(5, rank, world) == list(range(rank, 5, world))
print("rank", rank, "ok")
"""


def test_two_rank_gloo_broadcast(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1", MASTER_PORT="29613")
        procs.append(subprocess.Popen([sys.executable, str(script), ROOT], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        out, _ = p.communicate(timeout=120)
        assert p.returncode == 0, out.decode()


def test_bench_result_line_is_alone_on_stdout():
    """bench.py's contract is ONE JSON line on stdout; library banners written to fd 1 during the run (NCCL's version line)
    must end up on stderr."""
    import subprocess
    import sys as _sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import os, sys; sys.path.insert(0, %r); import bench; sys.stdout.flush(); bench._RESULT_FD = os.dup(1); "
            "os.dup2(2, 1); os.write(1, b'NCCL version x\\n'); print('python-level noise'); bench._emit({'a': 1})" % root)
    r = subprocess.run([_sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert r.stdout == '{"a": 1}\n'
    assert "NCCL version x" in r.stderr and "python-level noise" in r.stderr


def test_bench_dump_outputs_and_argument_checks(tmp_path):
    """bench.py --dump-outputs writes each returned array as DIR/<name>.npy in float32; --steps below 1 and a dump of
    the reference arm are refused before any work starts."""
    import bench
    lat = torch.randn(1, 4, 2, 8, 8).half()
    bench.dump_outputs(str(tmp_path / "out"), {"latents": lat, "latents_e2e": lat.float() * 2}, "_rank1")
    got = np.load(tmp_path / "out" / "latents_rank1.npy")
    assert got.dtype == np.float32 and np.array_equal(got, lat.float().numpy())
    assert np.load(tmp_path / "out" / "latents_e2e_rank1.npy").dtype == np.float32
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True,
                           timeout=300)
        assert r.returncode == 2 and r.stdout == "", r.stderr


def test_linear_into_residual_accumulates_in_place_only_without_grad():
    """spatial.linear_into_residual: the no-grad forwards accumulate the beta = 1 GEMM INTO the residual stream (no memcpy of
    the activation); under autograd the stream tensor is left untouched (it is saved by the LayerNorm that read it)."""
    import torch
    from motionclone_b200.spatial import linear_into_residual
    torch.manual_seed(0)
    lin = torch.nn.Linear(24, 16, bias=True)
    x = torch.randn(2, 5, 24)
    res = torch.randn(2, 5, 16)
    want = res + x @ lin.weight.t()  # the projection's bias is carried by the stream, not added here
    with torch.no_grad():
        r = res.clone()
        out = linear_into_residual(x, lin, r)
        assert out.data_ptr() == r.data_ptr()
        assert torch.allclose(out, want, atol=1e-5)
    r = res.clone().requires_grad_(True)
    out = linear_into_residual(x, lin, r)
    assert out.data_ptr() != r.data_ptr() and torch.equal(r.detach(), res)
    assert torch.allclose(out, want, atol=1e-5)
    out.sum().backward()
    assert torch.allclose(r.grad, torch.ones_like(res))


def test_exp2_polynomial_coefficients_accuracy():
    """csrc/tma_common.cuh ex2_poly_pair: the softmax kernels evaluate a quarter of their exponentials as
    2^round(x) * poly(x - round(x)) on the FMA pipe. The coefficients are read from the source and the fp32 arithmetic is
    replayed in numpy: max relative error vs 2^x must stay far below the fp16 rounding (4.9e-4) applied right after."""
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "motionclone_b200", "csrc", "tma_common.cuh")).read()
    body = src[src.index("ex2_poly_pair("):src.index("MC_EX2_POLY_PERIOD")]
    ks = {m.group(1): np.float32(m.group(2)) for m in re.finditer(r'"=l"\((k\d)\) : "f"\(([0-9.eE+-]+)f\)', body)}
    assert sorted(ks) == ["k0", "k1", "k2", "k3", "k4"]
    x = np.concatenate([np.linspace(-126, 8.5, 400001), np.linspace(-1, 1, 100001)]).astype(np.float32)
    magic = np.float32(12582912.0)
    t = (x + magic).astype(np.float32)
    n = (t - magic).astype(np.float32)
    f = (x - n).astype(np.float32)
    assert np.abs(f).max() <= 0.5
    p = np.full_like(f, ks["k4"])
    for k in ("k3", "k2", "k1", "k0"):
        p = (p * f + ks[k]).astype(np.float32)   # fma rounds once; two roundings here only loosen the bound
    bits = p.view(np.uint32) + (t.view(np.uint32) << np.uint32(23))
    got = bits.view(np.float32).astype(np.float64)
    want = np.exp2(x.astype(np.float64))
    rel = np.abs(got / want - 1.0).max()
    assert rel < 5e-6, rel


def test_fold_residual_biases_algebra():
    """spatial.fold_residual_biases: shifting the residual stream by the sum of a block's output biases and taking the
    remaining shift back out in front of every sub-block is the SAME function as adding each bias after its projection
    (attention.py:271-300). Checked in fp64 with arbitrary sub-block functions, including a missing bias."""
    import torch
    from motionclone_b200.spatial import fold_residual_biases
    torch.manual_seed(1)
    C = 12
    ws = [torch.randn(C, C, dtype=torch.float64) * 0.3 for _ in range(3)]
    fs = [lambda u, w=w: torch.tanh(u) @ w for w in ws]          # f_i: any function of the (un-shifted) stream
    for biases in ([torch.randn(C, dtype=torch.float64) for _ in range(3)],
                   [torch.randn(C, dtype=torch.float64), None, torch.randn(C, dtype=torch.float64)]):
        t = torch.randn(5, C, dtype=torch.float64)
        want = t
        for f, b in zip(fs, biases):
            want = want + f(want) + (b if b is not None else 0)
        shift, pre = fold_residual_biases(biases)
        s = t + shift                                              # what proj_in's folded bias produces
        for f, pb in zip(fs, pre):
            s = s + f(s + pb)                                      # beta = 1 GEMM into the stream; LN sees stream + pre_bias
        assert torch.allclose(s, want, atol=1e-12)
