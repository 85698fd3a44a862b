"""No-GPU checks: the C-ABI library loads and exports every symbol the header declares; the ctypes struct
mirrors the C struct; sampler host logic that needs no device; world_size-2 sharding over gloo."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib
from oracle import ds_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_header_symbol():
    lib = _lib.load()
    names = _lib.header_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), n
    assert set(names) == set(_lib._SIGNATURES), set(names) ^ set(_lib._SIGNATURES)
    assert lib.ds_version() >= 100


def test_struct_layout_matches_header(tmp_path):
    src = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "diffusynth_b200.h"
    int main(){ printf("%zu %zu %zu %zu %zu %zu\n", sizeof(ds_conv_gemm_args), offsetof(ds_conv_gemm_args, taps),
       offsetof(ds_conv_gemm_args, d_e2), offsetof(ds_conv_gemm_args, out_goff), offsetof(ds_conv_gemm_args, d_stats_out), offsetof(ds_conv_gemm_args, view_off)); return 0; }
    '''
    exe = str(tmp_path / "ds_layout_check")
    with open(exe + ".c", "w") as f:
        f.write(src)
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), exe + ".c", "-o", exe])
    got = [int(v) for v in subprocess.check_output([exe]).split()]
    A = _lib.ConvGemmArgs
    assert got == [C.sizeof(A), A.taps.offset, A.d_e2.offset, A.out_goff.offset, A.d_stats_out.offset, A.view_off.offset]


def test_module_level_struct_layouts_match_header(tmp_path):
    """The ctypes mirrors of the module-level structs (diffusynth_b200/engine.py) against the header, field by field at the ends that
    move when a field is added (ds_unet_config.batch_invariant, ds_vqgan_config.batch_invariant, the tail outputs of ds_sample_buffers)."""
    from diffusynth_b200 import engine
    src = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "diffusynth_b200.h"
    int main(){ printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n",
       sizeof(ds_unet_config), offsetof(ds_unet_config, up_dims), offsetof(ds_unet_config, n_label_class), offsetof(ds_unet_config, batch_invariant),
       sizeof(ds_vqgan_config), offsetof(ds_vqgan_config, attn_pos), offsetof(ds_vqgan_config, batch_invariant),
       sizeof(ds_sample_buffers), offsetof(ds_sample_buffers, d_wave),
       sizeof(ds_unet_plan_io), offsetof(ds_unet_plan_io, cond_launches)); return 0; }
    '''
    exe = str(tmp_path / "ds_layout_check")
    with open(exe + ".c", "w") as f:
        f.write(src)
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), exe + ".c", "-o", exe])
    got = [int(v) for v in subprocess.check_output([exe]).split()]
    U, V, S, P = engine.UnetConfig, engine.VqganConfig, engine.SampleBuffers, engine.UnetPlanIO
    assert got == [C.sizeof(U), U.up_dims.offset, U.n_label_class.offset, U.batch_invariant.offset,
                   C.sizeof(V), V.attn_pos.offset, V.batch_invariant.offset,
                   C.sizeof(S), S.d_wave.offset, C.sizeof(P), P.cond_launches.offset]


def test_invalid_arguments_fail_without_a_gpu():
    lib = _lib.load()
    assert lib.ds_ddim_step(None, None, None, None, None, None, 16, None) == -1
    assert b"ds_ddim_step" in lib.ds_last_error()
    a = _lib.ConvGemmArgs()
    assert lib.ds_conv_gemm(C.byref(a), None) == -1 and b"BK" in lib.ds_last_error()


def test_modify_rejects_a_guide_of_other_rows_before_the_device():
    from diffusynth_b200 import TextToTimbre
    pipe = TextToTimbre.__new__(TextToTimbre)
    pipe.channels, pipe.height = 4, 128
    cond = torch.zeros(2, 512)
    for guide in (torch.zeros(3, 4, 128, 64), torch.zeros(2, 3, 128, 64), torch.zeros(4, 128, 64)):
        with pytest.raises(ValueError):
            pipe.modify(guide, cond, None)


def test_noise_layout_column_map_matches_oracle():
    from diffusynth_b200.sampler import _column_map
    base = torch.arange(64).float().view(1, 1, 1, 64)
    for w in (17, 24, 63, 64, 65, 100, 144, 200):
        cols, pts = _column_map(w, 64)
        ref, ref_pts = O.noise_layout_repeat(base, 1, w)
        assert cols == [int(v) for v in ref.flatten()] and pts == ref_pts and len(cols) == w


def test_product_code_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "diffusynth_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            txt = open(os.path.join(pkg, f)).read()
            assert "import oracle" not in txt and "from oracle" not in txt and "/root/reference" not in txt, f


def test_two_rank_sharding_gloo():
    """N>1 path on CPU: contiguous shard ranges + the equal-count all-gather, world_size 2 over gloo."""
    code = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from diffusynth_b200.pipeline import shard_range, all_gather_waveforms
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["PORT"], rank=int(os.environ["RANK"]), world_size=2)
r = dist.get_rank()
total = 5
lo, hi = shard_range(total, r, 2)
local = torch.arange(lo, hi).float().view(-1, 1).repeat(1, 3)
out = all_gather_waveforms(local, total, 2)
assert out.shape == (5, 3) and torch.equal(out[:, 0], torch.arange(5).float()), out
print("rank", r, "ok")
''' % ROOT
    port = str(29500 + os.getpid() % 1000)
    procs = [subprocess.Popen([sys.executable, "-c", code], env=dict(os.environ, RANK=str(r), PORT=port), stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    for p in procs:
        out, _ = p.communicate(timeout=120)
        assert p.returncode == 0, out.decode()


def test_two_rank_chunked_gather_gloo():
    """configs[3] host logic on CPU: per-rank chunks submitted one by one, gathered into prompt order; uneven total (the last rank
    owns fewer prompts and pads), world_size 2 over gloo."""
    code = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from diffusynth_b200.pipeline import shard_range, ChunkGatherer
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["PORT"], rank=int(os.environ["RANK"]), world_size=2)
r = dist.get_rank()
total, chunk, L = 9, 2, 3
lo, hi = shard_range(total, r, 2)                       # rank 0: [0,5)  rank 1: [5,9)
g = ChunkGatherer(total, r, 2, chunk, L, "cpu")
assert g.n_chunks == 3 and g.per == 5
for k in range(g.n_chunks):
    ids = torch.arange(lo + k * chunk, min(lo + (k + 1) * chunk, hi)).float()
    w = torch.zeros((chunk, L)); w[:ids.numel()] = ids.view(-1, 1) + 100.0
    g.submit(k, w)
out = g.finish()
assert out.shape == (total, L) and torch.equal(out[:, 0], torch.arange(total).float() + 100.0), out
print("rank", r, "ok")
''' % ROOT
    port = str(30500 + os.getpid() % 1000)
    procs = [subprocess.Popen([sys.executable, "-c", code], env=dict(os.environ, RANK=str(r), PORT=port), stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    for p in procs:
        out, _ = p.communicate(timeout=120)
        assert p.returncode == 0, out.decode()


def test_shard_range_properties():
    from diffusynth_b200.pipeline import shard_range
    for total in (1, 5, 64, 1024, 1000):
        for world in (1, 2, 4, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))


def test_profiler_detection(monkeypatch):
    """Under Nsight Compute (which sets NV_COMPUTE_PROFILER_PERFWORKS_DIR for its children) the sampler asks the library for the
    eager form of the sampling graph: ncu 2025.2 dies on a cluster launch inside a stream capture."""
    from diffusynth_b200 import sampler
    monkeypatch.delenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR", raising=False)
    monkeypatch.delenv("CUDA_INJECTION64_PATH", raising=False)
    assert not sampler._profiler_attached()
    monkeypatch.setenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR", "/opt/nvidia/nsight-compute/2025.2.1/target/linux-desktop-glibc_2_11_3-x64/.")
    assert sampler._profiler_attached()
