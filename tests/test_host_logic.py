"""CPU: host-side logic — operand-image packing, C-ABI surface, module boundary behaviour."""
import ctypes
import os
import re

import pytest
import torch

import uformer_b200
from uformer_b200 import _lib, packing

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("N,K,nch,order", [(96, 32, 96, "nk"), (384, 128, 128, "nk"), (512, 2048, 128, "kn"), (64, 16, 64, "nk"), (32, 256, 32, "kn")])
def test_pack_roundtrip(N, K, nch, order):
    w = torch.randn(N, K)
    img = packing.pack_kmajor(w, nch, order)
    KB = (K + 63) // 64
    assert img.dtype == torch.bfloat16 and img.numel() == N * KB * 64
    back = packing.unpack_kmajor(img, N, K, nch, order)
    assert torch.equal(back, w.to(torch.bfloat16).float())


def test_pack_swizzle_matches_device_formula():
    """Element (n, k) of a chunk must sit at byte swz<128>(n, 2k) = (n*128 + 2k) ^ ((n & 7) << 4) (csrc/umma.cuh)."""
    nch = 16
    w = torch.arange(nch * 64, dtype=torch.float32).reshape(nch, 64) % 251
    img = packing.pack_kmajor(w, nch, "nk").reshape(-1).float()
    for n in range(nch):
        for k in range(64):
            lin = n * 128 + 2 * k
            off = lin ^ (((lin >> 7) & 7) << 4)
            assert img[off // 2] == w[n, k]


def test_pack_qkv_rows_and_scale():
    C, heads = 64, 2
    hd = C // heads
    wq, wkv = torch.randn(C, C), torch.randn(2 * C, C)
    bq, bkv = torch.randn(C), torch.randn(2 * C)
    img, bias = packing.pack_qkv(wq, bq, wkv, bkv, heads, 0.25)
    w = packing.unpack_kmajor(img, heads * 3 * hd, C, 3 * hd)
    assert torch.equal(w[3 * hd + hd:3 * hd + 2 * hd], wkv[hd:2 * hd].to(torch.bfloat16).float())          # k rows of head 1
    assert torch.equal(w[2 * hd:3 * hd], wkv[C:C + hd].to(torch.bfloat16).float())                           # v rows of head 0
    assert torch.equal(w[:hd], (wq[:hd] * 0.25).to(torch.bfloat16).float())
    assert torch.allclose(bias[:hd], bq[:hd] * 0.25) and torch.equal(bias[hd:2 * hd], bkv[:hd])


def test_pack_down_up_index_order():
    w = torch.randn(32, 16, 4, 4)
    wk = packing.unpack_kmajor(packing.pack_downsample(w, 32), 32, 256, 32, "kn")
    assert torch.equal(wk[:, (2 * 4 + 1) * 16 + 5], w[:, 5, 2, 1].to(torch.bfloat16).float())
    wu = torch.randn(64, 16, 2, 2)
    wn = packing.unpack_kmajor(packing.pack_upsample(wu, 64), 64, 64, 64, "nk")
    assert torch.equal(wn[(1 * 2 + 0) * 16 + 3], wu[:, 3, 1, 0].to(torch.bfloat16).float())


def test_c_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "lewin_b200.h")).read()
    declared = set(re.findall(r"\b(lw_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    lib = _lib.load()
    for s in declared:
        assert hasattr(lib, s), s
    assert lib.lw_abi_version() == 6
    # the ctypes mirrors have the compiled structs' sizes (also enforced at load time)
    for i, st in enumerate([_lib.WmsaArgs, _lib.Leff1Args, _lib.Leff2Args, _lib.LeffArgs, _lib.DownArgs, _lib.UpArgs, _lib.AdamWArgs]):
        assert lib.lw_struct_size(i) == ctypes.sizeof(st), st.__name__
    assert lib.lw_struct_size(99) == -1


def test_argument_validation_without_gpu():
    lib = _lib.load()
    a = _lib.WmsaArgs()
    assert lib.lw_wmsa_fwd(ctypes.byref(a), None) == -2          # NULL pointers
    b = _lib.DownArgs()
    assert lib.lw_downsample_fwd(ctypes.byref(b), None) == -2


def test_no_cpu_fallback_and_no_silent_training():
    blk = uformer_b200.LeWinTransformerBlock(32, (16, 16), 1, win_size=8, shift_size=0).eval()
    with pytest.raises(uformer_b200.EngineUnavailable):
        blk(torch.randn(1, 256, 32))
    att = uformer_b200.WindowAttention(32, (8, 8), 1)
    with pytest.raises(uformer_b200.EngineUnavailable):
        att(torch.randn(2, 64, 32))
    with pytest.raises(NotImplementedError):
        uformer_b200.LeWinTransformerBlock(32, (16, 16), 1, token_mlp='ffn')


def test_clamp_and_flops_surface():
    blk = uformer_b200.LeWinTransformerBlock(64, (8, 8), 2, win_size=8, shift_size=4)
    assert blk.shift_size == 0 and blk.win_size == 8               # model.py:863-865
    T = 16 * 16
    blk = uformer_b200.LeWinTransformerBlock(32, (16, 16), 1, win_size=8)
    expect = 2 * 32 * T + (3 * T * 32 * 32 + 2 * (T / 64) * 64 * 32 * 64 + T * 32 * 32) + (2 * T * 32 * 128 + T * 128 * 9)
    assert blk.flops() == expect


def test_pack_cache_invalidation():
    att = uformer_b200.WindowAttention(32, (8, 8), 1)
    p1 = att.packed()
    assert att.packed() is p1
    with torch.no_grad():
        att.proj.weight.add_(1.0)
    assert att.packed() is not p1


def test_pack_roundtrip_property():
    """hypothesis: pack/unpack is the identity on bf16-representable matrices for every legal (N, K, nch, order)."""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=25, deadline=None, derandomize=True)
    @given(nchunks=st.integers(1, 4), nch=st.sampled_from([16, 32, 48, 64, 96, 128, 256]), k=st.sampled_from([16, 32, 64, 96, 128, 320]),
           order=st.sampled_from(["nk", "kn"]), seed=st.integers(0, 2 ** 16))
    def run(nchunks, nch, k, order, seed):
        g = torch.Generator().manual_seed(seed)
        w = torch.randn(nchunks * nch, k, generator=g).to(torch.bfloat16).float()
        img = packing.pack_kmajor(w, nch, order)
        assert torch.equal(packing.unpack_kmajor(img, nchunks * nch, k, nch, order), w)
        # zero padding of K up to a multiple of 64 really is zero in the image
        assert img.float().abs().sum().item() == pytest.approx(w.abs().sum().item(), rel=1e-6)

    run()


def test_batched_prepack_is_bit_identical_to_lazy_packing():
    """uformer_b200.prepack.prepack(net): one permutation per (stage, weight kind) == per-module packing, and the
    modules' caches are hit afterwards."""
    from uformer_b200 import modules as M
    from uformer_b200.prepack import prepack
    from paramgen import randomize_state
    for cfg in [dict(img_size=128, embed_dim=16, depths=[2, 1, 2, 1, 2, 1, 2, 1, 2], win_size=8, modulator=True),
                dict(img_size=128, embed_dim=32, depths=[1, 2, 1, 1, 1, 1, 1, 2, 1], win_size=8, modulator=True),
                dict(img_size=128, embed_dim=16, depths=[2, 1, 1, 1, 1, 1, 1, 1, 2], win_size=8, modulator=False)]:
        net = uformer_b200.Uformer(**cfg)
        net.load_state_dict(randomize_state(net.state_dict(), 11))
        calls = []                                                        # (module, cache, packed-call)
        for m in net.modules():
            if isinstance(m, M.LeWinTransformerBlock):
                calls += [(m, m._cache, m.packed), (m.attn, m.attn._cache, m.attn.packed),
                          (m.mlp, m.mlp._cache_ln, lambda mm=m: mm.mlp.packed(mm.norm2))]
                if m.attn.tma_gather():                                   # LayerNorm-folded projection (+ modulator image) of the TMA-gather W-MSA
                    calls.append((m.attn, m.attn._cache_ln, lambda mm=m: mm.attn.packed_fold(mm.norm1, mm.modulator)))
            elif isinstance(m, (M.Downsample, M.Upsample)):
                calls.append((m, m._cache, m.packed))
        lazy = [{k: (v.clone() if torch.is_tensor(v) else v) for k, v in call().items()} for _, _, call in calls]
        assert any("w1f_img" in d for d in lazy) and (cfg["embed_dim"] == 16 or any("w1_img" in d for d in lazy))   # both LeFF paths
        assert any("wqkv_fold_img" in d for d in lazy) and (not cfg["modulator"] or any("wmod_fold_img" in d for d in lazy))
        M.invalidate_packed()
        assert prepack(net) == sum(cfg["depths"]) + 8
        for (m, cache, call), want in zip(calls, lazy):
            key_before = cache._entry[0]
            got = call()
            assert cache._entry[0] == key_before                          # cache hit: nothing was rebuilt
            assert set(got) == set(want), type(m)
            for k, v in want.items():
                if torch.is_tensor(v):
                    assert got[k].shape == v.shape and got[k].dtype == v.dtype and got[k].is_contiguous(), (type(m).__name__, k)
                    assert torch.equal(got[k], v), (type(m).__name__, k)
                else:
                    assert got[k] == v or (got[k] is None and v is None), (type(m).__name__, k)


def test_bench_reference_arm_contract():
    """bench.py --impl reference prints exactly one JSON line with the keys the driver reads (metric/unit/config of our
    arm, impl, cpu_baseline{kind,cores,sample,value}, e2e with zero copy bytes) and does not need a GPU."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images/sec Uformer-B 256x256 fwd" and d["unit"] == "img/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "images" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: one float32 .npy per output, whole while it fits the budget; past it, the same seeded sample of
    its elements on every run, and all arrays together within the budget."""
    import numpy as np
    import bench
    t = torch.randn(4, 3, 8, 8).to(torch.bfloat16)
    bench.dump_outputs(str(tmp_path / "a"), {"restored": t})
    a = np.load(tmp_path / "a" / "restored.npy")
    assert a.dtype == np.float32 and a.shape == (4, 3, 8, 8) and np.array_equal(a, t.float().numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 400)
    big = torch.randn(1000)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"restored": big, "loss": torch.tensor(0.5)})
    b, c = np.load(tmp_path / "b" / "restored.npy"), np.load(tmp_path / "c" / "restored.npy")
    assert b.dtype == np.float32 and b.shape == (50,) and np.array_equal(b, c) and np.isin(b, big.numpy()).all()
    assert np.load(tmp_path / "b" / "loss.npy") == np.float32(0.5)
    assert sum(f.stat().st_size - 128 for f in (tmp_path / "b").iterdir()) <= 400          # .npy header: 128 bytes


def test_bench_steps_argument():
    """--steps is the number of timed steps; zero or fewer is refused before anything runs."""
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 2 and "--steps" in out.stderr


@pytest.mark.skipif(torch.cuda.is_available(), reason="uses fake device pointers: only meaningful (and safe) where no launch can happen")
def test_alignment_validation_without_gpu():
    """Pointers the kernels access with 16-byte vectors / bulk copies must be 16-byte aligned: rejected with LW_ERR_ALIGN
    before any launch (a DataParallel replica's coalesced parameter views can be 4-byte aligned); 4-byte alignment is
    enough for the scalar-read tables (bqkv, relpos)."""
    lib = _lib.load()
    a = _lib.WmsaArgs()
    for f in ("x", "out", "wqkv_img", "bqkv", "wproj_img", "bproj", "relpos"):
        setattr(a, f, 0x10000)
    a.n_windows, a.windowed, a.C, a.head_dim = 2, 1, 32, 32
    for f in ("x", "out", "wqkv_img", "wproj_img", "bproj"):
        setattr(a, f, 0x10004)
        assert lib.lw_wmsa_fwd(ctypes.byref(a), None) == -5, f
        setattr(a, f, 0x10000)
    a.relpos = a.bqkv = 0x10004
    assert lib.lw_wmsa_fwd(ctypes.byref(a), None) in (0, -3)      # passes validation (-3: no CUDA device in this container)
    d = _lib.AdamWArgs()
    d.p, d.g, d.m, d.v, d.n, d.step, d.beta1, d.beta2 = 0x20000, 0x20004, 0x20000, 0x20000, 64, 1, 0.9, 0.999
    assert lib.lw_adamw_step(ctypes.byref(d), None) == -5
    assert _lib.LW_ERRORS[-5] == "LW_ERR_ALIGN"


def test_torch_cuda_attribute_chains_exist():
    """The launch plumbing (ops._launch, bench.py, tools/) only runs on a GPU box; a typo in a torch.cuda.* name there costs a
    whole GPU call.  Static check: every torch.cuda.<name> the repo mentions exists in the installed torch."""
    import glob
    import re
    files = glob.glob(os.path.join(ROOT, "uformer_b200", "*.py")) + glob.glob(os.path.join(ROOT, "tools", "*.py")) + [
        os.path.join(ROOT, "bench.py"), os.path.join(ROOT, "__graft_entry__.py")]
    bad = []
    for f in files:
        for m in re.finditer(r"torch\.cuda\.([A-Za-z_]+)", open(f).read()):
            if not hasattr(torch.cuda, m.group(1)):
                bad.append((os.path.basename(f), m.group(0)))
    assert not bad, bad


def test_qkv_layernorm_fold_identity():
    """packing.pack_qkv_fold: LN(x) Wqkv^T + b == rstd*(x Wg^T) - rstd*mean*cs + bf (the TMA-gather W-MSA kernel's projection,
    csrc/wmsa_tma.cuh), with Wg rounded to bf16 and cs taken from the rounded matrix; rows in pack_qkv's per-head order."""
    from uformer_b200 import packing
    torch.manual_seed(3)
    C, heads = 64, 2
    hd = C // heads
    wq, bq, wkv, bkv = torch.randn(C, C) * 0.1, torch.randn(C) * 0.1, torch.randn(2 * C, C) * 0.1, torch.randn(2 * C) * 0.1
    g, b = 1 + 0.2 * torch.randn(C), 0.1 * torch.randn(C)
    scale = hd ** -0.5
    img, bf, cs = packing.pack_qkv_fold(wq, bq, wkv, bkv, heads, scale, g, b)
    img0, b0 = packing.pack_qkv(wq, bq, wkv, bkv, heads, scale)
    assert img.shape == img0.shape and img.dtype == torch.bfloat16 and bf.shape == b0.shape == cs.shape
    wg = packing.unpack_kmajor(img, heads * 3 * hd, C, 3 * hd, "nk")
    w0 = packing.unpack_kmajor(img0, heads * 3 * hd, C, 3 * hd, "nk")
    assert torch.equal(cs, wg.sum(1))
    x = torch.randn(50, C) * 3 + 1.5
    mean = x.mean(1, keepdim=True)
    rstd = torch.rsqrt(x.var(1, unbiased=False, keepdim=True) + 1e-5)
    folded = rstd * (x @ wg.t()) - rstd * mean * cs + bf
    direct = torch.nn.functional.layer_norm(x, (C,), g, b) @ w0.t() + b0
    assert (folded - direct).abs().max() < 2e-2 * direct.abs().max()              # bf16 weight rounding on both sides
    # exact in fp64 without the bf16 rounding of the weights
    w3 = torch.cat([wq * scale, wkv], 0).double()
    x64 = x.double()
    ln = torch.nn.functional.layer_norm(x64, (C,), g.double(), b.double())
    m64, r64 = x64.mean(1, keepdim=True), torch.rsqrt(x64.var(1, unbiased=False, keepdim=True) + 1e-5)
    wg64 = w3 * g.double()[None]
    lhs = ln @ w3.t()
    rhs = r64 * (x64 @ wg64.t()) - r64 * m64 * wg64.sum(1) + (w3 * b.double()[None]).sum(1)
    assert (lhs - rhs).abs().max() < 1e-9


def test_window_size_validation_and_support_grid_without_gpu():
    """lw_wmsa_args.win_size (C ABI v6): 0 / 8 = 8x8 windows, 16 = 16x16 windows, anything else is rejected before any launch; the
    token-map geometry is validated against the window size; WindowAttention._check_supported follows lw_wmsa16_supported over
    the BASELINE configs[4] grid (21 of its 24 points are built)."""
    lib = _lib.load()
    a = _lib.WmsaArgs()
    for f in ("x", "out", "wqkv_img", "bqkv", "wproj_img", "bproj", "relpos"):
        setattr(a, f, 0x10000)
    a.n_windows, a.windowed, a.C, a.head_dim = 4, 0, 32, 32
    a.H = a.W = 32
    a.win_size = 7
    assert lib.lw_wmsa_fwd(ctypes.byref(a), None) == -1
    a.win_size, a.H = 16, 24                                      # 24 is a multiple of 8 but not of 16
    assert lib.lw_wmsa_fwd(ctypes.byref(a), None) == -1
    a.H, a.shift = 32, 16                                         # shift must stay below the window size
    assert lib.lw_wmsa_fwd(ctypes.byref(a), None) == -1
    a.shift, a.n_windows = 8, 3                                   # 32x32 tokens = 4 windows of 16x16 per image
    assert lib.lw_wmsa_fwd(ctypes.byref(a), None) == -1
    a.n_windows, a.C, a.head_dim = 4, 256, 64                     # not built: tiles exceed shared memory
    assert lib.lw_wmsa_fwd(ctypes.byref(a), None) == -1
    a.C, a.head_dim = 32, 32
    assert lib.lw_wmsa_fwd(ctypes.byref(a), None) in (0, -3)      # passes validation (-3: no CUDA device in this container)
    built = {}
    for ws in (8, 16):
        for hd in (16, 32, 64):
            for heads in (1, 2, 4, 8):
                att = uformer_b200.WindowAttention(hd * heads, (ws, ws), heads)
                try:
                    att._check_supported()
                    built[(ws, hd, heads)] = True
                except NotImplementedError:
                    built[(ws, hd, heads)] = False
                if ws == 16:
                    assert built[(ws, hd, heads)] == bool(lib.lw_wmsa16_supported(hd * heads, hd))
    assert sorted(k for k, v in built.items() if not v) == [(8, 64, 8), (16, 64, 4), (16, 64, 8)]
    with pytest.raises(NotImplementedError):
        uformer_b200.WindowAttention(32, (4, 4), 1)._check_supported()


def test_kernel_source_hash_identifies_the_profiled_build():
    """bench.py reports roofline.traffic from profiles/r02_kernel_metrics.json only while that table describes the current kernel
    sources: the identity is _lib.csrc_hash() (deterministic, unlike the nvcc output)."""
    import json
    h = _lib.csrc_hash()
    assert h == _lib.csrc_hash() and len(h) == 16 and int(h, 16) >= 0
    tj = json.load(open(os.path.join(ROOT, "profiles", "r02_kernel_metrics.json")))
    assert "csrc_sha256_16" in tj and set(tj["dram_bytes_per_launch"]) == set(tj["us_per_launch"])
