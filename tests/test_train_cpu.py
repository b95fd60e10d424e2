"""CPU: the training path's host logic and backward math.

* uformer_b200/restated.py (the statements backward differentiates) against the golden gradients generated from the
  unmodified reference (tests/golden/make_train_golden.py), and against the reference's own autograd on single blocks and
  samplers — incl. training-mode stochastic depth with a shared RNG seed (tests/golden/make_reference_checks.py);
* autograd.NativeFn wiring (recompute-from-input backward) with a stand-in forward;
* FlatArena layout, in-place gradient accumulation, bucket construction.
No native compute runs here (no GPU): the modules' forward still raises EngineUnavailable on CPU.
"""
import pytest
import torch

import uformer_b200 as U
from uformer_b200 import autograd as AG
from uformer_b200 import restated as R
from uformer_b200 import training as T
from helpers import load_golden, rel_l2, rel_l2_sampled, state_checksum
from paramgen import randomize_state


def _charbonnier(x, y, eps=1e-3):
    return torch.sqrt((x - y) ** 2 + eps * eps).mean()


def _sample(t, stride):
    return t.reshape(-1)[::stride]


def test_restated_backward_matches_reference_golden():
    g = load_golden("train_t2_128")
    net = U.Uformer(**g["cfg"])
    net.load_state_dict(randomize_state(net.state_dict(), g["seed"]), strict=True)
    net.train()
    y = R.uformer(net, g["x"])
    assert rel_l2(y.detach(), g["y"]) < 1e-5
    loss = _charbonnier(y, g["target"])
    assert abs(float(loss) - g["loss"]) < 1e-5 * abs(g["loss"])
    loss.backward()
    worst = 0.0
    for k, p in net.named_parameters():
        ref = g["grads"][k]
        assert p.grad is not None, k
        e = rel_l2(_sample(p.grad, ref["stride"]), ref["sample"])
        worst = max(worst, e)
        assert e < 1e-3, (k, e)
        assert abs(float(p.grad.double().norm()) - ref["norm"]) < 1e-3 * ref["norm"] + 1e-9, k
    print("worst sampled-gradient rel-L2 vs reference:", worst)


@pytest.mark.parametrize("dim,heads,H,shift,modu,dp", [(32, 1, 16, 0, False, 0.0), (64, 2, 24, 4, True, 0.3), (32, 2, 16, 4, True, 0.5)])
def test_restated_block_vs_reference_autograd(dim, heads, H, shift, modu, dp):
    """Forward, input gradient and every parameter gradient of one LeWin block, training mode, stochastic depth drawn
    from the same RNG state as the reference's (model.py:986-987)."""
    c = next(c for c in load_golden("reference_checks")["block_autograd"] if c["case"][:6] == (dim, heads, H, shift, modu, dp))
    xseed = c["case"][6]
    ours = U.LeWinTransformerBlock(dim, (H, H), heads, win_size=8, shift_size=shift, modulator=modu, drop_path=dp)
    st = randomize_state(ours.state_dict(), 21)
    assert abs(state_checksum(st) - c["checksum"]) <= 1e-6 * c["checksum"]
    ours.load_state_dict(st, strict=True)
    ours.train()
    B = 4
    gen = torch.Generator().manual_seed(xseed)
    xo = torch.randn(B, H * H, dim, generator=gen).requires_grad_(True)
    gout = torch.randn(B, H * H, dim, generator=gen)
    torch.manual_seed(99)
    s1 = ours.drop_path.draw(B, xo.device) if dp > 0 else None
    s2 = ours.drop_path.draw(B, xo.device) if dp > 0 else None
    yo = R.lewin_block(ours, xo, None, s1, s2)
    yo.backward(gout)
    assert rel_l2_sampled(yo, c["y"]) < 1e-5
    assert rel_l2_sampled(xo.grad, c["dx"]) < 1e-4
    assert set(c["grads"]) == {k for k, _ in ours.named_parameters()}
    for k, p in ours.named_parameters():
        assert rel_l2_sampled(p.grad, c["grads"][k]) < 1e-4, k


def test_restated_samplers_vs_reference_autograd():
    checks = load_golden("reference_checks")["samplers"]
    for name, ours, fn in [("down", U.Downsample(16, 32), R.downsample), ("up", U.Upsample(32, 8), R.upsample),
                           ("leff", U.LeFF(16, 64), R.leff)]:
        c = checks[name]
        st = randomize_state(ours.state_dict(), 3)
        assert abs(state_checksum(st) - c["checksum"]) <= 1e-6 * c["checksum"], name
        ours.load_state_dict(st, strict=True)
        gen = torch.Generator().manual_seed(c["seed"])
        xo = torch.randn(*c["shape"], generator=gen).requires_grad_(True)
        yo = fn(ours, xo)
        yo.backward(torch.randn(yo.shape, generator=gen))
        assert rel_l2_sampled(yo, c["y"]) < 1e-5 and rel_l2_sampled(xo.grad, c["dx"]) < 1e-4, name
        assert set(c["grads"]) == {k for k, _ in ours.named_parameters()}, name
        for k, p in ours.named_parameters():
            assert rel_l2_sampled(p.grad, c["grads"][k]) < 1e-4, (name, k)


def test_nativefn_recompute_backward_wiring():
    """NativeFn with a stand-in 'native' forward: gradients w.r.t. the activation and the parameters equal plain
    autograd through the restated statements; non-differentiable extra activations get None."""
    blk = U.LeWinTransformerBlock(32, (16, 16), 2, win_size=8, shift_size=4, modulator=True)
    blk.load_state_dict(randomize_state(blk.state_dict(), 5))
    params = [p for p in blk.parameters() if p.requires_grad]
    x = torch.randn(2, 256, 32)
    s1 = torch.tensor([1.25, 0.0]).view(2, 1, 1)
    s2 = torch.tensor([0.0, 1.25]).view(2, 1, 1)
    calls = []

    def native(t, a, b):
        calls.append(torch.is_grad_enabled())
        return R.lewin_block(blk, t, None, a, b)

    xa = x.clone().requires_grad_(True)
    y = AG.apply(native, lambda t, a, b: R.lewin_block(blk, t, None, a, b), [xa, s1, s2], params)
    assert calls == [False] and y.grad_fn is not None
    g = torch.randn_like(y)
    y.backward(g)
    got = [xa.grad.clone()] + [p.grad.clone() for p in params]
    for p in params:
        p.grad = None
    xb = x.clone().requires_grad_(True)
    R.lewin_block(blk, xb, None, s1, s2).backward(g)
    want = [xb.grad] + [p.grad for p in params]
    for a, b in zip(got, want):
        assert rel_l2(a, b) < 1e-6


def test_flat_arena_views_and_inplace_accumulation():
    net = torch.nn.Sequential(torch.nn.Linear(5, 7), torch.nn.LayerNorm(7), torch.nn.Linear(7, 3))
    before = [p.detach().clone() for p in net.parameters()]
    arena = T.FlatArena(list(net.parameters())[::-1])
    for p, b in zip(net.parameters(), before):
        assert torch.equal(p, b)                                  # values preserved
        assert p.data_ptr() >= arena.flat.data_ptr() and p.data_ptr() < arena.flat.data_ptr() + 4 * arena.numel
        assert p.grad.data_ptr() - arena.grad.data_ptr() == p.data_ptr() - arena.flat.data_ptr()
        assert (p.data_ptr() - arena.flat.data_ptr()) % 256 == 0  # sector-aligned views
    x = torch.randn(4, 5)
    net(x).sum().backward()
    g1 = arena.grad.clone()
    assert g1.abs().sum() > 0
    net(x).sum().backward()                                       # accumulates IN PLACE into the arena views
    assert torch.allclose(arena.grad, 2 * g1)
    arena.flat.mul_(0.5)                                          # an update of the arena is an update of the module
    for p, b in zip(net.parameters(), before):
        assert torch.allclose(p, 0.5 * b)
    arena.zero_grad()
    assert arena.grad.abs().sum() == 0 and all(p.grad is not None for p in net.parameters())


def test_execution_order_and_buckets():
    net = U.Uformer(img_size=128, embed_dim=16, depths=[1] * 9, win_size=8, modulator=True)
    order = T.execution_ordered_parameters(net)
    assert len(order) == len(list(net.parameters())) and len({id(p) for p in order}) == len(order)
    assert order[0] is net.input_proj.proj[0].weight and order[-1] is net.output_proj.proj[0].bias
    names = {id(p): k for k, p in net.named_parameters()}
    seq = [names[id(p)].split(".")[0] for p in order]
    assert seq.index("upsample_0") > seq.index("conv") > seq.index("dowsample_3") > seq.index("encoderlayer_3")
    arena = T.FlatArena(order[::-1])
    red = T.GradReducer(arena, None, bucket_bytes=1 << 20)
    assert red.world == 1 and len(red.buckets) > 3
    assert red.buckets[0][0] == 0 and red.buckets[-1][1] == arena.numel
    for (lo, hi, _), (lo2, _, _) in zip(red.buckets, red.buckets[1:]):
        assert hi == lo2 and (hi - lo) * 4 >= 1 << 20             # contiguous, each at least bucket_bytes
    assert sorted(i for b in red.buckets for i in b[2]) == list(range(len(order)))


def test_training_ops_have_no_cpu_path():
    with pytest.raises(U.EngineUnavailable):
        T.CharbonnierLoss()(torch.rand(1, 3, 8, 8), torch.rand(1, 3, 8, 8))
    net = torch.nn.Linear(4, 4)
    opt = T.FlatAdamW(T.FlatArena(list(net.parameters())))
    with pytest.raises(U.EngineUnavailable):
        opt.step()
    net = U.Uformer(img_size=128, embed_dim=16, depths=[1] * 9, win_size=8, modulator=True).train()
    with pytest.raises(U.EngineUnavailable):
        net(torch.rand(1, 3, 128, 128))


def test_stochastic_depth_schedule_and_flops_equal_reference():
    """Per-block drop_path rates (model.py:1093-1095 and the decoder slices :1170-1232) and Uformer.flops() of the engine's
    own caller equal the reference's for the Uformer-B configuration."""
    c = load_golden("reference_checks")["uformer_b"]
    o = U.Uformer(**c["cfg"])
    stages = ["encoderlayer_0", "encoderlayer_1", "encoderlayer_2", "encoderlayer_3", "conv", "decoderlayer_0", "decoderlayer_1",
              "decoderlayer_2", "decoderlayer_3"]
    rates = [round(getattr(b.drop_path, "drop_prob", 0.0), 7) for n in stages for b in getattr(o, n).blocks]
    assert rates == c["drop_path_rates"] and max(rates) == 0.1
    assert o.flops() == c["flops"]
