"""CPU: the COMPLETE host path — modules, operand-image packing, pack caches, stage wiring, concat fusion, autograd
wrappers, gradient arena, optimizer plumbing — driven end to end with tests/kernel_model.py standing in for the
native entry points (an executable model of the C-ABI contracts that decodes the packed images).  What this pins:
everything between the reference-facing API and the C ABI.  What it cannot pin: the CUDA kernels (tests -m gpu)."""
import pytest
import torch

import kernel_model as KM
import uformer_b200 as U
from helpers import build_module, golden_names, load_golden, rel_l2, rel_l2_sampled
from paramgen import randomize_state

TOL = 1e-2        # bf16 operands / bf16 HBM round trips are modelled, so the bf16 tolerance of north_star applies


@pytest.mark.parametrize("name", golden_names("wattn") + golden_names("leff") + golden_names("down") + golden_names("up") + golden_names("block"))
def test_modules_through_contract_model(name):
    g = load_golden(name)
    mod, _ = build_module(g)
    with KM.patched() as calls, torch.no_grad():
        y = mod(g["x"])
        assert rel_l2(y, g["y"]) < TOL, name
        if g["kind"] == "wattn":
            assert rel_l2(mod(g["x"], mask=g["mask"]), g["y_mask"]) < TOL
    assert sum(calls.values()) >= 1


@pytest.mark.parametrize("name", ["uformer_t1_128", "uformer_t2_128"])
def test_network_inference_schedule_through_contract_model(name):
    """Inference schedule incl. the in-place skip-concat fusion (Upsample writes the left half of the decoder input)."""
    g = load_golden(name)
    net, _ = build_module(g)
    with KM.patched() as calls:
        y = net(g["x"])                               # eval mode: runs under no_grad by itself
    assert not y.requires_grad
    assert rel_l2(y, g["y"]) < TOL and rel_l2(y - g["x"], g["y"] - g["x"]) < 2 * TOL
    nblk = sum(g["cfg"]["depths"])
    assert calls["wmsa"] == nblk and calls["leff"] == nblk and calls["downsample"] == 4 and calls["upsample"] == 4


def test_train_step_through_contract_model():
    """TrainStep end to end: training-mode forward through the autograd wrappers, Charbonnier, backward into the flat
    arena, AdamW over the arena, operand images rebuilt after the update.  Gradients of the first step are compared
    with the reference's (fp32) golden; then the loss must fall."""
    from uformer_b200.training import TrainStep
    g = load_golden("train_t2_128")
    net = U.Uformer(**g["cfg"])
    net.load_state_dict(randomize_state(net.state_dict(), g["seed"]), strict=True)
    with KM.patched() as calls:
        step = TrainStep(net, lr=2e-4, weight_decay=0.0)
        # first step by hand so the gradient arena can be inspected before the optimizer zeroes it
        net.train()
        restored = net(g["x"])
        assert restored.requires_grad
        loss = step.criterion(restored, g["target"])
        loss.backward()
        assert abs(loss.item() - g["loss"]) < 2e-2 * g["loss"]
        got, want = [], []
        for k, p in net.named_parameters():
            ref = g["grads"][k]
            assert p.grad is not None and p.grad.data_ptr() >= step.arena.grad.data_ptr(), k
            got.append(p.grad.reshape(-1)[::ref["stride"]].clone())
            want.append(ref["sample"])
        e = rel_l2(torch.cat(got), torch.cat(want))
        print("sampled-gradient rel-L2 vs reference golden (bf16-modelled forward, fp32 backward):", e)
        assert e < 5e-2
        step.optimizer.step(grad_scale=1.0, zero_grad=True)
        assert step.arena.grad.abs().sum() == 0
        n_pack_calls = calls["wmsa"]
        from uformer_b200 import packing
        n_perm, orig = [0], packing.pack_kmajor

        def counting(*a, **k):
            n_perm[0] += 1
            return orig(*a, **k)
        packing.pack_kmajor = counting
        try:
            losses = [loss.item()] + [step(g["x"], g["target"]).item() for _ in range(3)]
        finally:
            packing.pack_kmajor = orig
        # steps 2 and 3 re-pack through prepack(): <= 6 GEMM images per (stage shape, modulator?) group (qkv, folded qkv, modulator
        # image, proj, linear1, linear2) + 8 samplers, not 6 per block
        groups = len({(b.dim, b.num_heads, b.modulator is None) for b in net.modules() if isinstance(b, U.LeWinTransformerBlock)})
        assert n_perm[0] <= 6 * sum(g["cfg"]["depths"]) + 8 + 3 * (6 * groups + 8), n_perm[0]
        assert calls["wmsa"] > n_pack_calls and calls["adamw_step"] == 4 and calls["charbonnier"] == 4
    print("losses:", losses)
    assert losses[-1] < losses[0] and len({round(v, 7) for v in losses}) == 4      # weights (and their packed images) really moved


def test_block_training_mode_drop_path_through_contract_model():
    from uformer_b200 import restated as R
    blk = U.LeWinTransformerBlock(32, (16, 16), 2, win_size=8, shift_size=4, modulator=True, drop_path=0.5)
    blk.load_state_dict(randomize_state(blk.state_dict(), 17))
    blk.train()
    x = torch.randn(6, 256, 32).to(torch.bfloat16)
    with KM.patched():
        torch.manual_seed(5)
        y = blk(x)                                    # params require grad -> goes through NativeFn
        assert y.grad_fn is not None and y.dtype == torch.bfloat16
        torch.manual_seed(5)
        s1, s2 = blk.drop_path.draw(6, x.device), blk.drop_path.draw(6, x.device)
        ref = R.lewin_block(blk, x.float(), None, s1, s2)
        assert rel_l2(y.float().detach(), ref.detach()) < TOL
        # backward through the wrapper == autograd through the restated statements (same scales)
        gout = torch.randn_like(ref)
        y.backward(gout.to(torch.bfloat16))
        got = {k: p.grad.clone() for k, p in blk.named_parameters()}
        for p in blk.parameters():
            p.grad = None
        R.lewin_block(blk, x.float(), None, s1, s2).backward(gout.to(torch.bfloat16).float())
        for k, p in blk.named_parameters():
            assert rel_l2(got[k], p.grad) < 2e-2, k


def test_reference_model_with_engine_installed_through_contract_model():
    """install(model): the reference's own Uformer class builds on the engine's modules and produces the reference's
    output (model.py drives LeWinTransformerBlock / Downsample / Upsample through their nn.Module surface)."""
    from refshim import import_reference_model, reference_available
    if not reference_available():
        pytest.skip("reference not mounted")
    m = import_reference_model()
    g = load_golden("uformer_t1_128")
    U.install(m)
    try:
        net = m.Uformer(**g["cfg"])
        assert isinstance(net.encoderlayer_0.blocks[0], U.LeWinTransformerBlock) and isinstance(net.dowsample_0, U.Downsample)
        net.load_state_dict(randomize_state(net.state_dict(), g["seed"]), strict=True)
        net.eval()
        with KM.patched(), torch.no_grad():
            y = net(g["x"])
        assert rel_l2(y, g["y"]) < TOL
    finally:
        U.uninstall(m)


def test_reference_model_win16_with_engine_installed_through_contract_model():
    """The same drop-in with win_size = 16: the reference's Uformer(win_size=16) builds on the engine's modules and its forward
    through the kernel contracts equals its own forward on the reference's modules (same weights)."""
    from refshim import import_reference_model, reference_available
    if not reference_available():
        pytest.skip("reference not mounted")
    m = import_reference_model()
    cfg = dict(img_size=128, embed_dim=16, depths=[2] * 9, win_size=16, token_projection="linear", token_mlp="leff", modulator=False)
    ref_net = m.Uformer(**cfg).eval()
    st = randomize_state(ref_net.state_dict(), 31)
    ref_net.load_state_dict(st)
    x = torch.rand(1, 3, 128, 128, generator=torch.Generator().manual_seed(6))
    with torch.no_grad():
        want = ref_net(x)
    U.install(m)
    try:
        net = m.Uformer(**cfg)
        assert isinstance(net.encoderlayer_0.blocks[1], U.LeWinTransformerBlock) and net.encoderlayer_0.blocks[1].shift_size == 8
        net.load_state_dict(st, strict=True)
        net.eval()
        with KM.patched() as calls, torch.no_grad():
            y = net(x)
        assert calls["wmsa"] == 18 and rel_l2(y, want) < TOL
    finally:
        U.uninstall(m)


def test_arbitrary_resolution_restore_through_contract_model():
    """BASELINE configs[3]: model built for 128x128 restores a 200x150 image (padded to 256x256 by expand2square,
    test/test_sidd.py:79-108); compared with the oracle forward on the padded image and with what the reference's own model
    restored from it (a stored sample)."""
    from oracle import lewin_oracle as O
    g = load_golden("uformer_t1_128")
    net, st = build_module(g)
    torch.manual_seed(3)
    noisy = torch.rand(1, 3, 200, 150)
    padded, mask = U.expand2square(noisy, factor=128)
    assert padded.shape == (1, 3, 256, 256) and int(mask.sum()) == 200 * 150
    assert torch.equal(torch.masked_select(padded, mask.bool()).reshape(1, 3, 200, 150), noisy)
    with KM.patched():
        out = U.restore_image(net, noisy, factor=128)
    assert out.shape == noisy.shape and out.min() >= 0 and out.max() <= 1
    c = g["cfg"]
    r = O.uformer_forward(padded, st, c["img_size"], c["embed_dim"], c["depths"], win_size=c["win_size"])
    want = torch.masked_select(r, mask.bool()).reshape(1, 3, 200, 150).clamp(0, 1)
    assert rel_l2(out, want) < TOL
    assert rel_l2_sampled(out, load_golden("reference_checks")["restore_200x150"]["y"]) < TOL


def test_reference_training_loop_with_engine_installed_through_contract_model():
    """Drop-in for the training script (INTEGRATION.md): the REFERENCE's Uformer class, built on the engine's modules by
    install(), trained by TrainStep — its own InputProj/OutputProj/BasicUformerLayer code drives our blocks under autograd.
    The first step's gradients are compared with the golden produced by the unmodified reference."""
    from refshim import import_reference_model, reference_available
    from uformer_b200.training import TrainStep
    if not reference_available():
        pytest.skip("reference not mounted")
    m = import_reference_model()
    g = load_golden("train_t2_128")
    U.install(m)
    try:
        net = m.Uformer(**g["cfg"])
        net.load_state_dict(randomize_state(net.state_dict(), g["seed"]), strict=True)
        with KM.patched() as calls:
            step = TrainStep(net, lr=2e-4, weight_decay=0.0)
            net.train()
            loss = step.criterion(net(g["x"]), g["target"])
            loss.backward()
            assert calls["wmsa"] == sum(g["cfg"]["depths"]) and calls["input_proj"] == 0       # the reference's own projections ran
            got = torch.cat([p.grad.reshape(-1)[::g["grads"][k]["stride"]] for k, p in net.named_parameters()])
            want = torch.cat([g["grads"][k]["sample"] for k, _ in net.named_parameters()])
            assert abs(loss.item() - g["loss"]) < 2e-2 * g["loss"] and rel_l2(got, want) < 5e-2
            step.optimizer.step(zero_grad=True)
            l2 = step(g["x"], g["target"]).item()
            l3 = step(g["x"], g["target"]).item()
        assert l3 < l2 < loss.item()
    finally:
        U.uninstall(m)


def test_train_step_checkpoint_resume_through_contract_model():
    """state_dict()/load_state_dict(): 2 steps + save + 2 steps == restore into a fresh TrainStep + 2 steps, bit for bit."""
    from uformer_b200.training import TrainStep
    cfg = dict(img_size=128, embed_dim=16, depths=[1] * 9, win_size=8, modulator=True, drop_path_rate=0.0)
    torch.manual_seed(0)
    x, t = torch.rand(1, 3, 128, 128), torch.rand(1, 3, 128, 128)

    def fresh():
        net = U.Uformer(**cfg)
        net.load_state_dict(randomize_state(net.state_dict(), 2), strict=True)
        return net, TrainStep(net, lr=1e-4)
    with KM.patched():
        net, ts = fresh()
        for _ in range(2):
            ts(x, t)
        ck = ts.state_dict()
        assert set(ck["state_dict"]) == set(net.state_dict())          # the reference's checkpoint keys
        cont = [ts(x, t).item() for _ in range(2)]
        net2, ts2 = fresh()
        ts2.load_state_dict(ck)
        assert ts2.optimizer.steps == 2
        resumed = [ts2(x, t).item() for _ in range(2)]
    assert resumed == cont
    for a, b in zip(net.parameters(), net2.parameters()):
        assert torch.equal(a, b)


def test_smoke_host_logic_through_contract_model(capsys):
    """__graft_entry__.smoke() is what the driver runs on the B200 before the bench; its host logic (oracle calls,
    tolerances, arena / optimizer plumbing) is exercised here on CPU with the kernel model standing in."""
    import __graft_entry__ as ge
    with KM.patched() as calls:
        ge.smoke(device="cpu")
    assert "smoke: ok" in capsys.readouterr().out
    assert calls["wmsa"] >= 2 and calls["leff"] >= 2 and calls["downsample"] == 1 and calls["upsample"] == 1
    assert calls["charbonnier"] == 1 and calls["adamw_step"] == 1


@pytest.mark.parametrize("dim,heads", [(16, 1), (32, 1), (32, 2), (64, 2), (64, 4), (128, 4), (128, 8), (256, 8), (256, 16), (512, 16),
                                       (64, 1), (128, 2), (256, 4)])
def test_every_supported_channel_count_through_contract_model(dim, heads):
    """Operand-image packing for every (C, head_dim in {16, 32, 64}) the kernels are instantiated for: block through the
    contract model (which decodes the images) == oracle on the raw weights."""
    from oracle import lewin_oracle as O
    shift = 4 if dim % 64 == 0 else 0
    blk = U.LeWinTransformerBlock(dim, (16, 16), heads, win_size=8, shift_size=shift, modulator=dim >= 64).eval()
    st = randomize_state(blk.state_dict(), dim + heads)
    blk.load_state_dict(st)
    x = torch.randn(2, 256, dim).to(torch.bfloat16)
    with KM.patched(), torch.no_grad():
        y = blk(x).float()
    ref = O.lewin_block(x.float(), st, "", heads, 8, shift)
    assert rel_l2(y, ref) < TOL, (dim, heads, rel_l2(y, ref))
    for m, cin, cout in [(U.Downsample, dim, 2 * dim), (U.Upsample, dim, dim // 2)]:
        if cout > 512 or cout < 8:
            continue
        mod = m(cin, cout).eval()
        sm = randomize_state(mod.state_dict(), 1)
        mod.load_state_dict(sm)
        with KM.patched(), torch.no_grad():
            z = mod(x).float()
        want = O.downsample(x.float(), sm["conv.0.weight"], sm["conv.0.bias"]) if m is U.Downsample else \
            O.upsample(x.float(), sm["deconv.0.weight"], sm["deconv.0.bias"])
        assert rel_l2(z, want) < TOL, (m.__name__, cin, cout)


@pytest.mark.parametrize("name", ["uformer_b_256", "uformer_b_256_g05"])
def test_flagship_model_through_contract_model(name):
    """Uformer-B 256x256 (BASELINE configs[1], the bench's architecture; (a) the bench's weights, (b) scaled to a
    denoiser-like small residual branch) through the contract model with bf16 HBM round trips modelled: predicts the
    GPU's parity error (on uformer_t2_128 the model says 7.3e-3, the B200 measured 7.7e-3) and is held to the same
    bounds as the GPU test (helpers.model_tolerances)."""
    from helpers import model_tolerances
    g = load_golden(name)
    net, _ = build_module(g)
    with KM.patched():
        y = net(g["x"])
    tf, tr = model_tolerances(g)
    ef, er = rel_l2(y, g["y"]), rel_l2(y - g["x"], g["y"] - g["x"])
    print(f"{name}: modelled rel-L2 full {ef:.3e} (bound {tf:.3e}), residual branch {er:.3e} (bound {tr:.3e}); "
          f"reference's own bf16 autocast: {g['ref_bf16']}")
    assert ef < tf and er < tr                                      # default precision mode: plain tolerance, no slack


@pytest.mark.parametrize("name", ["uformer_b_256", "uformer_t2_128"])
def test_residual_precision_modes_through_contract_model(name):
    """fp32 residual stream inside a stage (x fp32 -> W-MSA writes x1 fp32 + a bf16 operand copy -> LeFF adds in fp32) vs the
    faster all-bf16 stream (set_residual_precision); the default policy picks fp32 for the stages of >= 4 blocks.  On the flagship with the bench's weights
    only the fp32 stream brings the modelled parity error under north_star's plain 1e-2."""
    g = load_golden(name)
    net, _ = build_module(g)
    with KM.patched():
        y_auto = net(g["x"])                                        # default policy: fp32 stream in stages of >= 4 blocks
        assert U.set_residual_precision(net, torch.float32) == sum(g["cfg"]["depths"])
        y_32 = net(g["x"])
        U.set_residual_precision(net, torch.bfloat16)
        y_bf = net(g["x"])
        U.set_residual_precision(net, torch.float32)
        assert torch.equal(net(g["x"]), y_32)                       # switching back restores the path exactly
    assert rel_l2(y_auto, g["y"]) < TOL
    e_bf, e_32 = rel_l2(y_bf, g["y"]), rel_l2(y_32, g["y"])
    print(f"{name}: bf16 residual stream {e_bf:.3e} -> fp32 residual stream {e_32:.3e}")
    assert e_32 < TOL and e_32 < 0.9 * e_bf
    assert rel_l2(y_32 - g["x"], g["y"] - g["x"]) < TOL


def test_block_property_random_shapes_through_contract_model():
    """hypothesis: for random (C, heads, map side, batch, shift, modulator, input mask) the module -> packing -> contract
    path equals the oracle (SURVEY §8c 'property tests over shapes')."""
    from hypothesis import given, settings, strategies as st
    from oracle import lewin_oracle as O

    @settings(max_examples=12, deadline=None, derandomize=True)
    @given(ch=st.sampled_from([(16, 1), (32, 1), (32, 2), (64, 2), (64, 4), (128, 4)]), side=st.sampled_from([8, 16, 24, 40]),
           batch=st.integers(1, 3), shifted=st.booleans(), modu=st.booleans(), masked=st.booleans(), seed=st.integers(0, 2 ** 16))
    def run(ch, side, batch, shifted, modu, masked, seed):
        dim, heads = ch
        shift = 4 if (shifted and side > 8) else 0
        blk = U.LeWinTransformerBlock(dim, (max(side, 16), max(side, 16)), heads, win_size=8, shift_size=shift, modulator=modu).eval()
        st_ = randomize_state(blk.state_dict(), seed)
        blk.load_state_dict(st_)
        g = torch.Generator().manual_seed(seed)
        x = torch.randn(batch, side * side, dim, generator=g).to(torch.bfloat16)
        mask = (torch.rand(batch, 1, side, side, generator=g) > 0.5).float() if masked else None
        if masked and shift > 0 and batch > 1:
            # the reference itself rejects this combination: model.py:942 adds the (B*nW,N,N) input mask to the (nW,N,N)
            # shift mask, which does not broadcast for B > 1 — oracle and engine both raise like it does
            with pytest.raises(RuntimeError):
                O.lewin_block(x.float(), st_, "", heads, 8, shift, input_mask=mask)
            with KM.patched(), torch.no_grad(), pytest.raises(RuntimeError):
                blk(x, mask=mask)
            return
        with KM.patched(), torch.no_grad():
            y = blk(x, mask=mask).float()
        ref = O.lewin_block(x.float(), st_, "", heads, 8, shift, input_mask=mask)
        assert rel_l2(y, ref) < TOL, (ch, side, batch, shift, modu, masked, rel_l2(y, ref))

    run()


def test_block_ws16_property_through_contract_model():
    """The same property for 16x16 windows (BASELINE configs[4]; lw_wmsa_args.win_size = 16): every (C, head_dim) pair the
    16x16-window kernel is built for, shift 0 / 8, modulator (256 x C), input mask, fp32 residual stream."""
    from hypothesis import given, settings, strategies as st
    from oracle import lewin_oracle as O

    @settings(max_examples=8, deadline=None, derandomize=True)
    @given(ch=st.sampled_from([(16, 1), (32, 2), (32, 1), (64, 2), (64, 1), (128, 8), (128, 2), (256, 8)]), side=st.sampled_from([16, 32]),
           batch=st.integers(1, 2), shifted=st.booleans(), modu=st.booleans(), masked=st.booleans(), fp32=st.booleans(), seed=st.integers(0, 2 ** 16))
    def run(ch, side, batch, shifted, modu, masked, fp32, seed):
        dim, heads = ch
        shift = 8 if (shifted and side > 16) else 0
        blk = U.LeWinTransformerBlock(dim, (32, 32), heads, win_size=16, shift_size=shift, modulator=modu).eval()
        assert blk.win_size == 16 and not blk.attn.tma_gather()
        blk.residual_fp32 = fp32
        st_ = randomize_state(blk.state_dict(), seed)
        blk.load_state_dict(st_)
        g = torch.Generator().manual_seed(seed)
        x = torch.randn(batch, side * side, dim, generator=g).to(torch.bfloat16)
        mask = (torch.rand(batch, 1, side, side, generator=g) > 0.5).float() if (masked and not (shift > 0 and batch > 1)) else None
        with KM.patched(), torch.no_grad():
            y = blk(x, mask=mask).float()
        ref = O.lewin_block(x.float(), st_, "", heads, 16, shift, input_mask=mask)
        assert rel_l2(y, ref) < TOL, (ch, side, batch, shift, modu, masked, fp32, rel_l2(y, ref))

    run()


def test_uformer_with_16x16_windows_through_contract_model():
    """A whole Uformer built with win_size = 16 (the reference's Uformer(win_size=...) argument, model.py:1076): the engine's own
    caller wires 16x16-window blocks (shifted by 8 on odd blocks), the construction-time clamp turns the 16x16-token stages into
    un-shifted single-window blocks and the 8x8-token bottleneck into 8x8-window blocks (model.py:863-865), and the whole
    forward through the kernel contracts equals the oracle."""
    from oracle import lewin_oracle as O
    cfg = dict(img_size=128, embed_dim=16, depths=[2] * 9, win_size=16, token_projection="linear", token_mlp="leff", modulator=False)
    net = U.Uformer(**cfg).eval()
    st = randomize_state(net.state_dict(), 31)
    net.load_state_dict(st)
    blocks = [m for m in net.modules() if isinstance(m, U.LeWinTransformerBlock)]
    assert {(b.win_size, b.shift_size) for b in blocks} == {(16, 0), (16, 8), (8, 0)}
    x = torch.rand(1, 3, 128, 128, generator=torch.Generator().manual_seed(5))
    with KM.patched(), torch.no_grad():
        y = net(x).float()
    ref = O.uformer_forward(x, st, 128, 16, [2] * 9, win_size=16)
    assert rel_l2(y, ref) < TOL and rel_l2(y - x, ref - x) < 2 * TOL, (rel_l2(y, ref), rel_l2(y - x, ref - x))


def _data_parallel_replica(mod):
    """What torch.nn.parallel.replicate builds for one device (it needs CUDA, so it is re-enacted here): every module is
    `_replicate_for_data_parallel()`-ed (its `_parameters` becomes {}), the broadcast copies of the parameters — autograd
    non-leaf tensors whose gradient flows back to the source parameter — are set as plain attributes and recorded in
    `_former_parameters`."""
    from collections import OrderedDict
    mods = list(mod.modules())
    idx = {m: i for i, m in enumerate(mods)}
    reps = []
    for m in mods:
        r = m._replicate_for_data_parallel()
        r._former_parameters = OrderedDict()
        reps.append(r)
    for m, r in zip(mods, reps):
        for k, child in m._modules.items():
            if child is None:
                r._modules[k] = None
            else:
                setattr(r, k, reps[idx[child]])
        for k, p in m._parameters.items():
            if p is None:
                r._parameters[k] = None
            else:
                cp = p.view_as(p)                     # stand-in for Broadcast.apply: non-leaf, grads reach p
                setattr(r, k, cp)
                r._former_parameters[k] = cp
    return reps[0]


def test_data_parallel_replica_gets_parameter_gradients():
    """ADVICE r1 (high): the reference wraps the model in nn.DataParallel (train/train_denoise.py:83); replicas have an
    empty `_parameters`, so collecting trainable tensors with `mod.parameters()` silently trained nothing."""
    from uformer_b200 import autograd as AG
    blk = U.LeWinTransformerBlock(32, (16, 16), 2, win_size=8, shift_size=4, modulator=True)
    blk.load_state_dict(randomize_state(blk.state_dict(), 3))
    blk.train()
    rep = _data_parallel_replica(blk)
    assert len(list(rep.parameters())) == 0 and len(AG.trainable_tensors(rep)) == len(list(blk.parameters()))
    x = torch.randn(2, 256, 32).to(torch.bfloat16)
    with KM.patched():
        y = rep(x)
        assert y.grad_fn is not None
        y.float().pow(2).mean().backward()
    for k, p in blk.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all() and p.grad.abs().sum() > 0, k
