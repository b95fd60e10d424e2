"""CPU: the oracle against the unmodified reference on inputs other than the golden fixtures'.  What the reference computed is
stored in tests/golden/reference_checks.pt (tests/golden/make_reference_checks.py); the install() check needs the reference's
own model.py and is skipped where it is not present."""
import pytest
import torch

from helpers import load_golden, max_err_sampled, rel_l2_sampled, state_checksum
from refshim import reference_available


@pytest.fixture(scope="module")
def ref():
    return load_golden("reference_checks")


def _same_weights(st, c):
    assert abs(state_checksum(st) - c["checksum"]) <= 1e-6 * c["checksum"], "state-dict keys/shapes differ from the reference"


def test_block_live(ref):
    import uformer_b200 as U
    from oracle import lewin_oracle as O
    from paramgen import randomize_state
    for c in ref["block_live"]:
        dim, heads, H, shift, modu, xseed = c["case"]
        st = randomize_state(U.LeWinTransformerBlock(dim, (H, H), heads, win_size=8, shift_size=shift, modulator=modu).state_dict(), 21)
        _same_weights(st, c)
        x = torch.randn(2, H * H, dim, generator=torch.Generator().manual_seed(xseed))
        got = O.lewin_block(x, st, "", heads, 8, shift)
        assert max_err_sampled(got, c["y"]) < 1e-4


def test_input_mask_path_live(ref):
    """The optional input-mask branch (model.py:914-921) with batch 1."""
    import uformer_b200 as U
    from oracle import lewin_oracle as O
    from paramgen import randomize_state
    c = ref["input_mask"]
    st = randomize_state(U.LeWinTransformerBlock(32, (16, 16), 2, win_size=8, shift_size=0).state_dict(), 22)
    _same_weights(st, c)
    gen = torch.Generator().manual_seed(8)
    x = torch.randn(1, 256, 32, generator=gen)
    mask = (torch.rand(1, 1, 16, 16, generator=gen) > 0.5).float()
    got = O.lewin_block(x, st, "", 2, 8, 0, input_mask=mask)
    assert max_err_sampled(got, c["y"]) < 1e-4


@pytest.mark.skipif(not reference_available(), reason="reference not mounted")
def test_install_builds_reference_uformer_on_engine():
    import uformer_b200
    from refshim import import_reference_model
    m = import_reference_model()
    cfg = dict(img_size=128, embed_dim=16, depths=[1] * 9, win_size=8, token_projection="linear", token_mlp="leff", modulator=True)
    ref_state = m.Uformer(**cfg).state_dict()
    uformer_b200.install(m)
    try:
        net = m.Uformer(**cfg)
        assert type(net.encoderlayer_0.blocks[0]) is uformer_b200.LeWinTransformerBlock
        assert type(net.dowsample_0) is uformer_b200.Downsample and type(net.upsample_3) is uformer_b200.Upsample
        net.load_state_dict(ref_state, strict=True)
        with pytest.raises(uformer_b200.EngineUnavailable):
            net(torch.rand(1, 3, 128, 128))       # no CPU fallback
    finally:
        uformer_b200.uninstall(m)
    assert m.Uformer(**cfg).encoderlayer_0.blocks[0].__class__.__module__ == "model"


def test_uformer_win16_live(ref):
    """A whole reference Uformer built with win_size = 16 (16x16 windows, shift 8, the clamp of model.py:863-865 at the 16x16- and
    8x8-token stages) against the oracle — the pin behind tests/test_host_path_cpu.py::test_uformer_with_16x16_windows_..."""
    import uformer_b200 as U
    from oracle import lewin_oracle as O
    from paramgen import randomize_state
    c = ref["uformer_win16"]
    st = randomize_state(U.Uformer(**c["cfg"]).state_dict(), 31)
    _same_weights(st, c)
    x = torch.rand(1, 3, 128, 128, generator=torch.Generator().manual_seed(5))
    got = O.uformer_forward(x.double(), {k: (v.double() if torch.is_floating_point(v) else v) for k, v in st.items()}, 128, 16, [2] * 9, win_size=16)
    assert rel_l2_sampled(got.float(), c["y"]) < 1e-5
