"""Generate reference_checks.pt: what the original Uformer computes in the checks of tests/test_oracle_vs_reference.py and the
reference-autograd checks of tests/test_train_cpu.py and the arbitrary-resolution restore of tests/test_host_path_cpu.py, so those
checks run wherever the test suite runs.

    python tests/golden/make_reference_checks.py

Needs the original project's model.py (located by tests/refshim.py).  Inputs come from the per-case seeded generators below and
are re-drawn by the tests; weights are re-derived from their seed (tests/paramgen.py) and pinned by a checksum.  Outputs and
gradients are stored as a strided sample (`flat[::stride]`, at most CAP elements) with the full tensor's L2 norm and max-abs.
"""
import contextlib
import io
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from refshim import import_reference_model  # noqa: E402
from paramgen import randomize_state  # noqa: E402
from helpers import state_checksum  # noqa: E402
import uformer_b200 as U  # noqa: E402

CAP_OUT, CAP_PARAM = 2048, 256

# (dim, heads, H, shift, modulator, input seed)
BLOCK_LIVE = [(32, 1, 16, 4, True, 71), (64, 4, 32, 4, False, 72)]
# (dim, heads, H, shift, modulator, drop_path, input seed)
BLOCK_AUTOGRAD = [(32, 1, 16, 0, False, 0.0, 81), (64, 2, 24, 4, True, 0.3, 82), (32, 2, 16, 4, True, 0.5, 83)]
WIN16_CFG = dict(img_size=128, embed_dim=16, depths=[2] * 9, win_size=16, token_projection="linear", token_mlp="leff", modulator=False)
UFORMER_B_CFG = dict(img_size=256, embed_dim=32, win_size=8, token_projection="linear", token_mlp="leff", depths=[1, 2, 8, 8, 2, 8, 8, 2, 1],
                     modulator=True, dd_in=3, drop_path_rate=0.1)
STAGES = ["encoderlayer_0", "encoderlayer_1", "encoderlayer_2", "encoderlayer_3", "conv", "decoderlayer_0", "decoderlayer_1",
          "decoderlayer_2", "decoderlayer_3"]


def pack(t, cap=CAP_OUT):
    flat = t.detach().reshape(-1)
    stride = max(1, -(-flat.numel() // cap))
    return dict(stride=stride, sample=flat[::stride].clone(), norm=float(flat.double().norm()), absmax=float(flat.abs().max()))


def load_random(mod, seed):
    st = randomize_state(mod.state_dict(), seed)
    mod.load_state_dict(st, strict=True)
    return st


def drop_path_rates(net):
    return [round(getattr(b.drop_path, "drop_prob", 0.0), 7) for n in STAGES for b in getattr(net, n).blocks]


def main():
    m = import_reference_model()
    out = dict(kind="reference_checks")

    with torch.no_grad():
        out["block_live"] = []
        for dim, heads, H, shift, modu, xseed in BLOCK_LIVE:
            blk = m.LeWinTransformerBlock(dim, (H, H), heads, win_size=8, shift_size=shift, modulator=modu).eval()
            st = load_random(blk, 21)
            x = torch.randn(2, H * H, dim, generator=torch.Generator().manual_seed(xseed))
            out["block_live"].append(dict(case=(dim, heads, H, shift, modu, xseed), checksum=state_checksum(st), y=pack(blk(x))))

        blk = m.LeWinTransformerBlock(32, (16, 16), 2, win_size=8, shift_size=0).eval()
        st = load_random(blk, 22)
        gen = torch.Generator().manual_seed(8)
        x = torch.randn(1, 256, 32, generator=gen)
        mask = (torch.rand(1, 1, 16, 16, generator=gen) > 0.5).float()
        out["input_mask"] = dict(checksum=state_checksum(st), y=pack(blk(x, mask)))

        net = m.Uformer(**WIN16_CFG).eval()
        st = load_random(net, 31)
        x = torch.rand(1, 3, 128, 128, generator=torch.Generator().manual_seed(5))
        out["uformer_win16"] = dict(cfg=WIN16_CFG, checksum=state_checksum(st), y=pack(net(x)))

        # tests/test_host_path_cpu.py::test_arbitrary_resolution_restore_through_contract_model: the uformer_t1_128 model restores a
        # 200x150 image padded to 256x256 (test/test_sidd.py:79-108); stored: the valid region of the restored image
        g = torch.load(os.path.join(HERE, "uformer_t1_128.pt"), weights_only=False)
        net = m.Uformer(**g["cfg"]).eval()
        load_random(net, g["seed"])
        torch.manual_seed(3)
        noisy = torch.rand(1, 3, 200, 150)
        padded, mask = U.expand2square(noisy, factor=128)
        restored = torch.masked_select(net(padded), mask.bool()).reshape(1, 3, 200, 150).clamp(0, 1)
        out["restore_200x150"] = dict(y=pack(restored))

    out["block_autograd"] = []
    for dim, heads, H, shift, modu, dp, xseed in BLOCK_AUTOGRAD:
        ref = m.LeWinTransformerBlock(dim, (H, H), heads, win_size=8, shift_size=shift, modulator=modu, drop_path=dp).train()
        st = load_random(ref, 21)
        gen = torch.Generator().manual_seed(xseed)
        x = torch.randn(4, H * H, dim, generator=gen).requires_grad_(True)
        gout = torch.randn(4, H * H, dim, generator=gen)
        torch.manual_seed(99)                                        # the stochastic-depth draws (model.py:986-987)
        y = ref(x)
        y.backward(gout)
        out["block_autograd"].append(dict(case=(dim, heads, H, shift, modu, dp, xseed), checksum=state_checksum(st), y=pack(y), dx=pack(x.grad),
                                          grads={k: pack(p.grad, CAP_PARAM) for k, p in ref.named_parameters()}))

    out["samplers"] = {}
    for name, ref, shape, seed in [("down", m.Downsample(16, 32), (2, 256, 16), 91), ("up", m.Upsample(32, 8), (2, 64, 32), 92),
                                   ("leff", m.LeFF(16, 64), (2, 256, 16), 93)]:
        st = load_random(ref, 3)
        gen = torch.Generator().manual_seed(seed)
        x = torch.randn(*shape, generator=gen).requires_grad_(True)
        y = ref(x)
        y.backward(torch.randn(y.shape, generator=gen))
        out["samplers"][name] = dict(shape=shape, seed=seed, checksum=state_checksum(st), y=pack(y), dx=pack(x.grad),
                                     grads={k: pack(p.grad, CAP_PARAM) for k, p in ref.named_parameters()})

    net = m.Uformer(**UFORMER_B_CFG)
    with contextlib.redirect_stdout(io.StringIO()):                 # the reference prints per-layer GFLOPs
        flops = net.flops()
    out["uformer_b"] = dict(cfg=UFORMER_B_CFG, drop_path_rates=drop_path_rates(net), flops=flops)

    path = os.path.join(HERE, "reference_checks.pt")
    torch.save(out, path)
    print("reference_checks %8.1f KB" % (os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
