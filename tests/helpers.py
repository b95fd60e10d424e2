"""Shared helpers for the parity tests."""
import os

import torch

from paramgen import randomize_state

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# north_star tolerances: 1e-3 relative for fp32 arithmetic, 1e-2 for bf16 arithmetic.
TOL_FP32 = 1e-3
TOL_BF16 = 1e-2


def load_golden(name):
    g = torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)
    if "x" not in g and "x_seed" in g:                    # large inputs are re-derived from their seed instead of stored
        g["x"] = torch.rand(*g["x_shape"], generator=torch.Generator().manual_seed(g["x_seed"]))
    return g


def golden_names(kind):
    out = []
    for f in sorted(os.listdir(GOLDEN)):
        if f.endswith(".pt"):
            g = torch.load(os.path.join(GOLDEN, f), weights_only=False)
            if g["kind"] == kind:
                out.append(f[:-3])
    return out


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def rel_max(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30)).item()


def rel_l2_sampled(t, ref):
    """rel-L2 of `t` against a stored sample of a reference tensor (dict(stride, sample, norm), see
    golden/make_reference_checks.py): the larger of the error over the sample and the relative difference of the norms."""
    t = t.detach()
    return max(rel_l2(t.reshape(-1)[::ref["stride"]], ref["sample"]), abs(float(t.double().norm()) - ref["norm"]) / ref["norm"])


def max_err_sampled(t, ref):
    """max |t - ref| over a stored sample of a reference tensor, relative to the full reference tensor's max |ref|."""
    return float((t.detach().reshape(-1)[::ref["stride"]].double() - ref["sample"].double()).abs().max()) / ref["absmax"]


def state_checksum(state):
    s = 0.0
    for k in sorted(state):
        if torch.is_floating_point(state[k]):
            s += float(state[k].double().abs().sum())
    return s


def build_module(g):
    """Construct OUR module for a golden fixture (CPU), load the seeded synthetic weights, return (module, state)."""
    import uformer_b200 as U
    kind = g["kind"]
    if kind == "wattn":
        mod = U.WindowAttention(g["dim"], win_size=(g.get("ws", 8),) * 2, num_heads=g["heads"])
    elif kind == "leff":
        mod = U.LeFF(g["dim"], 4 * g["dim"])
    elif kind == "down":
        mod = U.Downsample(g["cin"], g["cout"])
    elif kind == "up":
        mod = U.Upsample(g["cin"], g["cout"])
    elif kind == "block":
        mod = U.LeWinTransformerBlock(g["dim"], (max(g["H"], 32),) * 2 if g.get("ws", 8) == 16 else (g["H"], g["H"]), g["heads"], win_size=g.get("ws", 8),
                                      shift_size=g["shift"], modulator=g["modulator"])
    elif kind == "model":
        mod = U.Uformer(**g["cfg"])
    else:
        raise KeyError(kind)
    st = randomize_state(mod.state_dict(), g["seed"], g.get("gain", 1.0))
    mod.load_state_dict(st, strict=True)
    return mod.eval(), st


def model_tolerances(g):
    """(full-output, residual-branch) rel-L2 bounds for a whole-model fixture: north_star's 1e-2 (bf16 arithmetic) on the
    output; the residual branch out - x gets 2x (the identity term hides error, SURVEY §8c).  No fixture-specific slack: the
    engine's default precision mode (fp32 residual stream inside a stage) must meet the plain bound on every fixture,
    including the 40-block flagship with the bench's O(1)-activation weights, where the reference's own bf16-autocast forward
    is 1.3e-2 away from its fp32 forward (recorded in the fixture as `ref_bf16` for information)."""
    return TOL_BF16, 2 * TOL_BF16


def oracle_run(g, st, x, dtype=torch.float32, mask=None):
    """Run the CPU oracle for a fixture description."""
    from oracle import lewin_oracle as O
    st = {k: (v.to(dtype) if torch.is_floating_point(v) else v) for k, v in st.items()}
    x = x.to(dtype)
    kind = g["kind"]
    if kind == "wattn":
        return O.window_attention(x, st, "", g["heads"], g.get("ws", 8), None if mask is None else mask.to(dtype))
    if kind == "leff":
        return O.leff(x, st, "")
    if kind == "down":
        return O.downsample(x, st["conv.0.weight"], st["conv.0.bias"])
    if kind == "up":
        return O.upsample(x, st["deconv.0.weight"], st["deconv.0.bias"])
    if kind == "block":
        return O.lewin_block(x, st, "", g["heads"], g.get("ws", 8), g["shift"])
    if kind == "model":
        c = g["cfg"]
        return O.uformer_forward(x, st, c["img_size"], c["embed_dim"], c["depths"], win_size=c["win_size"])
    raise KeyError(kind)
