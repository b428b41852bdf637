"""CPU self-test of oracle/tc_bound.py, the error bound of the tensor-core forward (csrc/tc_mlp.cuh).

Soundness: a float32 numpy emulation of the kernel's arithmetic -- tf32 operands formed with the kernel's integer
rounding, tensor-core sums truncated to float32 after every addition in a random order, tanh.approx perturbed by the
full 2^-10.987 with adversarial signs, the head's float32 FMA chains in the kernel's order -- stays inside the bound
for many policies and observation rows (1e4-sized rows, exact zeros, ties at the tf32 rounding point).
Power: the bound rejects three planted faults of the same emulation (b2 missing from one 16-column chunk, one row of
the action head shifted by one hidden unit, the layer-1 bias column dropped)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ppo_oracle as po  # noqa: E402
from oracle.tc_bound import TANH_REL, tc_forward_bound, tf32_rna  # noqa: E402

SCALES = np.array([3.0] * 3 + [4.0] * 3 + [2.0] * 3 + [10.0] * 3 + [1.0] * 3)
PERTURB = [0.01, 0.03, 0.1, 0.3]        # 0.1 to 3 times the 0.1 perturbation of the GPU tests


def _policy(seed, sigma):
    g = torch.Generator().manual_seed(seed)
    flat = po.init_params(seed, dtype=torch.float64) + sigma * torch.randn(po.N_PARAMS, generator=g, dtype=torch.float64)
    return flat.float().numpy()


def _rows(rng, B):
    x = rng.standard_normal((B, 15)) * SCALES
    x[:8] *= 1e4                                                     # 1e4-sized rows
    x[8:12] = 0.0                                                    # exact zero rows
    x[12:40, rng.integers(0, 15, 28)] = 0.0
    x = x.astype(np.float32)
    tie = (x[40:120].view(np.uint32) & np.uint32(0xFFFFE000)) | np.uint32(0x1000)  # exactly half a tf32 ulp
    x[40:120] = tie.view(np.float32)
    return x


def _trunc32(s):
    """float64 -> float32, rounded toward zero"""
    f = s.astype(np.float32)
    over = np.abs(f.astype(np.float64)) > np.abs(s)
    f[over] = np.nextafter(f[over], np.float32(0))
    return f


def _tc_sum(a, w, rng):
    """sum_k a[b, k] w[j, k]: exact tf32 products, float32 partial sums truncated, k in a random order"""
    acc = np.zeros((a.shape[0], w.shape[0]), np.float32)
    for k in rng.permutation(a.shape[1]):
        acc = _trunc32(acc.astype(np.float64) + a[:, k:k + 1].astype(np.float64) * w[:, k].astype(np.float64))
    return acc


def _mufu(z, sign):
    """tanh.approx.f32 with its full relative error, in the direction `sign` (+-1 per element)"""
    return (np.tanh(z.astype(np.float64)) * (1 + sign * TANH_REL * (1 - 2.0 ** -12))).astype(np.float32)


def _fma(a, b, c):
    return (a.astype(np.float64) * b + c).astype(np.float32)


def _emulate(theta, x, rng, signs, fault=None):
    """float32 emulation of tc::forward -> (mean [B, 4], value [B])"""
    p = {k: v.numpy() for k, v in po.unpack(torch.from_numpy(theta)).items()}
    B = x.shape[0]
    xt = np.concatenate([tf32_rna(x), np.ones((B, 1), np.float32)], 1)
    outs = []
    for t in ("pi", "vf"):
        W1 = np.concatenate([p[f"{t}.W1"], p[f"{t}.b1"][:, None]], 1)
        if fault == "bias_column":
            W1[:, 15] = 0
        b2, W3 = p[f"{t}.b2"].copy(), p[f"{t}.W3"].copy()
        if fault == "b2_chunk":
            b2[16:32] = 0
        if fault == "w3_shift" and t == "pi":
            W3[0] = np.roll(W3[0], 1)
        d1 = _tc_sum(xt, tf32_rna(W1), rng)
        s1 = rng.choice([-1.0, 1.0], d1.shape) if signs == "random" else np.full(d1.shape, float(signs == "up") * 2 - 1)
        h1 = tf32_rna(_mufu(d1, s1))
        v = _tc_sum(h1, tf32_rna(p[f"{t}.W2"]), rng) + b2              # add2: float32
        # layer-2 signs: random, all up / down, or aligned with the first output's head weights (errors add up there)
        s2 = {"random": rng.choice([-1.0, 1.0], v.shape), "up": np.ones(v.shape), "down": -np.ones(v.shape),
              "head": np.broadcast_to(np.sign(W3[0]) * np.sign(np.tanh(v.astype(np.float64))), v.shape)}[signs]
        h2 = _mufu(v, s2)
        if t == "pi":
            out = np.broadcast_to(p["pi.b3"], (B, 4)).astype(np.float32)
            for i in range(64):
                out = _fma(W3[:, i][None], h2[:, i:i + 1], out)
        else:
            even = np.full(B, p["vf.b3"][0], np.float32)
            odd = np.zeros(B, np.float32)
            for i in range(0, 64, 2):
                even = _fma(W3[0, i], h2[:, i], even)
                odd = _fma(W3[0, i + 1], h2[:, i + 1], odd)
            out = even + odd
        outs.append(out)
    return outs[0], outs[1]


def _excess(theta, x, fault, rng, signs):
    m_ref, v_ref, mb, vb = tc_forward_bound(theta, x)
    m, v = _emulate(theta, x, rng, signs, fault)
    return max(float((np.abs(m - m_ref) / mb).max()), float((np.abs(v - v_ref) / vb).max())), (m_ref, v_ref, mb, vb)


def test_bound_is_sound_under_adversarial_emulation():
    rng = np.random.default_rng(0)
    worst, rel = 0.0, []
    for seed in range(3):
        for sigma in PERTURB:
            theta = _policy(seed, sigma)
            x = _rows(rng, 600)
            for signs in ("random", "up", "down", "head"):
                r, (m_ref, v_ref, mb, vb) = _excess(theta, x, None, rng, signs)
                worst = max(worst, r)
            rel.append(np.concatenate([(mb / np.maximum(1, np.abs(m_ref))).ravel(), vb / np.maximum(1, np.abs(v_ref))]))
    rel = np.concatenate(rel)
    med = float(np.median(rel))
    print(f"tc bound: worst emulated err/bound {worst:.3f}; bound / max(1, |ref|): median {med:.2e}, "
          f"99th percentile {np.percentile(rel, 99):.2e}, max {rel.max():.2e}")
    assert worst <= 1.0
    assert med < 1e-2, "the bound should be well below the flat 2e-2 it replaces"


def test_reference_is_the_oracle_forward():
    theta = _policy(1, 0.1)
    x = _rows(np.random.default_rng(1), 300)
    m_ref, v_ref, mb, vb = tc_forward_bound(theta, x)
    rm, rv, _ = po.forward(torch.from_numpy(theta).double(), torch.from_numpy(x).double())
    assert np.array_equal(m_ref, rm.numpy()) and np.array_equal(v_ref, rv.numpy())
    assert mb.shape == (300, 4) and vb.shape == (300,) and (mb > 0).all() and (vb > 0).all()


def test_tf32_rounding_is_round_half_away():
    x = np.array([1.0, 1 + 2.0 ** -11, 1 + 3 * 2.0 ** -11, -(1 + 2.0 ** -11), 1 + 2.0 ** -11 - 2.0 ** -23, 0.0, -0.0, 1e4],
                 np.float32)
    want = np.array([1.0, 1 + 2.0 ** -10, 1 + 4 * 2.0 ** -11, -(1 + 2.0 ** -10), 1.0, 0.0, -0.0, 1e4], np.float32)
    assert np.array_equal(tf32_rna(x).view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("fault", ["b2_chunk", "w3_shift", "bias_column"])
def test_bound_rejects_planted_faults(fault):
    rng = np.random.default_rng(2)
    theta = _policy(4, 0.1)
    x = _rows(rng, 600)
    r, _ = _excess(theta, x, fault, rng, "random")
    print(f"{fault}: worst err/bound {r:.3g}")
    assert r > 1.0
