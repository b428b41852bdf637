"""TEST INFRASTRUCTURE: a per-element error bound for the tensor-core policy / value forward (csrc/tc_mlp.cuh).

The reference is ``ppo_oracle.forward`` of the float32 parameters in float64: the function SB3 computes and the one
the fp32 CUDA-core kernels are held to.  ``tc::forward`` departs from it in these steps, each bounded here:

  operands     observations: to_tf32_fast (add 0x1000, the tensor core ignores the low 13 bits = round to nearest,
               ties away from zero); W1 with b1 in column 15, and W2: cvt.rna.tf32 (the same rounding); H1: to_tf32_fast.
               Modelled exactly -- the rounded operands are formed here with the kernel's integer ops.
  MMA          products of tf32 operands are exact in float32; the float32 accumulation of K terms is bounded generously
               by K * 2^-23 * sum |terms| (one truncation per addition), so no adder detail is assumed.
  tanh         tanh.approx.f32: relative error <= 2^-10.987 (PTX ISA).  An input error e passes through with the largest
               slope of tanh over [z - e, z + e] (<= 1).  The H1 errors are shared by every unit of layer 2: they are
               carried to each output through its linearised sensitivity, with the second-order remainder of layer 2's
               tanh (<= 0.385 d^2) added, so they are not counted once per unit.
  head         b2 added in float32 (add2), then the float32 FMA chain of the head (64 terms; the value's even / odd
               chains and their final add are 65 roundings at most): gamma_65 * (|b3| + sum |w h|).

Errors are propagated as a first-order sum of magnitudes, per sample and per output, plus that remainder.  b2, W3, b3 and log_std are
used in full float32, as the kernel does.  Rows must be finite.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ppo_oracle as po

U = 2.0 ** -24                 # float32 unit roundoff
TANH_REL = 2.0 ** -10.987      # tanh.approx.f32, max relative error
TF32_REL = 2.0 ** -11          # round to nearest with 10 explicit mantissa bits
CHUNK = 1 << 15


def tf32_rna(x):
    """float32 -> float32 holding the tf32 value: round to nearest, ties away from zero (finite inputs)."""
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def _slope(z, e):
    """largest |tanh'| over [z - e, z + e]"""
    with np.errstate(over="ignore"):
        return 1.0 / np.cosh(np.maximum(np.abs(z) - e, 0.0)) ** 2


def _tower(p, t, x32):
    """(reference output [B, nout], bound [B, nout]) of one tower for float32 rows x32 [B, 15]."""
    W1 = np.concatenate([p[f"{t}.W1"], p[f"{t}.b1"][:, None]], 1)          # [64, 16]: bias in column 15
    W2, b2, W3, b3 = p[f"{t}.W2"], p[f"{t}.b2"], p[f"{t}.W3"], p[f"{t}.b3"]
    W1t = tf32_rna(W1.astype(np.float32)).astype(np.float64)
    W2t = tf32_rna(W2.astype(np.float32)).astype(np.float64)
    ones = np.ones((x32.shape[0], 1))
    A = np.concatenate([x32.astype(np.float64), ones], 1)
    At = np.concatenate([tf32_rna(x32).astype(np.float64), ones], 1)
    # layer 1 on the tensor cores
    z1 = A @ W1.T
    e1 = np.abs(At @ W1t.T - z1) + 16 * 2.0 * U * (np.abs(At) @ np.abs(W1t).T)
    t1 = np.tanh(z1)
    a1 = _slope(z1, e1) * e1
    eh1 = a1 + (np.abs(t1) + a1) * (TANH_REL + TF32_REL * (1 + TANH_REL))      # MUFU, then to_tf32_fast
    # layer 2 on the tensor cores, b2 added in float32.  E2: magnitude bound of the error of D2 + b2; p2: its part that
    # belongs to one unit alone (W2 rounding, accumulation, the b2 add)
    z2 = t1 @ W2.T + b2
    mag1 = np.abs(t1) + eh1
    p2 = np.abs(t1 @ (W2t - W2).T) + 64 * 2.0 * U * (mag1 @ np.abs(W2t).T)
    E2 = p2 + eh1 @ np.abs(W2t).T
    p2 = p2 + U * (np.abs(z2) + E2)
    E2 = E2 + U * (np.abs(z2) + E2)
    t2 = np.tanh(z2)
    s2 = 1.0 / np.cosh(z2) ** 2
    a2 = _slope(z2, E2) * E2
    # per output o: the H1 errors are shared by all 64 units of layer 2, so they enter through the linearised
    # sensitivity g_k = sum_j W3_oj tanh'(z2_j) W2t_jk; the rest is per unit: tanh(z2 + d) - tanh(z2) - tanh'(z2) d
    # is at most max|tanh''| / 2 * d^2 <= 0.385 d^2, then the MUFU error of layer 2 and the head's FMA chain
    unit = s2 * p2 + 0.385 * E2 ** 2 + TANH_REL * (np.abs(t2) + a2)
    eh2 = a2 + TANH_REL * (np.abs(t2) + a2)
    y = t2 @ W3.T + b3
    bound = np.empty_like(y)
    for o in range(W3.shape[0]):
        g = (s2 * W3[o]) @ W2t
        bound[:, o] = (np.abs(g) * eh1).sum(1) + unit @ np.abs(W3[o])
    bound += 1.01 * 65 * U * (np.abs(b3) + (np.abs(t2) + eh2) @ np.abs(W3).T)
    return y, bound


def tc_forward_bound(theta32, obs32):
    """theta32: float32 parameter vector [10697]; obs32: float32 rows [B, 15] (finite).
    Returns float64 (mean_ref [B, 4], value_ref [B], mean_bound [B, 4], value_bound [B]): the reference
    po.forward of the float32 parameters, and per element a bound on |tc::forward - reference|."""
    theta = torch.as_tensor(np.asarray(theta32, np.float32)).double()
    x32 = np.asarray(obs32, np.float32)
    assert np.isfinite(x32).all(), "the bound covers finite rows only"
    p = {k: v.numpy() for k, v in po.unpack(theta).items()}
    out = [[], [], [], []]
    for s in range(0, x32.shape[0], CHUNK):
        xc = x32[s:s + CHUNK]
        m_ref, v_ref, _ = po.forward(theta, torch.from_numpy(xc).double())
        _, mb = _tower(p, "pi", xc)
        _, vb = _tower(p, "vf", xc)
        for lst, a in zip(out, (m_ref.numpy(), v_ref.numpy(), mb, vb[:, 0])):
            lst.append(a)
    return tuple(np.concatenate(o) if o else np.zeros((0,)) for o in out)
