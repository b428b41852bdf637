"""The data-parallel update (csrc/ppo_dp.cuh) against float64 at every world size one GPU can hold, and the peer-backend
PPO loop teacher-forced per optimiser step.

Every simulated rank is one dronecu_ppo handle with its own CUDA stream; the mailboxes are wired with raw pointers
(``dronecu_ppo_dp_connect(world, NULL, mailboxes)``), so the push / flag / wait / fixed-order sum runs exactly as across
GPUs, with the peers' slots in the same HBM.

  a. ``ppo_apply_dp_kernel`` (A) and ``dp_allreduce_f64_kernel`` (R) at world 1, 2, 3, 4, 5, 8 and 16, over the sequence
     A A R A R R A A A R A R R A R A: both kernels at both mailbox parities, each after itself and after the other.
     After every exchange, on every rank:
       - the gradient is the float32 sum of the rank vectors in rank order 0 .. world-1, bit for bit, and within
         gamma_{world-1} sum_r |g_r| of the float64 sum (gamma_k = k 2^-24 / (1 - k 2^-24));
       - parameters, Adam moments, the Adam clock, ``info`` and ``info_sum`` are bit-identical across the ranks and equal
         ``dronecu_ppo_apply`` of that sum with inv_count = 1 / f32(count) on a separate handle;
       - the step is within the bounds of test_gpu_update_parity._check_step against float64 clip_grad_norm_ + Adam of
         the device's summed gradient.  The count the kernel divides by is the float32 sum of the float32 counts; above
         2^24 (counts 8,388,609 + r) it is rounded, and the test asserts |f32(sum) - sum| <= gamma_{world-1} sum: the
         applied step's scale is within that relative error of SB3's 1 / (sample count);
       - the all-reduce is ((0.0 + x_0) + x_1) + ... in float64, bit for bit (NaN compared only as NaN; an index that is
         -0.0 on every rank becomes +0.0 through the leading 0.0), over lengths 1 .. 5376 with the 2-float push tail,
         several values per thread and a slot filled exactly, and the buffer past n untouched;
       - a NaN and an inf in one rank's gradient poison every parameter and moment, as they do in torch.
     Host-side rejections (all-reduce of 0 or 5377 values, a misaligned buffer or gradient, an unconnected handle, a
     second connect, a connect with a world the mailbox was not sized for) launch nothing: the exchange count stays and
     the next exchange is checked like every other.
  b. the same kernels captured into one CUDA graph per rank and replayed three times: bit-identical to the same exchanges
     issued eagerly on fresh handles (PPO captures an epoch this way with dp_backend="peer").
  c. ``PPO.collect_rollouts()`` + ``PPO.train()`` with world 2, 3 and 4: one thread per rank under its own stream, the
     models built with a stand-in for the four torch.distributed calls PPO makes.  Every optimiser step: each rank's rows
     are its own partition / permutation slice, the advantage statistics are bit-identical across ranks and equal the
     float64 moments of the union, the summed gradient is the rank-order float32 sum of the ranks' own gradients and
     within the update-parity tolerance of the float64 gradient over the union, the step passes _check_step, and the
     replicas stay bit-identical.  At the end the logs agree across ranks, the explained variance matches float64 over
     the union within the rounding of the float32 moments it is formed from, and with one minibatch per epoch the
     parameters match one rank training on the union.

Ranks on one GPU progress only if their kernels run at the same time, so every rank stream is created fresh, one after
another (the driver hands out its hardware queues round robin), and worlds above 3, and every PPO loop, run in a
spawned child with CUDA_DEVICE_MAX_CONNECTIONS=32 (a per-process driver setting; the default of 8 queues would serialise
two ranks behind each other).  Before the rank threads start, a warm-up takes out of them what synchronises the whole
device on a first run: kernel loading, the partition scratch and new allocator segments.  Nothing synchronises the whole device while a rank has an exchange outstanding, and every handle has a
20-second exchange time-out, so a harness mistake ends as a timed-out status and a failed assertion.
"""
import contextlib
import ctypes as C
import math
import multiprocessing
import os
import queue
import threading
import time
import traceback

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import philox  # noqa: E402
from tests.test_gpu_tc import _separated_buffers  # noqa: E402
from tests.test_gpu_update_parity import (HYPER, N, P, _check_step, _grad_error, _normalised, _ref_grad,  # noqa: E402
                                          _spy_train, _torch_step, f32)

GRAD_LEN = N + 8
U = 2.0 ** -24
TIMEOUT_S = 20.0                 # exchange time-out on every handle
CHILD_TIMEOUT_S = 900.0
WORLDS = (1, 2, 3, 4, 5, 8, 16)
MAX_F64 = 5376                   # kDpSlot / 2


def gamma(k):
    return k * U / (1.0 - k * U)


@pytest.fixture(scope="module")
def drl():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import drone_rl_b200
    import drone_rl_b200.ppo  # noqa: F401
    return drone_rl_b200


# ------------------------------------------------------------------------------------------------------------------------
# harness
# ------------------------------------------------------------------------------------------------------------------------
def _run(world, fn, *args, in_process_max=3):
    """fn(world, *args) -> report: in this process up to world ``in_process_max``, above in a spawned child with 32
    hardware queues."""
    if world <= in_process_max:
        return fn(world, *args)
    ctx = multiprocessing.get_context("spawn")
    q = ctx.Queue()
    old = os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS")
    os.environ["CUDA_DEVICE_MAX_CONNECTIONS"] = "32"
    try:
        p = ctx.Process(target=_child, args=(fn.__name__, world, args, q))
        p.start()
    finally:
        if old is None:
            del os.environ["CUDA_DEVICE_MAX_CONNECTIONS"]
        else:
            os.environ["CUDA_DEVICE_MAX_CONNECTIONS"] = old
    out, deadline = None, time.monotonic() + CHILD_TIMEOUT_S
    try:
        while out is None and time.monotonic() < deadline:
            try:
                out = q.get(timeout=2.0)
            except queue.Empty:
                if not p.is_alive():
                    try:
                        out = q.get(timeout=5.0)
                    except queue.Empty:
                        out = ("err", f"the child exited with code {p.exitcode} and no result")
    finally:
        p.join(timeout=60)
        if p.is_alive():
            p.kill()
            p.join()
    assert out is not None, f"world {world}: no result within {CHILD_TIMEOUT_S:.0f} s"
    assert out[0] == "ok", out[1]
    return out[1]


def _child(name, world, args, q):
    try:
        q.put(("ok", globals()[name](world, *args)))
    except BaseException:
        q.put(("err", traceback.format_exc()))


def _rank_streams(world):
    """``world`` non-blocking streams created one after another: consecutive hardware queues, and never ordered by the
    legacy default stream."""
    torch.cuda.init()
    rt = C.CDLL("libcudart.so.12")
    out = []
    for _ in range(world):
        s = C.c_void_p()
        assert rt.cudaStreamCreateWithFlags(C.byref(s), 1) == 0
        out.append(torch.cuda.ExternalStream(s.value))
    return out


def _destroy_streams(streams):
    rt = C.CDLL("libcudart.so.12")
    for s in streams:
        rt.cudaStreamDestroy(C.c_void_p(s.cuda_stream))


def _same(a, b):
    """Bit-identical, except that a NaN only has to meet a NaN."""
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    ui = {4: np.uint32, 8: np.uint64}[a.dtype.itemsize]
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a.view(ui)[~na], b.view(ui)[~nb]))


class Ranks:
    """``world`` optimiser handles (default configuration) wired into one exchange with raw mailbox pointers, each with
    its stream, info row and info accumulator."""

    def __init__(self, lib, world, streams):
        from drone_rl_b200 import _lib
        self.lib, self.world, self.streams = lib, world, streams
        self.cfg = _lib.PPOConfig()
        lib.dronecu_ppo_config_default(C.byref(self.cfg))
        self.h, mails = [], []
        for r in range(world):
            h, mail = C.c_void_p(), C.c_void_p()
            _lib.check(lib.dronecu_ppo_create(C.byref(self.cfg), 0, C.byref(h)))
            _lib.check(lib.dronecu_ppo_dp_alloc(h, r, world, None, C.byref(mail)))
            self.h.append(h)
            mails.append(mail.value)
        self.mails = (C.c_void_p * world)(*mails)
        self.info = [torch.zeros(9, device="cuda") for _ in range(world)]
        self.info_sum = [torch.zeros(10, device="cuda") for _ in range(world)]
        for r, h in enumerate(self.h):
            _lib.check(lib.dronecu_ppo_dp_connect(h, world, None, self.mails))
            _lib.check(lib.dronecu_ppo_dp_set_timeout(h, TIMEOUT_S))
            _lib.check(lib.dronecu_ppo_set_info_accumulator(h, P(self.info_sum[r])))

    def st(self, r):
        return C.c_void_p(self.streams[r].cuda_stream)

    def apply(self, r, params, grad):
        from drone_rl_b200 import _lib
        _lib.check(self.lib.dronecu_ppo_apply_dp(self.h[r], P(params), P(grad), P(self.info[r]), self.st(r)), "apply_dp")

    def allreduce(self, r, buf, n):
        from drone_rl_b200 import _lib
        _lib.check(self.lib.dronecu_ppo_dp_allreduce_f64(self.h[r], P(buf), n, self.st(r)), "allreduce_f64")

    def status(self):
        """[(status, exchanges)] per rank; the caller has synchronised the device (every exchange issued)."""
        out = []
        for h in self.h:
            st, n = C.c_int(), C.c_int64()
            assert self.lib.dronecu_ppo_dp_status(h, C.byref(st), C.byref(n)) == 0
            out.append((st.value, n.value))
        return out

    def state(self, r):
        return _handle_state(self.lib, self.h[r])

    def close(self):
        torch.cuda.synchronize()
        for h in self.h:
            self.lib.dronecu_ppo_destroy(h)
        self.h = []


def _handle_state(lib, h):
    from drone_rl_b200 import _lib
    mom, step = torch.empty(2 * N, device="cuda"), C.c_int64()
    _lib.check(lib.dronecu_ppo_get_state(h, P(mom), C.byref(step), None))
    torch.cuda.synchronize()
    return mom, step.value


# ------------------------------------------------------------------------------------------------------------------------
# connect validation
# ------------------------------------------------------------------------------------------------------------------------
def test_connect_accepts_only_the_allocated_world_and_only_once(drl):
    """The mailbox holds 2 x world slots and its flags sit behind them: a handle connected with another world than it was
    allocated for would index slots and flags with the wrong world, and a larger one would write past every mailbox; a
    second connect would re-map (and leak) the peers.  Both are refused.  Nothing here launches an exchange."""
    from drone_rl_b200 import _lib
    lib = _lib.load()
    cfg = _lib.PPOConfig()
    lib.dronecu_ppo_config_default(C.byref(cfg))
    hs, mails = [], []
    for rank, world in ((0, 2), (1, 2), (1, 3)):
        h, mail = C.c_void_p(), C.c_void_p()
        _lib.check(lib.dronecu_ppo_create(C.byref(cfg), 0, C.byref(h)))
        _lib.check(lib.dronecu_ppo_dp_alloc(h, rank, world, None, C.byref(mail)))
        hs.append(h)
        mails.append(mail.value)
    try:
        pair, three = (C.c_void_p * 2)(*mails[:2]), (C.c_void_p * 3)(*mails)
        assert lib.dronecu_ppo_dp_connect(hs[0], 3, None, three) != 0, "a world larger than the mailbox was sized for"
        assert lib.dronecu_ppo_dp_connect(hs[2], 2, None, pair) != 0, "a world smaller than the mailbox was sized for"
        assert lib.dronecu_ppo_dp_connect(hs[0], 2, None, pair) == 0
        assert lib.dronecu_ppo_dp_connect(hs[1], 2, None, pair) == 0
        assert lib.dronecu_ppo_dp_connect(hs[0], 2, None, pair) != 0, "a second connect"
        for h in hs:
            st, n = C.c_int(), C.c_int64()
            _lib.check(lib.dronecu_ppo_dp_status(h, C.byref(st), C.byref(n)))
            assert (st.value, n.value) == (0, 0)
    finally:
        for h in hs:
            lib.dronecu_ppo_destroy(h)


# ------------------------------------------------------------------------------------------------------------------------
# a. both kernels at every world size
# ------------------------------------------------------------------------------------------------------------------------
SEQ = "AARARRAAARARRARA"
A_CASES = ("clipped", "unclipped", "zero", "big_clipped", "unclipped", "zero", "big_unclipped", "clipped", "nonfinite")
LENGTHS = (1, 2, 3, 4, 5, 1023, 1024, 1025, 2048, 2049, 5375, 5376)
SENTINEL = -1234.5
assert SEQ.count("A") == len(A_CASES) and SEQ[-1] == "A"          # the non-finite step is the last one: it poisons the state


def _rank_grads(case, world, g):
    """[world, GRAD_LEN] float32 sum-form gradients (mean gradient x count, statistics x count, count at N + 4) whose
    rank-order sum is in the regime of ``case``: clipped, unclipped, zero (ranks cancel pairwise, exactly), counts above
    2^24 in total, or a NaN and an inf on one rank."""
    big = case.startswith("big")
    counts = [8388609 + r for r in range(world)] if big else [int(c) for c in torch.randint(1, 5000, (world,), generator=g)]
    scale = {"clipped": 0.1, "unclipped": 1e-4, "zero": 1.0, "nonfinite": 1e-3}[case.split("_")[-1]]
    rows = []
    for r in range(world):
        v = torch.cat([scale * torch.randn(N, generator=g, dtype=torch.float64),
                       torch.tensor([0.3, 2.0, 0.01, 0.2, 0.0, 0.1, 0.1, 0.1], dtype=torch.float64)
                       + 0.1 * torch.randn(8, generator=g, dtype=torch.float64)]) * counts[r]
        v[N + 4] = counts[r]
        rows.append(v.float().numpy())
    G = np.stack(rows)
    if case == "zero":
        for r in range(1, world, 2):
            G[r, :N] = -G[r - 1, :N]
        if world % 2:
            G[world - 1, :N] = 0.0
    if case == "nonfinite":
        G[world // 2, 5] = np.nan
        G[world // 2, 4321] = np.inf
    return G, counts


def _f32_rank_sum(G):
    acc = G[0].copy()
    with np.errstate(all="ignore"):
        for r in range(1, G.shape[0]):
            acc = acc + G[r]                  # numpy float32 adds: round to nearest, as the kernel's FADD
    return acc


KINDS = ("negzero", "cancel", "subnormal", "inf", "inf_minus_inf", "nan", "f32_nan_halves", "f32_subnormal_halves")


def _special(X, p, kind, world):
    """Put one adversarial pattern at index p of every rank's values X [world, n] (float64)."""
    bits = X.view(np.uint64)
    if kind == "negzero":
        X[:, p] = -0.0
    elif kind == "cancel":                                    # 1e16 + 1 - 1e16: 0 in float64, in this order
        X[:, p] = 0.0
        for r, v in zip(range(world), (1e16, 1.0, -1e16)):
            X[r, p] = v
    elif kind == "subnormal":
        X[:, p] = [(-1) ** r * (r + 1) * 2.5e-310 for r in range(world)]
    elif kind == "inf":
        X[0, p] = np.inf
    elif kind == "inf_minus_inf":
        X[0, p] = np.inf
        X[world - 1, p] = -np.inf if world > 1 else np.inf
    elif kind == "nan":
        X[world // 2, p] = np.nan
    elif kind == "f32_nan_halves":                            # the push moves floats: quiet and signalling NaN halves
        for r in range(world):
            bits[r, p] = ((0x3FF00000 + r) << 32 | 0x7FC00001) if r % 2 == 0 else (0x7FC00000 << 32 | (0x7F800001 + r))
    elif kind == "f32_subnormal_halves":
        for r in range(world):
            bits[r, p] = (0x00000001 << 32 | (r + 1)) if r % 2 == 0 else (0x3FF00000 << 32 | 0x007FFFFF)


def _allreduce_values(n, e, world, rng):
    X = rng.standard_normal((world, n)) * 10.0 ** rng.integers(-6, 7, size=(world, n))
    marks = set(range(min(n, 8))) | {n - 1 - k for k in range(8) if n - 1 - k >= 0}
    marks |= {b + k for b in (1023, 2047, 4095) for k in (-1, 0, 1, 2) if 0 <= b + k < n}
    negzero = []
    for p in sorted(marks):
        kind = KINDS[(p + e) % len(KINDS)]
        _special(X, p, kind, world)
        if kind == "negzero":
            negzero.append(p)
    return X, negzero


def _exchanges(world):
    from drone_rl_b200 import _lib
    lib, dev = _lib.load(), torch.device("cuda", 0)
    streams = _rank_streams(world)
    ranks = Ranks(lib, world, streams)
    cfg = ranks.cfg
    href = C.c_void_p()
    _lib.check(lib.dronecu_ppo_create(C.byref(cfg), 0, C.byref(href)))
    iref, isref = torch.zeros(9, device=dev), torch.zeros(10, device=dev)
    _lib.check(lib.dronecu_ppo_set_info_accumulator(href, P(isref)))
    g = torch.Generator().manual_seed(100 + world)
    rng = np.random.default_rng(world)
    theta0 = (0.1 * torch.randn(N, generator=g)).to(dev)
    params, pref = [theta0.clone() for _ in range(world)], theta0.clone()
    grads = [torch.zeros(GRAD_LEN, device=dev) for _ in range(world)]
    bufs = [torch.zeros(MAX_F64 + 2, dtype=torch.float64, device=dev) for _ in range(world)]
    acc_info = np.zeros(10, dtype=np.float32)
    worst = {"grad": 0.0, "step": 0.0, "count": 0.0}
    lengths, n_a, n_r = [], 0, 0
    try:
        for e, kind in enumerate(SEQ):
            if e == 8:
                _reject(lib, ranks, params, bufs, e, apply=True)
            if e == 9:
                _reject(lib, ranks, params, bufs, e, apply=False)
            what = f"world {world} exchange {e}"
            if kind == "A":
                case = A_CASES[n_a]
                n_a += 1
                G, counts = _rank_grads(case, world, g)
                for r in range(world):
                    grads[r].copy_(torch.from_numpy(G[r]))
                mom0, t0 = _handle_state(lib, href)
                th0 = pref.clone()
                torch.cuda.synchronize()
                for r in range(world):
                    ranks.apply(r, params[r], grads[r])
                S = _f32_rank_sum(G)
                count = np.float32(S[N + 4])
                inv = float(np.float32(1.0) / count)
                _lib.check(lib.dronecu_ppo_apply(href, P(pref), P(torch.from_numpy(S).to(dev)), inv, P(iref), None))
                torch.cuda.synchronize()
                # the summed gradient: rank-order float32 sum bit for bit, float64 sum within gamma_{world-1} sum |g_r|
                got = grads[0].cpu().numpy()
                for r in range(world):
                    assert _same(grads[r], S), f"{what} ({case}): rank {r} does not hold the rank-order float32 sum"
                fin = np.isfinite(S)
                S64, A64 = G.astype(np.float64).sum(0), np.abs(G.astype(np.float64)).sum(0)
                bound = gamma(world - 1) * A64[fin]
                err = np.abs(S[fin].astype(np.float64) - S64[fin])
                ratio = float((err / np.maximum(bound, 1e-300)).max()) if world > 1 else 0.0
                assert world > 1 or not err.any()
                assert (err <= bound).all(), f"{what}: f32 sum vs float64 err/bound {ratio:.3g}"
                worst["grad"] = max(worst["grad"], ratio)
                # replicas: bit-identical across ranks and to dronecu_ppo_apply of the sum
                mref, tref = _handle_state(lib, href)
                assert tref == t0 + 1
                for r in range(world):
                    mom, t = ranks.state(r)
                    assert t == tref, f"{what}: rank {r} Adam clock {t} != {tref}"
                    assert _same(params[r], pref) and _same(mom, mref), f"{what} ({case}): rank {r} != apply(sum)"
                    assert _same(ranks.info[r], iref) and _same(ranks.info_sum[r], isref), f"{what}: rank {r} info"
                # info = [statistics / count, count, pre-clip norm]; info_sum accumulates it and counts the steps
                info = iref.cpu().numpy()
                want = S[N:] * np.float32(inv)
                want[4] = count
                assert _same(info[:8], want), f"{what}: info {info[:8]} != {want}"
                acc_info[:9] += info
                acc_info[9] += np.float32(1.0)
                assert _same(isref, acc_info), f"{what}: info_sum"
                if case == "big_clipped" or case == "big_unclipped":
                    total = sum(counts)
                    c_err = abs(float(count) - total)
                    assert c_err <= gamma(world - 1) * total
                    worst["count"] = max(worst["count"], c_err / (gamma(world - 1) * total) if world > 1 else 0.0)
                if case == "nonfinite":                       # torch: a non-finite norm poisons every parameter
                    ref = _torch_step(th0, torch.from_numpy(got[:N]).double() * inv, mom0, t0, cfg)
                    assert bool(torch.isnan(ref[0]).all()) and bool(torch.isnan(pref).all())
                    assert bool(torch.isnan(mref).all()) and math.isnan(info[8])
                else:
                    ref = _torch_step(th0, torch.from_numpy(got[:N]).double() * inv, mom0, t0, cfg)
                    norm = ref[3]
                    regime = case.split("_")[-1]
                    assert {"clipped": norm > cfg.max_grad_norm, "unclipped": 0 < norm < cfg.max_grad_norm,
                            "zero": norm == 0}[regime], f"{what}: norm {norm} is not {regime}"
                    worst["step"] = max(worst["step"], _check_step(pref, mref, ref, cfg, what, float(info[8])))
            else:
                n = LENGTHS[(7 * WORLDS.index(world) + n_r) % len(LENGTHS)]
                n_r += 1
                lengths.append(n)
                X, negzero = _allreduce_values(n, e + world, world, rng)
                for r in range(world):
                    bufs[r].fill_(SENTINEL)
                    bufs[r][:n] = torch.from_numpy(X[r])
                torch.cuda.synchronize()
                for r in range(world):
                    ranks.allreduce(r, bufs[r], n)
                ref = np.zeros(n)
                with np.errstate(all="ignore"):
                    for r in range(world):
                        ref = ref + X[r]                      # ((0.0 + x_0) + x_1) + ...
                torch.cuda.synchronize()
                for r in range(world):
                    out = bufs[r].cpu().numpy()
                    assert _same(out[:n], ref), f"{what}: rank {r} all-reduce of {n} values"
                    assert (out[n:] == SENTINEL).all(), f"{what}: rank {r} wrote past n = {n}"
                    z = out[negzero]
                    assert (z == 0).all() and not np.signbit(z).any(), f"{what}: -0.0 on every rank must sum to +0.0"
        torch.cuda.synchronize()
        assert ranks.status() == [(0, len(SEQ))] * world
    finally:
        ranks.close()
        lib.dronecu_ppo_destroy(href)
        _destroy_streams(streams)
    return (f"world {world}: {len(SEQ)} exchanges, all-reduce lengths {lengths}; worst err/bound: gradient "
            f"{worst['grad']:.3g}, step {worst['step']:.3g}, count rounding {worst['count']:.3g}")


def _reject(lib, ranks, params, bufs, e, apply):
    """Arguments refused on the host: no launch, the exchange count stays (the next exchange then checks the mailbox)."""
    from drone_rl_b200 import _lib
    world = ranks.world
    torch.cuda.synchronize()
    before = ranks.status()
    assert before == [(0, e)] * world
    loose, mail = C.c_void_p(), C.c_void_p()
    _lib.check(lib.dronecu_ppo_create(C.byref(ranks.cfg), 0, C.byref(loose)))
    _lib.check(lib.dronecu_ppo_dp_alloc(loose, 0, 1, None, C.byref(mail)))
    spare = torch.zeros(GRAD_LEN + 4, device="cuda")
    try:
        if apply:
            for r in range(world):
                odd = C.c_void_p(spare.data_ptr() + 8)
                assert lib.dronecu_ppo_apply_dp(ranks.h[r], P(params[r]), odd, None, ranks.st(r)) != 0
                assert lib.dronecu_ppo_dp_connect(ranks.h[r], world, None, ranks.mails) != 0, "a second connect"
            assert lib.dronecu_ppo_apply_dp(loose, P(params[0]), P(spare), None, None) != 0, "not connected"
            two = (C.c_void_p * 2)(mail.value, ranks.mails[0])
            assert lib.dronecu_ppo_dp_connect(loose, 2, None, two) != 0, "connect with a world the mailbox was not sized for"
        else:
            for r in range(world):
                st = ranks.st(r)
                assert lib.dronecu_ppo_dp_allreduce_f64(ranks.h[r], P(bufs[r]), 0, st) != 0
                assert lib.dronecu_ppo_dp_allreduce_f64(ranks.h[r], P(bufs[r]), MAX_F64 + 1, st) != 0
                assert lib.dronecu_ppo_dp_allreduce_f64(ranks.h[r], C.c_void_p(bufs[r].data_ptr() + 8), 4, st) != 0
            assert lib.dronecu_ppo_dp_allreduce_f64(loose, P(bufs[0]), 4, None) != 0, "not connected"
        torch.cuda.synchronize()
        assert ranks.status() == before
    finally:
        lib.dronecu_ppo_destroy(loose)


@pytest.mark.parametrize("world", WORLDS)
def test_exchange_kernels_match_float64_at_every_world(drl, world):
    print(_run(world, _exchanges))


# ------------------------------------------------------------------------------------------------------------------------
# b. the exchange inside CUDA graphs
# ------------------------------------------------------------------------------------------------------------------------
SEQ_GRAPH = "ARAARRA"
N_GRAPH = 1025


def _graph_inputs(world):
    g = torch.Generator().manual_seed(7 * world)
    G, _ = _rank_grads("unclipped", world, g)
    X, _ = _allreduce_values(N_GRAPH, 3, world, np.random.default_rng(7 * world))
    X[np.isnan(X) | np.isinf(X)] = 1.0            # keep the repeated sums finite: the replays compare bits
    theta0 = 0.1 * torch.randn(N, generator=g)
    return G, X, theta0


def _graphs(world):
    from drone_rl_b200 import _lib
    lib, dev = _lib.load(), torch.device("cuda", 0)
    G, X, theta0 = _graph_inputs(world)
    streams = _rank_streams(world)
    out = {}
    try:
        for mode in ("graph", "eager"):
            ranks = Ranks(lib, world, streams)
            params = [theta0.to(dev) for _ in range(world)]
            grads = [torch.from_numpy(G[r]).to(dev) for r in range(world)]
            bufs = [torch.from_numpy(X[r]).to(dev) for r in range(world)]
            torch.cuda.synchronize()

            def issue(r):
                for kind in SEQ_GRAPH:
                    if kind == "A":
                        ranks.apply(r, params[r], grads[r])
                    else:
                        ranks.allreduce(r, bufs[r], N_GRAPH)
            try:
                if mode == "graph":
                    graphs = []
                    for r in range(world):                # one rank after another: capture executes nothing
                        gr = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(gr, stream=streams[r]):
                            issue(r)
                        graphs.append(gr)
                    torch.cuda.synchronize()
                    assert ranks.status() == [(0, 0)] * world, "capture must not execute an exchange"
                    for _ in range(3):
                        for r in range(world):
                            with torch.cuda.stream(streams[r]):
                                graphs[r].replay()
                    torch.cuda.synchronize()
                    del graphs
                else:
                    for _ in range(3):
                        for r in range(world):
                            issue(r)
                    torch.cuda.synchronize()
                out[mode] = [(params[r].cpu(), *ranks.state(r), grads[r].cpu(), bufs[r].cpu(), ranks.info[r].cpu(),
                              ranks.info_sum[r].cpu()) for r in range(world)]
                out[mode + "_status"] = ranks.status()
            finally:
                ranks.close()
    finally:
        _destroy_streams(streams)
    assert out["graph_status"] == out["eager_status"] == [(0, 3 * len(SEQ_GRAPH))] * world
    names = ("params", "moments", "Adam clock", "gradient", "all-reduced buffer", "info", "info_sum")
    for r in range(world):
        for name, a, b in zip(names, out["graph"][r], out["eager"][r]):
            assert a == b if name == "Adam clock" else _same(a, b), f"world {world} rank {r}: {name} of the replays"
            assert a == out["graph"][0][2] if name == "Adam clock" else _same(a, out["graph"][0][names.index(name)])
    return f"world {world}: 3 replays of {SEQ_GRAPH} per rank == the same exchanges issued eagerly, bit for bit"


@pytest.mark.parametrize("world", [2, 3, 8])
def test_exchange_inside_cuda_graphs_equals_eager(drl, world):
    print(_run(world, _graphs))


# ------------------------------------------------------------------------------------------------------------------------
# c. the peer-backend PPO loop, teacher-forced
# ------------------------------------------------------------------------------------------------------------------------
DP_CONFIGS = {
    # name: (n_envs per rank, n_steps, batch_size, n_epochs, PPO keywords, EnvConfig keywords, teacher-forced steps)
    "one_minibatch_fp32": (64, 16, 1024, 2, {}, {}, None),
    "one_minibatch_bf16": (64, 16, 1024, 2, {"update_precision": "bf16"}, {}, None),
    "ragged_tail": (5, 13, 16, 2, {}, {}, None),                     # 65 rows per rank: 4 x 16 + 1
    "per_minibatch_stats": (32, 160, 4, 1, {}, {}, 97),              # 1280 minibatches > _max_mb
    "permutation": (16, 64, 8, 1, {}, {}, None),                     # 128 minibatches > 64
    "no_normalisation": (16, 64, 256, 2, {"normalize_advantage": False}, {}, None),
    "tf32": (16, 64, 256, 2, dict(update_precision="tf32", **HYPER), {}, None),         # on SEPARATED data
    "norm_timeout": (16, 64, 256, 2, {"norm_obs": True, "norm_reward": True, "handle_timeout_termination": True},
                     {"max_steps": 7}, None),
}
# synthetic buffers whose old log-probs keep every sample away from the clip boundaries (tests/test_gpu_tc.py): a
# reduced-precision forward of a rollout buffer flips the clipped objective of the samples that sit on a boundary
SEPARATED = {"tf32"}
UNION_TOL = {"one_minibatch_fp32": 1e-6, "one_minibatch_bf16": 5e-6}     # the two-GPU test's bounds
SEED = 12


@contextlib.contextmanager
def _one_gpu_ranks(world):
    """PPO objects built in this thread as ranks of ``world``: a stand-in for the four torch.distributed calls
    PPO.__init__ / close make, and PPO._dp_setup replaced by nothing (cudaIpcOpenMemHandle cannot open a handle of its own
    process; the caller wires the mailboxes with raw pointers).  ``state["rank"]`` is the rank of the next model,
    ``state["on"] = False`` builds a plain one-rank model."""
    from drone_rl_b200.ppo import PPO
    dist = torch.distributed
    state = {"rank": 0, "on": True}
    names = ("is_initialized", "get_rank", "get_world_size", "barrier")
    saved, saved_setup = {k: getattr(dist, k) for k in names}, PPO._dp_setup
    dist.is_initialized = lambda: state["on"]
    dist.get_rank = lambda group=None: state["rank"]
    dist.get_world_size = lambda group=None: world
    dist.barrier = lambda *a, **k: None
    PPO._dp_setup = lambda self: None
    try:
        yield state
    finally:
        for k, v in saved.items():
            setattr(dist, k, v)
        PPO._dp_setup = saved_setup


def _ppo_loop(world, name):
    import drone_rl_b200 as drl
    from drone_rl_b200 import _lib
    from drone_rl_b200.ppo import PPO
    n, K, bs, E, kw, env_kw, every = DP_CONFIGS[name]
    B = n * K
    n_mb = (B + bs - 1) // bs
    steps = E * n_mb
    lib = _lib.load()
    streams = _rank_streams(world)
    models = []
    with _one_gpu_ranks(world) as state:
        try:
            for r in range(world):
                state["rank"] = r
                env = drl.DroneBatch(n, drl.EnvConfig.single(**env_kw), seed=SEED, env_offset=r * n)
                models.append(PPO(env, n_steps=K, batch_size=bs, n_epochs=E, seed=SEED, cuda_graph=False, **kw))
            mails = []
            for r, m in enumerate(models):
                assert m.world == world and m.rank == r and m.dp_backend == "peer"
                mail = C.c_void_p()
                _lib.check(lib.dronecu_ppo_dp_alloc(m._h, r, world, None, C.byref(mail)))
                mails.append(mail.value)
            arr = (C.c_void_p * world)(*mails)
            for m in models:
                _lib.check(lib.dronecu_ppo_dp_connect(m._h, world, None, arr))
                _lib.check(lib.dronecu_ppo_dp_set_timeout(m._h, TIMEOUT_S))
            if name == "per_minibatch_stats":
                assert n_mb > models[0]._max_mb
            if name in SEPARATED:
                for r, m in enumerate(models):
                    _separated_buffers(m, 7 + r, clip=m.cfg.clip_range)
                    m.buf.value.zero_()
                    if m.padded_obs:
                        m.buf.obs_store[..., 15] = 1.0
            state["on"] = False
            _warm_up(lib, models, streams, name)
            state["on"] = True
            forced = (lambda k: True) if every is None else (lambda k: k % every == 0 or k == steps - 1)
            recs, summed = [None] * world, [[] for _ in range(world)]
            errors, abort = [], threading.Event()

            def body(r):
                m = models[r]
                with torch.cuda.stream(streams[r]):
                    if name not in SEPARATED:
                        m.collect_rollouts()
                    own_step = m._minibatch

                    def step(index, first, mm, stats=None):
                        if abort.is_set():
                            raise RuntimeError("another rank failed")
                        own_step(index, first, mm, stats)
                        summed[r].append(m._grad.clone())
                        # a rank may run at most one exchange ahead: a failing peer costs one time-out, not one per step
                        torch.cuda.current_stream().synchronize()
                    m._minibatch = step
                    recs[r] = _spy_train(m, 1, forced, own_grad=True)

            def run(r):
                try:
                    body(r)
                except BaseException:
                    errors.append(traceback.format_exc())
                    abort.set()
            threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
            for t in threads:
                t.start()
            for t in threads:
                t.join(timeout=CHILD_TIMEOUT_S)
            assert not any(t.is_alive() for t in threads), f"{name}: a rank thread did not finish"
            assert not errors, errors[0]
            torch.cuda.synchronize()
            report = _check_ppo_loop(world, name, models, recs, summed, steps, n_mb)
            if name in UNION_TOL:
                state["on"] = False
                one = PPO(drl.DroneBatch(world * n, drl.EnvConfig.single(**env_kw), seed=SEED), n_steps=K,
                          batch_size=world * bs, n_epochs=E, seed=SEED, cuda_graph=False, **kw)
                one.collect_rollouts()
                one.train()
                err = float((models[0].params - one.params).abs().max())
                one.close()
                state["on"] = True
                assert err <= UNION_TOL[name], f"{name}: {world} ranks vs one rank on the union: {err:.3g}"
                report += f"; params vs one rank on the union {err:.3g} (<= {UNION_TOL[name]:g})"
            return report
        finally:
            torch.cuda.synchronize()
            for m in models:
                m.close()
            _destroy_streams(streams)


def _warm_up(lib, models, streams, name):
    """Take every device-wide synchronisation of a first run out of the rank threads, where it would wait for a peer's
    exchange that its own thread has not issued yet (the exchange then times out): the loading of each kernel on its first
    launch (CUDA lazy loading), the partition scratch the first dronecu_minibatch_partition allocates, and the caching
    allocator's cudaMalloc of new segments for the per-step clones.  A one-rank model of the same configuration runs the
    loop once and one one-rank exchange handle runs both exchange kernels; nothing here touches the ranks' models but
    their partition scratch."""
    import drone_rl_b200 as drl
    from drone_rl_b200 import _lib
    from drone_rl_b200.ppo import PPO
    n, K, bs, E, kw, env_kw, _ = DP_CONFIGS[name]
    B = n * K
    one = PPO(drl.DroneBatch(n, drl.EnvConfig.single(**env_kw), seed=SEED + 1), n_steps=K, batch_size=bs, n_epochs=E,
              seed=SEED, cuda_graph=False, **kw)
    one.collect_rollouts()
    _spy_train(one, 1, lambda k: k < 2, own_grad=True)
    one.close()
    h, mail = C.c_void_p(), C.c_void_p()
    _lib.check(lib.dronecu_ppo_create(C.byref(models[0].cfg), 0, C.byref(h)))
    try:
        _lib.check(lib.dronecu_ppo_dp_alloc(h, 0, 1, None, C.byref(mail)))
        _lib.check(lib.dronecu_ppo_dp_connect(h, 1, None, (C.c_void_p * 1)(mail.value)))
        buf, grad = torch.zeros(8, dtype=torch.float64, device="cuda"), torch.zeros(GRAD_LEN, device="cuda")
        grad[N + 4] = 1.0
        theta = torch.zeros(N, device="cuda")
        _lib.check(lib.dronecu_ppo_dp_allreduce_f64(h, P(buf), 8, None))
        _lib.check(lib.dronecu_ppo_apply_dp(h, P(theta), P(grad), None, None))
        torch.cuda.synchronize()
    finally:
        lib.dronecu_ppo_destroy(h)
    scratch = torch.empty(B, dtype=torch.int32, device="cuda")
    for m, s in zip(models, streams):
        if (B + bs - 1) // bs <= 64:
            _lib.check(lib.dronecu_minibatch_partition(m._h, B, bs, SEED + 1, 0, P(scratch), None))
        with torch.cuda.stream(s):                   # cached blocks of the rank's own stream for its clones
            blocks = [torch.empty(1 << 18, device="cuda") for _ in range(256)]
            del blocks
    torch.cuda.synchronize()


def _check_ppo_loop(world, name, models, recs, summed, steps, n_mb):
    n, K, bs, E, kw, env_kw, every = DP_CONFIGS[name]
    B = n * K
    m0 = models[0]
    mode, cfg, clip, vf, ent = m0.update_precision, m0.cfg, m0.cfg.clip_range, m0.cfg.vf_coef, m0.cfg.ent_coef
    for r, m in enumerate(models):
        assert len(recs[r]) == len(summed[r]) == steps and m.n_updates == steps, f"{name}: rank {r} steps"
    cat = lambda f: torch.cat([f(m.buf).reshape(B, -1).double().cpu() for m in models])  # noqa: E731
    obs, act = cat(lambda b: b.obs), cat(lambda b: b.actions)
    old_logp, adv, ret, value = (cat(lambda b, a=a: getattr(b, a)).reshape(-1) for a in ("logp", "adv", "ret", "value"))
    worst = {"grad": 0.0, "step": 0.0, "stats": 0.0}
    for e in range(E):
        perm = philox.minibatch_partition(B, bs, SEED + 1, e) if n_mb <= 64 else philox.minibatch_permutation(B, SEED + 1, e)
        for k in range(n_mb):
            step = e * n_mb + k
            rows = perm[k * bs:(k + 1) * bs]
            m = len(rows)
            what = f"{name} world {world} step {step} (m = {m} per rank)"
            rec = [recs[r][step] for r in range(world)]
            for r in range(world):
                assert rec[r]["m"] == m and rec[r]["first"] == 0 and np.array_equal(rec[r]["index"].cpu().numpy(), rows), \
                    f"{what}: rank {r} rows"
            idx = torch.cat([torch.from_numpy(rows.astype(np.int64)) + r * B for r in range(world)])
            a = adv[idx]
            if not m0.normalize_advantage:
                assert all(x["stats"] is None for x in rec)
            else:
                st = rec[0]["stats"].cpu().numpy()
                for r in range(1, world):
                    assert _same(rec[r]["stats"], st), f"{what}: rank {r} statistics row"
                want = [float(a.sum()), float((a * a).sum())]
                assert st[2] == world * m, f"{what}: count {st[2]}"
                scale = 1e-12 * float(a.abs().sum() + (a * a).sum())
                worst["stats"] = max(worst["stats"], float(np.abs(st[:2] - want).max()) / scale)
                np.testing.assert_allclose(st[:2], want, rtol=1e-12, atol=scale, err_msg=what)
            own = np.stack([x["own_grad"].cpu().numpy() for x in rec])
            S = _f32_rank_sum(own)
            for r in range(world):
                assert _same(summed[r][step], S), f"{what}: rank {r} summed gradient != rank-order float32 sum"
            if "grad" not in rec[0]:
                continue
            for r in range(1, world):
                for key in ("theta", "mom", "theta_after", "mom_after"):
                    assert _same(rec[r][key], rec[0][key]), f"{what}: rank {r} {key}"
                assert rec[r]["t"] == rec[0]["t"] and rec[r]["t_after"] == rec[0]["t_after"] == rec[0]["t"] + 1
            theta = rec[0]["theta"].double().cpu()
            if mode != "fp32":                            # the reduced-precision forward must not straddle a clip boundary
                from oracle import ppo_oracle as po
                mean, _, log_std = po.forward(theta, obs[idx])
                lr_ = po.log_prob(mean, log_std, act[idx]) - old_logp[idx]
                gap = torch.minimum((lr_ - math.log1p(-clip)).abs(), (lr_ - math.log1p(clip)).abs()).min()
                assert float(gap) > 0.02, f"{what}: a sample within {float(gap):.3g} of a clip boundary"
            an = _normalised(adv, idx, "stats") if m0.normalize_advantage else a
            ref, _ = _ref_grad(theta, (obs, act, old_logp, None, ret), idx, an, clip, vf, ent)
            got = rec[0]["grad"].double().cpu().numpy()
            assert _same(rec[0]["grad"], S)
            wg, report = _grad_error(got, ref, mode)
            assert wg <= 1.0, f"{what}: {report}"
            assert got[N + 4] == world * m
            worst["grad"] = max(worst["grad"], wg)
            sref = _torch_step(rec[0]["theta"], rec[0]["grad"][:N].double().cpu() * f32(1.0 / (world * m)), rec[0]["mom"],
                               rec[0]["t"], cfg)
            worst["step"] = max(worst["step"], _check_step(rec[0]["theta_after"], rec[0]["mom_after"], sref, cfg, what,
                                                           rec[0]["norm"]))
    for r, m in enumerate(models):
        assert _same(m.params, m0.params), f"{name}: rank {r} final parameters"
        a, b = m.logger_values, m0.logger_values
        assert a.keys() == b.keys() and all(a[k] == b[k] or (a[k] != a[k] and b[k] != b[k]) for k in a), \
            f"{name}: rank {r} logs {a} != {b}"
    # SB3 explained_variance(values, returns) over the union, float64 from the float32 buffers.  Each rank forms its moments
    # from float32 var_mean (a reduction tree of depth log2 B) and f32(var + mean^2): every variance is off by at most
    # (16 + log2 B) u E[x^2], and 1 - var_d / var_y by var_d / var_y times the two relative errors
    d = ret - value
    var_y, var_d = float(ret.var(unbiased=False)), float(d.var(unbiased=False))
    ev_ref = 1.0 - var_d / var_y
    ev = m0.logger_values["train/explained_variance"]
    c = (16 + math.log2(B)) * U
    ev_bound = var_d / var_y * c * (float((d * d).mean()) / var_d + float((ret * ret).mean()) / var_y)
    ev_ratio = abs(ev - ev_ref) / ev_bound
    assert ev_ratio <= 1.0, f"{name}: explained variance {ev} vs float64 {ev_ref} (bound {ev_bound:.3g})"
    return (f"{name} world {world}: {steps} steps; worst err/bound gradient {worst['grad']:.3g}, step {worst['step']:.3g}, "
            f"statistics {worst['stats']:.3g}, explained variance {ev_ratio:.3g} (|err| {abs(ev - ev_ref):.3g} at {ev_ref:.4g})")


def _ppo_loops(world):
    return "\n".join(_ppo_loop(world, name) for name in DP_CONFIGS)


@pytest.mark.parametrize("world", [2, 3, 4])
def test_peer_ppo_loop_is_teacher_forced_at_every_step(drl, world):
    # always in a child: a fresh process whose first streams are the ranks' own, with 32 hardware queues
    print(_run(world, _ppo_loops, in_process_max=0))
