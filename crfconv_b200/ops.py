"""Thin torch-tensor wrappers over the C-ABI layer kernels (include/crfconv_b200.h).  torch is used for device memory
and streams only; every arithmetic op below runs in libcrfconv_b200.so.  All activations are row-major [rows, C] fp32
CUDA tensors."""
from __future__ import annotations

import os

import torch

from . import _lib

# 0 = 3xTF32 (fp32-grade, default: matches the fp32 reference to ~1e-6), 1 = single-pass TF32, 2 = single-pass bf16 in the
# persistent kernels (single-pass TF32 elsewhere; DESIGN.md §5).  The Linear entry points refuse any other value.
PRECISION = int(os.environ.get("CRFCONV_PRECISION", "0"))
STAT_SLOTS = 64      # include/crfconv_b200.h: CRFCONV_STAT_SLOTS
GRAD_SLOTS = 32      # CRFCONV_GRAD_SLOTS


# Debug aid: the gather kernels trust their index tensors (a bad index is an out-of-bounds device read where the reference's
# torch.gather raises).  With CHECK_INDICES = True every forward entry point that takes indices checks their range first
# (one min/max reduction and a host sync per call — off by default; not usable under CUDA-graph capture).
CHECK_INDICES = False


def check_index(idx, limit, what):
    if not CHECK_INDICES or idx is None or idx.numel() == 0:
        return
    lo, hi = int(idx.min()), int(idx.max())
    if lo < 0 or hi >= limit:
        raise IndexError(f"crfconv_b200 {what}: index out of range [{lo}, {hi}] for {limit} rows")


COUNTERS = {"launches": 0}       # number of crfconv_b200 kernels launched (bench.py's gpu_launches)
_PROFILE = None                   # when a dict: name -> list of (start_event, end_event, algorithmic_bytes)


def _nbytes(*tensors):
    return sum(t.numel() * t.element_size() for t in tensors if t is not None)


class _call:
    """Counts kernel launches and, in profiling mode, brackets the C-ABI call with CUDA events on the launching stream."""

    def __init__(self, name, kernels, nbytes):
        self.name, self.kernels, self.nbytes = name, kernels, nbytes

    def __enter__(self):
        COUNTERS["launches"] += self.kernels
        if _PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if _PROFILE is not None:
            self.e1.record()
            _PROFILE.setdefault(self.name, []).append((self.e0, self.e1, self.nbytes))
        return False


def profile_calls(fn, repeats=3):
    """Runs fn() `repeats` times with per-call CUDA-event timing; returns {kernel-name: {ms, calls, bytes}} per fn() call."""
    global _PROFILE
    fn()
    torch.cuda.synchronize()
    _PROFILE = {}
    try:
        for _ in range(repeats):
            fn()
        torch.cuda.synchronize()
        out = {}
        for name, recs in _PROFILE.items():
            out[name] = {"ms": sum(a.elapsed_time(b) for a, b, _ in recs) / repeats, "calls": len(recs) / repeats,
                         "bytes": sum(n for _, _, n in recs) / repeats}
        return out
    finally:
        _PROFILE = None


def _p(t):
    return None if t is None else t.data_ptr()


def _chk(t, name, dtype=torch.float32):
    assert t.is_cuda and t.dtype == dtype and t.is_contiguous(), f"{name}: need contiguous CUDA {dtype} tensor"
    return t


def as2d(x):
    """[B,N,C] or [M,C] → contiguous fp32 [M,C] view/copy."""
    x = x.detach()
    if x.dtype != torch.float32:
        x = x.float()
    return x.reshape(-1, x.shape[-1]).contiguous()


# ---- per-step arena for scratch that is zero on entry and consumed inside the call that takes it -------------------------------------
# A PointConvResNet step needs ≈130 small zero-initialised buffers (BatchNorm Σ / Σ² slots, backward sums, weight-gradient partial
# slots): as separate torch.zeros they are 130 fill kernels per step (≈0.35 ms of launches in a 7 ms step).  The network's forward
# calls scratch_begin_step(): ONE memset re-zeroes what earlier steps dirtied, and zeros_scratch() hands out slices.  Invariant after
# begin_step: the whole arena is zero; during a step arena[off:] is zero.  Only for buffers that are dead when the call that took them returns (never for saved / returned tensors).
class _ZeroArena:
    CAP = 16 * 1024 * 1024          # floats (64 MB)

    def __init__(self, device):
        self.buf = torch.zeros(self.CAP, dtype=torch.float32, device=device)
        self.off = 0
        self.hw = 0                 # highest offset any step reached: a captured step replays its memset / its slices without telling Python


_ARENAS = {}


def _arena_key(device):
    device = torch.device(device)
    return device.index if device.index is not None else torch.cuda.current_device()


def scratch_begin_step(device):
    """Start of a step (the network's forward): re-zero the part of the arena the previous step used and rewind."""
    key = _arena_key(device)
    a = _ARENAS.get(key)
    if a is None:
        if torch.cuda.is_current_stream_capturing():
            return                                   # never allocate the arena inside a graph's private pool
        a = _ARENAS[key] = _ZeroArena(device)
    a.hw = max(a.hw, a.off)
    if a.hw:
        a.buf[:a.hw].zero_()                         # everything any earlier step (eager or a graph replay) may have dirtied
    a.off = 0


def zeros_scratch(numel, device):
    a = _ARENAS.get(_arena_key(device))
    n = (int(numel) + 63) & ~63                      # 256-byte granules
    if a is None or a.off + n > a.CAP:
        return torch.zeros(int(numel), dtype=torch.float32, device=device)
    v = a.buf[a.off:a.off + int(numel)]
    a.off += n
    return v


class BN:
    """Per-BatchNorm scratch: slotted f32 Σ/Σ² partial accumulators, fused affine (scale, shift), saved mean/invstd, backward k1/k2."""
    __slots__ = ("C", "stats", "scale", "shift", "mean", "invstd", "k1", "k2", "count", "training")

    def __init__(self, C, device, stats=None, alloc_stats=True):
        self.C = C
        if stats is None and alloc_stats:
            stats = zeros_scratch(STAT_SLOTS * 2 * C, device)   # zeroed; consumed by the finalize right after the producing GEMM
        self.stats = stats
        buf = torch.empty(6, C, dtype=torch.float32, device=device)
        self.scale, self.shift, self.mean, self.invstd, self.k1, self.k2 = buf.unbind(0)
        self.count = 0
        self.training = True


def linear_fwd(X1, W, *, scale1=None, shift1=None, slope1=1.0, idx1=None, rows_dst=0, rows_src=0, X2=None, bias=None,
               stats=None, M=None, out=None):
    L = _lib.lib()
    C1 = X1.shape[1]
    C2 = X2.shape[1] if X2 is not None else 0
    if M is None:
        M = idx1.numel() if idx1 is not None else X1.shape[0]
    Cout = W.shape[0]
    assert W.shape[1] == C1 + C2 and W.is_contiguous()
    Y = out if out is not None else torch.empty((M, Cout), dtype=torch.float32, device=X1.device)
    nb = M * (C1 + C2 + Cout) * 4 + (M * 8 if idx1 is not None else 0)
    with _call(f"linear_fwd[{C1 + C2}->{Cout}]", 1, nb):
        rc = _linear_fwd_call(L, X1, C1, scale1, shift1, slope1, idx1, rows_dst, rows_src, X2, C2, W, bias, Y, stats, M, Cout)
    _lib.check(rc, "linear_fwd")
    return Y


def _linear_fwd_call(L, X1, C1, scale1, shift1, slope1, idx1, rows_dst, rows_src, X2, C2, W, bias, Y, stats, M, Cout):
    return L.crfconv_linear_fwd(_p(X1), C1, _p(scale1), _p(shift1), float(slope1), _p(idx1), int(rows_dst), int(rows_src), _p(X2), C2,
                              _p(W), _p(bias), _p(Y), _p(stats), int(M), int(Cout), PRECISION, _lib.stream_ptr())


def grad_slots_reduce(scratch, dW_flat, n, stride):
    L = _lib.lib()
    COUNTERS["launches"] += 1
    _lib.check(L.crfconv_grad_slots_reduce(_p(scratch), _p(dW_flat), int(n), int(stride), _lib.stream_ptr()), "grad_slots_reduce")


class Flat:
    """One zero-filled allocation carved into views (a single memset instead of one fill kernel per small tensor)."""

    def __init__(self, numel, dtype, device, scratch=False):
        """scratch=True: every view dies inside the call that takes it (zeros_scratch arena)."""
        self.buf = zeros_scratch(numel, device) if (scratch and dtype == torch.float32) else torch.zeros(int(numel), dtype=dtype, device=device)
        self.off = 0

    def take(self, *shape):
        n = 1
        for d in shape:
            n *= int(d)
        v = self.buf[self.off:self.off + n].view(*shape)
        self.off += n
        return v


def bn_finalize_fwd(bn: BN, count, gamma, beta, eps, momentum, training, running_mean, running_var):
    L = _lib.lib()
    bn.count, bn.training = int(count), bool(training)
    COUNTERS["launches"] += 1
    rc = L.crfconv_bn_finalize_fwd(_p(bn.stats), int(count), _p(gamma), _p(beta), float(eps), float(momentum), int(bool(training)),
                                   _p(running_mean), _p(running_var), _p(bn.scale), _p(bn.shift), _p(bn.mean), _p(bn.invstd),
                                   bn.C, _lib.stream_ptr())
    _lib.check(rc, "bn_finalize_fwd")


def bn_act_fwd(H, bn: BN, slope, R=None, out=None):
    L = _lib.lib()
    Y = out if out is not None else torch.empty_like(H)
    with _call(f"bn_act_fwd[{H.shape[1]}]", 1, _nbytes(H, R, Y)):
        rc = L.crfconv_bn_act_fwd(_p(H), _p(bn.scale), _p(bn.shift), _p(R), float(slope), _p(Y), H.shape[0], H.shape[1], _lib.stream_ptr())
    _lib.check(rc, "bn_act_fwd")
    return Y


def bn_backward_prepare(dY, H, bn: BN, slope, dgamma, dbeta, act_ref=None, sums=None):
    """Reduces Σ dV and Σ dV·Ĥ, accumulates dγ / dβ and fills bn.k1 / bn.k2 for the on-the-fly dH transform.
    `sums` (optional) = zero-initialised f64 scratch of STAT_SLOTS·2·C entries."""
    L = _lib.lib()
    if sums is None:
        sums = zeros_scratch(STAT_SLOTS * 2 * bn.C, H.device)
    if bn.C <= 128 and bn.count == H.shape[0]:
        # one launch: the last CTA of the reduction folds the slots into k1 / k2 / dγ / dβ (two-level arrival tickets)
        counter = zeros_scratch(counter_ints(), H.device)
        with _call(f"bn_bwd_reduce[{bn.C}]", 1, _nbytes(dY, H, act_ref)):
            rc = L.crfconv_bn_bwd_reduce_fin(_p(dY), _p(H), _p(act_ref), _p(bn.scale), _p(bn.shift), _p(bn.mean), _p(bn.invstd), float(slope),
                                             _p(sums), H.shape[0], bn.C, _p(counter), _p(bn.k1), _p(bn.k2), _p(dgamma), _p(dbeta),
                                             _lib.stream_ptr())
        _lib.check(rc, "bn_bwd_reduce_fin")
    else:
        with _call(f"bn_bwd_reduce[{bn.C}]", 1, _nbytes(dY, H, act_ref)):
            rc = L.crfconv_bn_bwd_reduce(_p(dY), _p(H), _p(act_ref), _p(bn.scale), _p(bn.shift), _p(bn.mean), _p(bn.invstd), float(slope),
                                         _p(sums), H.shape[0], bn.C, _lib.stream_ptr())
        _lib.check(rc, "bn_bwd_reduce")
        COUNTERS["launches"] += 1
        rc = L.crfconv_bn_finalize_bwd(_p(sums), bn.count, _p(bn.k1), _p(bn.k2), _p(dgamma), _p(dbeta), bn.C, _lib.stream_ptr())
        _lib.check(rc, "bn_finalize_bwd")
    if not bn.training:      # eval-mode BN is a fixed affine map: dH = scale·dV
        bn.k1.zero_()
        bn.k2.zero_()


def linear_bwd(dY, H, bn, slope, X1, W, *, scale1=None, shift1=None, slope1=1.0, idx1=None, rows_dst=0, rows_src=0, X2=None,
               dX1=None, acc1=False, dX2=None, acc2=False, dW=None, dbias=None, act_ref=None, scratch=None, scratch_stride=0):
    """bn = BN (after bn_backward_prepare) or None for a plain Linear."""
    L = _lib.lib()
    C1 = X1.shape[1]
    C2 = X2.shape[1] if X2 is not None else 0
    M, Cout = dY.shape
    b = bn
    if dW is not None and Cout * (C1 + C2) > 1024 and scratch_stride == 0:
        scratch = None      # wide outputs: a CTA's adds are spread over >1024 addresses, direct atomics are cheaper than a reduce pass
    elif dW is not None and scratch is None:
        scratch = zeros_scratch(GRAD_SLOTS * Cout * (C1 + C2), dY.device)
    nb = _nbytes(dY, H if b else None, act_ref, X1 if dW is not None else None, X2 if dW is not None else None, dX1, dX2,
                 dX1 if acc1 else None, dX2 if acc2 else None)
    with _call(f"linear_bwd[{Cout}<-{C1 + C2}]" + ("" if dW is not None else ":dgrad") + ("" if (dX1 is not None or dX2 is not None) else ":wgrad"),
               0, nb):
        rc = _linear_bwd_call(L, dY, H, act_ref, b, slope, X1, C1, scale1, shift1, slope1, idx1, rows_dst, rows_src, X2, C2, W, dX1, acc1,
                              dX2, acc2, dW, dbias, scratch, scratch_stride, M, Cout)
    _lib.check(rc, "linear_bwd")
    COUNTERS["launches"] += L.crfconv_linear_bwd_launches()     # the input and weight gradient may share one kernel


def _linear_bwd_call(L, dY, H, act_ref, b, slope, X1, C1, scale1, shift1, slope1, idx1, rows_dst, rows_src, X2, C2, W, dX1, acc1, dX2, acc2,
                     dW, dbias, scratch, scratch_stride, M, Cout):
    return L.crfconv_linear_bwd(_p(dY), _p(H), _p(act_ref), _p(b.scale) if b else None, _p(b.shift) if b else None,
                              _p(b.mean) if b else None, _p(b.invstd) if b else None, _p(b.k1) if b else None,
                              _p(b.k2) if b else None, float(slope),
                              _p(X1), C1, _p(scale1), _p(shift1), float(slope1), _p(idx1), int(rows_dst), int(rows_src), _p(X2), C2,
                              _p(W), _p(dX1), int(acc1), _p(dX2), int(acc2), _p(dW), _p(dbias), _p(scratch), int(scratch_stride), int(M), int(Cout), PRECISION,
                              _lib.stream_ptr())


# ------------------------------------------------------------------------------------------ CRF mean-field
def crf_compat_fwd(c, out=None, scratch=None):
    """`out` / `scratch`: preallocated (Cm, Minv) and f64 scratch, for callers that launch on a side stream."""
    L = _lib.lib()
    F = c.shape[0]
    Cm, Minv = out if out is not None else (torch.empty_like(c), torch.empty_like(c))
    if scratch is None:
        scratch = torch.empty(3 * F * F, dtype=torch.float64, device=c.device)
    COUNTERS["launches"] += 1
    _lib.check(L.crfconv_crf_compat_fwd(_p(c), _p(Cm), _p(Minv), _p(scratch), F, _lib.stream_ptr()), "crf_compat_fwd")
    return Cm, Minv


def crf_compat_bwd(c, Minv, GC, GM, Gc, scratch=None):
    L = _lib.lib()
    F = c.shape[0]
    if scratch is None:
        scratch = torch.empty(3 * F * F, dtype=torch.float64, device=c.device)
    COUNTERS["launches"] += 1
    _lib.check(L.crfconv_crf_compat_bwd(_p(c), _p(Minv), _p(GC), _p(GM), _p(Gc), _p(scratch), F, _lib.stream_ptr()), "crf_compat_bwd")


def crf_upsample_fwd(Hu, bn: BN, up_idx, B, N, Nc):
    L = _lib.lib()
    check_index(up_idx, Nc, "crf_upsample_fwd")
    F = Hu.shape[1]
    z = torch.empty((B * N, F), dtype=torch.float32, device=Hu.device)
    with _call(f"crf_upsample_fwd[{F}]", 1, _nbytes(Hu, up_idx, z)):
        rc = L.crfconv_crf_upsample_fwd(_p(Hu), _p(bn.scale), _p(bn.shift), _p(up_idx), _p(z), B, N, Nc, F, _lib.stream_ptr())
    _lib.check(rc, "crf_upsample_fwd")
    return z


def crf_upsample_bwd(Gz, G0, up_idx, Gu, B, N, Nc):
    L = _lib.lib()
    with _call(f"crf_upsample_bwd[{Gz.shape[1]}]", 1, _nbytes(Gz, G0, up_idx, Gu)):
        rc = L.crfconv_crf_upsample_bwd(_p(Gz), _p(G0), _p(up_idx), _p(Gu), B, N, Nc, Gz.shape[1], _lib.stream_ptr())
    _lib.check(rc, "crf_upsample_bwd")


def crf_step_fwd(Hy, scale_y, z, xprev, nbr, Cm, Minv, B, N, K):
    L = _lib.lib()
    check_index(nbr, N, "crf_step_fwd")
    xout = torch.empty_like(z)
    with _call(f"crf_step_fwd[{z.shape[1]}]", 1, _nbytes(Hy, z, xprev, nbr, xout)):
        rc = L.crfconv_crf_step_fwd(_p(Hy), _p(scale_y), _p(z), _p(xprev), _p(nbr), _p(Cm), _p(Minv), _p(xout), B, N, K, z.shape[1],
                                    _lib.stream_ptr())
    _lib.check(rc, "crf_step_fwd")
    return xout


def crf_step_bwd(Hy, scale_y, z, xprev, nbr, Cm, Minv, g, Gz, gprev, Gy, m_out, v_out, h_out, gz_acc, B, N, K):
    L = _lib.lib()
    with _call(f"crf_step_bwd[{z.shape[1]}]", 1, _nbytes(Hy, z, xprev, nbr, g, Gz, Gz, gprev, Gy, m_out, v_out, h_out)):
        rc = L.crfconv_crf_step_bwd(_p(Hy), _p(scale_y), _p(z), _p(xprev), _p(nbr), _p(Cm), _p(Minv), _p(g), _p(Gz), _p(gprev), _p(Gy),
                                    _p(m_out), _p(v_out), _p(h_out), int(gz_acc), B, N, K, z.shape[1], _lib.stream_ptr())
    _lib.check(rc, "crf_step_bwd")


# ------------------------------------------------------------------------- point-conv gather / aggregation
def relpos(support, centres, idx):
    """support [B,Ns,3], centres [B,Nq,3], idx [B,Nq,K] → rel [B·Nq·K, 3]."""
    L = _lib.lib()
    B, Ns, _ = support.shape
    check_index(idx, Ns, "relpos")
    Nq, K = idx.shape[1], idx.shape[2]
    rel = torch.empty((B * Nq * K, 3), dtype=torch.float32, device=support.device)
    with _call("relpos", 1, _nbytes(support, centres, idx, rel)):
        rc = L.crfconv_relpos(_p(support), _p(centres), _p(idx), _p(rel), B, Ns, Nq, K, _lib.stream_ptr())
    _lib.check(rc, "relpos")
    return rel


def pointconv_aggregate_fwd(x, H2, bn: BN, idx, B, Ns, Nq, K):
    L = _lib.lib()
    check_index(idx, Ns, "pointconv_aggregate_fwd")
    C = x.shape[1]
    out = torch.empty((B * Nq, C), dtype=torch.float32, device=x.device)
    with _call(f"pointconv_aggregate_fwd[{C}]", 1, _nbytes(x, H2, idx, out)):
        rc = L.crfconv_pointconv_aggregate_fwd(_p(x), _p(H2), _p(bn.scale), _p(bn.shift), _p(idx), _p(out), B, Ns, Nq, K, C, _lib.stream_ptr())
    _lib.check(rc, "pointconv_aggregate_fwd")
    return out


def pointconv_aggregate_bwd(x, H2, bn: BN, idx, g, dx, B, Ns, Nq, K):
    L = _lib.lib()
    C = x.shape[1]
    dWgt = torch.empty_like(H2)
    with _call(f"pointconv_aggregate_bwd[{C}]", 1, _nbytes(x, H2, idx, g, dWgt, dx)):
        rc = L.crfconv_pointconv_aggregate_bwd(_p(x), _p(H2), _p(bn.scale), _p(bn.shift), _p(idx), _p(g), _p(dWgt), _p(dx), B, Ns, Nq, K, C,
                                               _lib.stream_ptr())
    _lib.check(rc, "pointconv_aggregate_bwd")
    return dWgt


# ---- PointConv without per-edge tensors (csrc/pointconv_fused.cu, hidden width 8) ------------------------------------------------
def pcf_supported(d):
    return bool(_lib.lib().crfconv_pcf_supported(int(d)))


def pcf_scratch_floats(d):
    L = _lib.lib()
    return L.crfconv_pcf_fwd_scratch_floats(int(d)), L.crfconv_pcf_bwd_scratch_floats(int(d))


def pcf_relpos_moments(support, centres, idx, mom):
    L = _lib.lib()
    B, Ns, _ = support.shape
    check_index(idx, Ns, "pcf_relpos_moments")
    Nq, K = idx.shape[1], idx.shape[2]
    rel = torch.empty((B * Nq * K, 3), dtype=torch.float32, device=support.device)
    with _call("pcf_relpos_moments", 1, _nbytes(support, centres, idx, rel)):
        rc = L.crfconv_pcf_relpos_moments(_p(support), _p(centres), _p(idx), _p(rel), _p(mom), B, Ns, Nq, K, _lib.stream_ptr())
    _lib.check(rc, "pcf_relpos_moments")
    return rel


def pcf_stats1(mom, W1, stats1):
    L = _lib.lib()
    COUNTERS["launches"] += 1
    _lib.check(L.crfconv_pcf_stats1(_p(mom), _p(W1), _p(stats1), int(W1.shape[0]), _lib.stream_ptr()), "pcf_stats1")


def pcf_fwd(x, rel, idx, W1, W2, bn1: BN, slope1, stats2, asum, B, Ns, Nq, K):
    L = _lib.lib()
    d = x.shape[1]
    P = torch.empty((B * Nq, d), dtype=torch.float32, device=x.device)
    Q = torch.empty((B * Nq, d), dtype=torch.float32, device=x.device)
    with _call("pcf_fwd", 1, _nbytes(x, rel, idx, P, Q)):
        rc = L.crfconv_pcf_fwd(_p(x), _p(rel), _p(idx), _p(W1), _p(W2), _p(bn1.scale), _p(bn1.shift), float(slope1), _p(P), _p(Q), _p(stats2),
                               _p(asum), B, Ns, Nq, K, d, _lib.stream_ptr())
    _lib.check(rc, "pcf_fwd")
    return P, Q


def pcf_out(P, Q, bn2: BN):
    L = _lib.lib()
    out = torch.empty_like(P)
    with _call("pcf_out", 1, _nbytes(P, Q, out)):
        rc = L.crfconv_pcf_out(_p(P), _p(Q), _p(bn2.scale), _p(bn2.shift), _p(out), P.shape[0], P.shape[1], _lib.stream_ptr())
    _lib.check(rc, "pcf_out")
    return out


def pcf_bwd1(x, rel, idx, g, W1, W2, bn1: BN, slope1, bn2: BN, dx, sums2, mdw, B, Ns, Nq, K):
    L = _lib.lib()
    with _call("pcf_bwd1", 1, _nbytes(x, rel, idx, g, dx, dx)):
        rc = L.crfconv_pcf_bwd1(_p(x), _p(rel), _p(idx), _p(g), _p(W1), _p(W2), _p(bn1.scale), _p(bn1.shift), float(slope1), _p(bn2.scale),
                                _p(bn2.shift), _p(bn2.mean), _p(bn2.invstd), _p(dx), _p(sums2), _p(mdw), B, Ns, Nq, K, x.shape[1], _lib.stream_ptr())
    _lib.check(rc, "pcf_bwd1")


def pcf_bwd2(x, rel, idx, g, W1, W2, bn1: BN, slope1, bn2: BN, sums1, s1, B, Ns, Nq, K):
    L = _lib.lib()
    with _call("pcf_bwd2", 1, _nbytes(x, rel, idx, g)):
        rc = L.crfconv_pcf_bwd2(_p(x), _p(rel), _p(idx), _p(g), _p(W1), _p(W2), _p(bn1.scale), _p(bn1.shift), float(slope1), _p(bn1.mean),
                                _p(bn1.invstd), _p(bn2.scale), _p(bn2.mean), _p(bn2.invstd), _p(bn2.k1), _p(bn2.k2), _p(sums1), _p(s1),
                                B, Ns, Nq, K, x.shape[1], _lib.stream_ptr())
    _lib.check(rc, "pcf_bwd2")


def bn_finalize_bwd(sums, bn: BN, dgamma, dbeta):
    """k1 / k2 of `bn` from slotted sums Σ dV | Σ dV·Ĥ; dγ += Σ dV·Ĥ, dβ += Σ dV."""
    L = _lib.lib()
    COUNTERS["launches"] += 1
    _lib.check(L.crfconv_bn_finalize_bwd(_p(sums), bn.count, _p(bn.k1), _p(bn.k2), _p(dgamma), _p(dbeta), bn.C, _lib.stream_ptr()), "bn_finalize_bwd")


def pcf_param_grads(mom, asum, mdw, s1, W1, W2, bn1: BN, bn2: BN, dW1, dW2):
    L = _lib.lib()
    COUNTERS["launches"] += 1
    rc = L.crfconv_pcf_param_grads(_p(mom), _p(asum), _p(mdw), _p(s1), _p(W1), _p(W2), _p(bn1.scale), _p(bn1.mean), _p(bn1.invstd), _p(bn1.k1),
                                   _p(bn1.k2), _p(bn2.scale), _p(bn2.mean), _p(bn2.invstd), _p(bn2.k1), _p(bn2.k2), _p(dW1), _p(dW2),
                                   int(W2.shape[0]), _lib.stream_ptr())
    _lib.check(rc, "pcf_param_grads")


def gather_max_fwd(x, idx, B, Ns, Nq, K):
    L = _lib.lib()
    check_index(idx, Ns, "gather_max_fwd")
    C = x.shape[1]
    out = torch.empty((B * Nq, C), dtype=torch.float32, device=x.device)
    arg = torch.empty((B * Nq, C), dtype=torch.int32, device=x.device)
    with _call(f"gather_max_fwd[{C}]", 1, _nbytes(x, idx, out, arg)):
        rc = L.crfconv_gather_max_fwd(_p(x), _p(idx), _p(out), _p(arg), B, Ns, Nq, K, C, _lib.stream_ptr())
    _lib.check(rc, "gather_max_fwd")
    return out, arg


def gather_max_bwd(g, arg, dx):
    L = _lib.lib()
    with _call(f"gather_max_bwd[{g.shape[1]}]", 1, _nbytes(g, arg, dx)):
        rc = L.crfconv_gather_max_bwd(_p(g), _p(arg), _p(dx), g.shape[0], g.shape[1], _lib.stream_ptr())
    _lib.check(rc, "gather_max_bwd")


def lrelu_bwd(g, out, slope):
    L = _lib.lib()
    dS = torch.empty_like(out)
    with _call("lrelu_bwd", 1, _nbytes(g, out, dS)):
        rc = L.crfconv_lrelu_bwd(_p(g), _p(out), float(slope), _p(dS), out.numel(), _lib.stream_ptr())
    _lib.check(rc, "lrelu_bwd")
    return dS


def add_inplace(y, x):
    L = _lib.lib()
    with _call("add_inplace", 1, _nbytes(y, y, x)):
        rc = L.crfconv_add_inplace(_p(y), _p(x), y.numel(), _lib.stream_ptr())
    _lib.check(rc, "add_inplace")


def scatter_add_rows(src, idx, dst, B, Nq, Ns):
    L = _lib.lib()
    with _call(f"scatter_add_rows[{src.shape[1]}]", 1, _nbytes(src, idx, dst)):
        rc = L.crfconv_scatter_add_rows(_p(src), _p(idx), _p(dst), B, Nq, Ns, src.shape[1], _lib.stream_ptr())
    _lib.check(rc, "scatter_add_rows")


# --------------------------------------------------------------------- layer-specialised (fused) CRF kernels, F = 16
def fused_max_parts():
    return int(_lib.lib().crfconv_fused_max_parts())


def fused_part_floats():
    return int(_lib.lib().crfconv_fused_part_floats())


def counter_ints():
    """uint32 per `counter` argument of the fused kernels (two-level arrival tickets); zeroed by the caller, left zero."""
    return int(_lib.lib().crfconv_fused_counter_ints())


def out_bwd_part_floats():
    return int(_lib.lib().crfconv_out_bwd_part_floats())


def _bn_fin_args(bn_module):
    """(gamma, beta, running_mean, running_var, eps, momentum) of an nn.BatchNorm1d in training mode."""
    if bn_module.momentum is None:
        raise RuntimeError("crfconv_b200: BatchNorm momentum=None (cumulative average) is not supported by the fused kernels")
    track = bn_module.track_running_stats and bn_module.running_mean is not None
    return (_p(bn_module.weight), _p(bn_module.bias), _p(bn_module.running_mean) if track else None,
            _p(bn_module.running_var) if track else None, float(bn_module.eps), float(bn_module.momentum))


def lin16_fwd(X, W, bn: BN, bn_module, part, counter, pre: BN = None, pslope=1.0, out=None):
    """H = act(X)·Wᵀ (16 output channels) with `bn`'s scale/shift/mean/invstd (and the module's running statistics) finalized by
    the same launch.  pre: BN state whose affine + LeakyReLU(pslope) is applied to X on the fly (X has 16 channels then)."""
    L = _lib.lib()
    M, Cin = X.shape
    Y = out if out is not None else torch.empty((M, 16), dtype=torch.float32, device=X.device)
    gm, bt, rm, rv, eps, mom = _bn_fin_args(bn_module)
    bn.count, bn.training = int(M), True
    with _call(f"lin16_fwd[{Cin}]", 1, _nbytes(X, Y)):
        rc = L.crfconv_lin16_fwd(_p(X), int(Cin), _p(W), _p(pre.scale) if pre else None, _p(pre.shift) if pre else None, float(pslope),
                                 _p(Y), int(M), _p(part), _p(counter), gm, bt, rm, rv, eps, mom, _p(bn.scale), _p(bn.shift), _p(bn.mean),
                                 _p(bn.invstd), _lib.stream_ptr())
    _lib.check(rc, "lin16_fwd")
    return Y


def up16_fwd(X, W, bn: BN, bn_module, counter, out=None):
    """H[M,Cout] = X[M,16]·Wᵀ (Cout = 64) with `bn` finalized by the same launch; bn.stats zeroed."""
    L = _lib.lib()
    M, Cout = X.shape[0], W.shape[0]
    Y = out if out is not None else torch.empty((M, Cout), dtype=torch.float32, device=X.device)
    gm, bt, rm, rv, eps, mom = _bn_fin_args(bn_module)
    bn.count, bn.training = int(M), True
    with _call(f"up16_fwd[{Cout}]", 1, _nbytes(X, Y)):
        rc = L.crfconv_up16_fwd(_p(X), _p(W), int(Cout), _p(Y), int(M), _p(bn.stats), _p(counter), gm, bt, rm, rv, eps, mom, _p(bn.scale),
                                _p(bn.shift), _p(bn.mean), _p(bn.invstd), _lib.stream_ptr())
    _lib.check(rc, "up16_fwd")
    return Y


def linear_fwd_bn(X1, W, bn: BN, bn_module, counter, *, scale1=None, shift1=None, slope1=1.0, X2=None, out=None):
    """linear_fwd + BatchNorm finalize of the output in one launch (tcgen05 kernel) or two (other shapes).  bn.stats zeroed."""
    L = _lib.lib()
    M, C1 = X1.shape
    C2 = X2.shape[1] if X2 is not None else 0
    Cout = W.shape[0]
    Y = out if out is not None else torch.empty((M, Cout), dtype=torch.float32, device=X1.device)
    gm, bt, rm, rv, eps, mom = _bn_fin_args(bn_module)
    bn.count, bn.training = int(M), True
    with _call(f"linear_fwd_bn[{C1 + C2}->{Cout}]", 1, M * (C1 + C2 + Cout) * 4):
        rc = L.crfconv_linear_fwd_bn(_p(X1), int(C1), _p(scale1), _p(shift1), float(slope1), _p(X2), int(C2), _p(W), _p(Y), _p(bn.stats),
                                     int(M), int(Cout), PRECISION, _p(counter), gm, bt, rm, rv, eps, mom, _p(bn.scale), _p(bn.shift),
                                     _p(bn.mean), _p(bn.invstd), _lib.stream_ptr())
    _lib.check(rc, "linear_fwd_bn")
    return Y


def bn_backward_prepare_fin(dY, H, bn: BN, slope, dgamma, dbeta, sums, counter):
    """bn_backward_prepare in one launch (C = 64) or two."""
    L = _lib.lib()
    with _call(f"bn_bwd_reduce_fin[{bn.C}]", 1, _nbytes(dY, H)):
        rc = L.crfconv_bn_bwd_reduce_fin(_p(dY), _p(H), None, _p(bn.scale), _p(bn.shift), _p(bn.mean), _p(bn.invstd), float(slope),
                                         _p(sums), H.shape[0], bn.C, _p(counter), _p(bn.k1), _p(bn.k2), _p(dgamma), _p(dbeta),
                                         _lib.stream_ptr())
    _lib.check(rc, "bn_bwd_reduce_fin")


def mid16_bwd(dY, H2, bn2: BN, H1, bn1: BN, slope1, W2, dW2_slots, slot_stride, part, counter, dgamma1, dbeta1, out=None):
    L = _lib.lib()
    dV1 = out if out is not None else torch.empty_like(H1)
    with _call("mid16_bwd", 1, _nbytes(dY, H2, H1, dV1)):
        rc = L.crfconv_mid16_bwd(_p(dY), _p(H2), _p(bn2.scale), _p(bn2.mean), _p(bn2.invstd), _p(bn2.k1), _p(bn2.k2), _p(H1), _p(bn1.scale),
                                 _p(bn1.shift), _p(bn1.mean), _p(bn1.invstd), float(slope1), _p(W2), _p(dV1), _p(dW2_slots), int(slot_stride),
                                 H1.shape[0], _p(part), _p(counter), _p(bn1.k1), _p(bn1.k2), _p(dgamma1), _p(dbeta1), _lib.stream_ptr())
    _lib.check(rc, "mid16_bwd")
    return dV1


def in16_dgrad(dV1, H1, bn1: BN, W1, dX, accumulate):
    L = _lib.lib()
    Cin = W1.shape[1]
    with _call(f"in16_dgrad[{Cin}]", 1, _nbytes(dV1, H1, dX, dX if accumulate else None)):
        rc = L.crfconv_in16_dgrad(_p(dV1), _p(H1), _p(bn1.scale), _p(bn1.mean), _p(bn1.invstd), _p(bn1.k1), _p(bn1.k2), _p(W1), int(Cin),
                                  _p(dX), int(bool(accumulate)), H1.shape[0], _lib.stream_ptr())
    _lib.check(rc, "in16_dgrad")


def in16_wgrad(dV1, H1, bn1: BN, X, dW_slots, slot_stride):
    L = _lib.lib()
    Cin = X.shape[1]
    with _call(f"in16_wgrad[{Cin}]", 1, _nbytes(dV1, H1, X)):
        rc = L.crfconv_in16_wgrad(_p(dV1), _p(H1), _p(bn1.scale), _p(bn1.mean), _p(bn1.invstd), _p(bn1.k1), _p(bn1.k2), _p(X), int(Cin),
                                  _p(dW_slots), int(slot_stride), H1.shape[0], _lib.stream_ptr())
    _lib.check(rc, "in16_wgrad")


def out16_bwd(dO, H3, bn3: BN, slope3, X, W3, part, counter, dgamma, dbeta, dW3, Q, a0, out=None):
    L = _lib.lib()
    T = out if out is not None else torch.empty_like(X)
    with _call("out16_bwd", 1, _nbytes(dO, H3, X, T)):
        rc = L.crfconv_out16_bwd(_p(dO), _p(H3), _p(bn3.scale), _p(bn3.shift), _p(bn3.mean), _p(bn3.invstd), float(slope3), _p(X), _p(W3),
                                 _p(T), X.shape[0], _p(part), _p(counter), _p(bn3.k1), _p(bn3.k2), _p(dgamma), _p(dbeta), _p(dW3), _p(Q),
                                 _p(a0), _lib.stream_ptr())
    _lib.check(rc, "out16_bwd")
    return T


def crf_step_bwd_fused(Hy, bn_y: BN, z, xprev, nbr, Cm, Minv, g, xT, Q, a0, Gz, gz_acc, gprev, Gy, GC_slots, GM_slots, slot_stride, ysum,
                       B, N, K, finalize, counter, gamma_y, dgamma, dbeta):
    L = _lib.lib()
    with _call("crf_step_bwd_fused", 1, _nbytes(Hy, z, xprev, nbr, g, xT, Gz, gprev, Gy)):
        rc = L.crfconv_crf_step_bwd_fused(_p(Hy), _p(bn_y.scale), _p(z), _p(xprev), _p(nbr), _p(Cm), _p(Minv), _p(g), _p(xT), _p(Q), _p(a0),
                                          _p(Gz), int(gz_acc), _p(gprev), _p(Gy), _p(GC_slots), _p(GM_slots), int(slot_stride), _p(ysum),
                                          B, N, K, Gz.shape[1], int(bool(finalize)), _p(counter), _p(gamma_y), _p(bn_y.k1), _p(bn_y.k2),
                                          _p(dgamma), _p(dbeta), _lib.stream_ptr())
    _lib.check(rc, "crf_step_bwd_fused")


def crf_upsample_bwd_fused(Gz, G0, up_idx, Hu, bn_u: BN, Gu, B, N, Nc, part, counter, dgamma, dbeta):
    L = _lib.lib()
    with _call("crf_upsample_bwd_fused", 1, _nbytes(Gz, G0, up_idx, Gu)):
        rc = L.crfconv_crf_upsample_bwd_fused(_p(Gz), _p(G0), _p(up_idx), _p(Hu), _p(bn_u.mean), _p(bn_u.invstd), _p(Gu), B, N, Nc, _p(part),
                                              _p(counter), _p(bn_u.k1), _p(bn_u.k2), _p(dgamma), _p(dbeta), _lib.stream_ptr())
    _lib.check(rc, "crf_upsample_bwd_fused")
