"""Drop-in for the reference's ``models/continuous_crf_conv_big.py`` (:7-78): ``ContinuousGaussianCRFConv`` with the same
constructor, forward signature, sub-module names and ``state_dict`` keys (``unary_nn.{0,1}.*``, ``pairwise_nn.{0,1}.*``,
``out_nn.*``, ``fusion_nn.*``, ``c``), executed as ONE autograd node that drives the sm_100a kernels:

    unary_nn / pairwise_nn : tensor-core Linear passes with BN statistics in the epilogue and BN+LeakyReLU on the fly
    z = u[up_idx]          : fused with unary_nn's last BatchNorm                                      (:60)
    mean-field steps       : csrc/crf.cu — distances, softmax over k, aggregation, C / (I+C)^-1 in registers   (:68-72)
    out_nn, fusion_nn      : the concat [x, pairwise] (:76) is never materialised (two-segment GEMM)

Unlike the reference it accepts B = 1 (the reference crashes there: ``.squeeze()`` at :43), and ``(I+C)^-1`` is computed
once per forward instead of once per step.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .common import MLP, bn_forward_state


USE_FUSED = True      # tests flip this to compare the layer-specialised kernels with the generic ones

_SIDE = {}


def _side_stream(dev):
    """Second stream per device: the unary and pairwise MLP chains are independent until the upsample, and at hidden width
    each of their kernels is latency-bound (≈300 persistent CTAs, little work each), so the two chains run concurrently
    (forward and backward).  Captured CUDA graphs keep the fork/join as parallel branches."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=dev)
    return _SIDE[key]


_AUX = {}


def _aux_stream(dev):
    """Third stream: the F×F compatibility algebra (C = cᵀc, (I+C)⁻¹ and its backward) is a single-CTA kernel of 10-16 us that
    depends on nothing but `c` (forward) / GC, GM (backward); on its own graph branch it costs nothing."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _AUX:
        _AUX[key] = torch.cuda.Stream(device=dev)
    return _AUX[key]


def _param_grads(gbuf, grads):
    """Parameter gradients of a CRF layer: returned to autograd, or — when the parameters opted into direct accumulation
    (common.direct_grad_buffers) — added into the bound .grad views with ONE multi-tensor kernel (instead of one AccumulateGrad add
    per parameter) and reported as None."""
    if gbuf is None:
        return grads
    torch._foreach_add_(list(gbuf), [g.view_as(b) for g, b in zip(grads, gbuf)])
    return [None] * len(grads)


def _mlp_params(m: MLP):
    return m.lin.weight, m.bn.batch_norm.weight, m.bn.batch_norm.bias


class _CRFConvFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, unary, pairwise, up_idx, neighbor_idx, steps, training, mods, gbuf, c, *params):
        if not (unary.is_cuda and pairwise.is_cuda):
            raise RuntimeError("crfconv_b200 layers run on CUDA tensors only (no CPU fallback)")
        ctx.gbuf = gbuf
        (W1u, _, _, W2u, _, _, W1p, _, _, W2p, _, _, Wo, _, _, Wf, _, _) = [p.detach().contiguous().float() for p in params]
        bns = [m.bn.batch_norm for m in mods]          # order: u0, u1, p0, p1, out, fusion
        sl = [m.slope for m in mods]                   # LeakyReLU slopes (1.0 = no activation), reference: .1, 1, .1, 1, .1, .1
        if any(v is None for v in sl) or sl[1] != 1.0 or sl[3] != 1.0:
            raise RuntimeError("ContinuousGaussianCRFConv: only LeakyReLU/ReLU/None activations in the reference positions are fused")
        B, Nc, Cu = unary.shape
        _, N, Cp = pairwise.shape
        K = neighbor_idx.shape[-1]
        dev = unary.device
        U, P = ops.as2d(unary), ops.as2d(pairwise)
        up = up_idx.detach().reshape(B, N).contiguous().to(torch.int64)
        nbr = neighbor_idx.detach().contiguous().to(torch.int64)
        Mc, M = B * Nc, B * N
        F, Co = W2u.shape[0], Wf.shape[0]

        def tr(bn):
            return training or not bn.track_running_stats

        fstats = ops.Flat(ops.STAT_SLOTS * 2 * (4 * F + 2 * Co), torch.float32, dev, scratch=True)
        nbt = []

        # unary_nn / pairwise_nn, layer 1 and 2 (:58-59) — two independent chains on two streams; every buffer is allocated on the
        # main stream first, the side stream only launches kernels
        s1u, fin1u = bn_forward_state(F, dev, Mc, bns[0], tr(bns[0]), fstats.take(ops.STAT_SLOTS * 2 * F), nbt)
        s2u, fin2u = bn_forward_state(F, dev, Mc, bns[1], tr(bns[1]), fstats.take(ops.STAT_SLOTS * 2 * F), nbt)
        s1p, fin1p = bn_forward_state(F, dev, M, bns[2], tr(bns[2]), fstats.take(ops.STAT_SLOTS * 2 * F), nbt)
        s2p, fin2p = bn_forward_state(F, dev, M, bns[3], tr(bns[3]), fstats.take(ops.STAT_SLOTS * 2 * F), nbt)
        H1u, H2u = torch.empty((Mc, F), dtype=torch.float32, device=dev), torch.empty((Mc, F), dtype=torch.float32, device=dev)
        main, side, aux = torch.cuda.current_stream(dev), _side_stream(dev), _aux_stream(dev)
        fork, join, join_aux = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
        cc = c.detach().contiguous().float()
        Cm, Minv = torch.empty_like(cc), torch.empty_like(cc)
        cscr = torch.empty(3 * F * F, dtype=torch.float64, device=dev)
        fork.record(main)
        side.wait_event(fork)
        aux.wait_event(fork)
        with torch.cuda.stream(aux):
            ops.crf_compat_fwd(cc, out=(Cm, Minv), scratch=cscr)
            join_aux.record(aux)
        with torch.cuda.stream(side):
            ops.linear_fwd(U, W1u, stats=s1u.stats, out=H1u); fin1u()
            ops.linear_fwd(H1u, W2u, scale1=s1u.scale, shift1=s1u.shift, slope1=sl[0], stats=s2u.stats, out=H2u); fin2u()
            join.record(side)
        H1p = ops.linear_fwd(P, W1p, stats=s1p.stats); fin1p()
        H2p = ops.linear_fwd(H1p, W2p, scale1=s1p.scale, shift1=s1p.shift, slope1=sl[2], stats=s2p.stats); fin2p()
        # mean field (:60-72)
        main.wait_event(join)
        main.wait_event(join_aux)
        z = ops.crf_upsample_fwd(H2u, s2u, up, B, N, Nc)
        xs = [z]
        for _ in range(steps):
            xs.append(ops.crf_step_fwd(H2p, s2p.scale, z, xs[-1], nbr, Cm, Minv, B, N, K))
        # out_nn, fusion_nn (:74-76)
        so, fin = bn_forward_state(Co, dev, M, bns[4], tr(bns[4]), fstats.take(ops.STAT_SLOTS * 2 * Co), nbt)
        H3 = ops.linear_fwd(xs[-1], Wo, stats=so.stats); fin()
        sf, fin = bn_forward_state(Co, dev, M, bns[5], tr(bns[5]), fstats.take(ops.STAT_SLOTS * 2 * Co), nbt)
        Hf = ops.linear_fwd(H3, Wf, scale1=so.scale, shift1=so.shift, slope1=sl[4], X2=P, stats=sf.stats); fin()
        out = ops.bn_act_fwd(Hf, sf, sl[5])
        if nbt:
            torch._foreach_add_(nbt, 1)                  # six num_batches_tracked counters, one launch

        ctx.dims = (B, N, Nc, K, F, Co, Cu, Cp, steps)
        ctx.bn = (s1u, s2u, s1p, s2p, so, sf)
        ctx.sl = sl
        ctx.save_for_backward(U, P, up, nbr, H1u, H2u, H1p, H2p, H3, Hf, Cm, Minv, cc, W1u, W2u, W1p, W2p, Wo, Wf, *xs)
        return out.view(B, N, Co)

    @staticmethod
    def backward(ctx, gout):
        (U, P, up, nbr, H1u, H2u, H1p, H2p, H3, Hf, Cm, Minv, cc, W1u, W2u, W1p, W2p, Wo, Wf, *xs) = ctx.saved_tensors
        B, N, Nc, K, F, Co, Cu, Cp, steps = ctx.dims
        s1u, s2u, s1p, s2p, so, sf = ctx.bn
        sl = ctx.sl
        dev = gout.device
        Mc, M = B * Nc, B * N
        z = xs[0]
        g2 = ops.as2d(gout)

        wl = (("1u", W1u), ("2u", W2u), ("1p", W1p), ("2p", W2p), ("o", Wo), ("f", Wf))
        cl = (("1u", F), ("2u", F), ("1p", F), ("2p", F), ("o", Co), ("f", Co))
        n_small = sum(w.numel() for _, w in wl) + 2 * sum(n for _, n in cl) + 3 * F * F
        n_sums = ops.STAT_SLOTS * 2 * sum(n for _, n in cl)
        n_big = (steps + 1) * M * F + Mc * F
        # ONE zero-filled allocation: [small grads | weight-grad partial slots | BN-backward Σ slots | scatter targets]
        flat = ops.Flat(n_small * (1 + ops.GRAD_SLOTS) + n_sums + n_big, torch.float32, dev)
        small = flat.take(n_small)
        wscr = flat.take(ops.GRAD_SLOTS * n_small)          # slot pitch n_small: same layout as `small`, folded by one reduce at the end
        sums = ops.Flat.__new__(ops.Flat); sums.buf, sums.off = flat.take(n_sums), 0
        big = ops.Flat.__new__(ops.Flat); big.buf, big.off = flat.take(n_big), 0
        cursor = [0]

        def take_small(*shape):
            n = 1
            for d in shape:
                n *= int(d)
            v = small[cursor[0]:cursor[0] + n].view(*shape)
            cursor[0] += n
            return v

        def scr(t):                                          # partial-slot region that mirrors the small-gradient view `t`
            return wscr[(t.data_ptr() - small.data_ptr()) // 4:]

        zeros = take_small
        GC, GM = take_small(F, F), take_small(F, F)         # first in the layout: folded on their own before the c-gradient algebra
        dW = {k: take_small(*w.shape) for k, w in wl}
        dg = {k: take_small(n) for k, n in cl}
        db = {k: take_small(n) for k, n in cl}
        # fusion_nn
        ops.bn_backward_prepare(g2, Hf, sf, sl[5], dg["f"], db["f"], sums=sums.take(ops.STAT_SLOTS * 2 * Co))
        dO = torch.empty((M, Co), dtype=torch.float32, device=dev)
        dP = torch.empty((M, Cp), dtype=torch.float32, device=dev)
        ops.linear_bwd(g2, Hf, sf, sl[5], H3, Wf, scale1=so.scale, shift1=so.shift, slope1=sl[4], X2=P, dX1=dO, dX2=dP, dW=dW["f"], scratch=scr(dW["f"]), scratch_stride=n_small)
        # out_nn
        ops.bn_backward_prepare(dO, H3, so, sl[4], dg["o"], db["o"], sums=sums.take(ops.STAT_SLOTS * 2 * Co))
        g = torch.empty((M, F), dtype=torch.float32, device=dev)
        ops.linear_bwd(dO, H3, so, sl[4], xs[-1], Wo, dX1=g, dW=dW["o"], scratch=scr(dW["o"]), scratch_stride=n_small)
        # mean-field steps, last to first
        Gy = big.take(M, F)
        Gz, m_out, v_out, h_out = (torch.empty((M, F), dtype=torch.float32, device=dev) for _ in range(4))
        for t in range(steps, 0, -1):
            gprev = big.take(M, F)
            ops.crf_step_bwd(H2p, s2p.scale, z, xs[t - 1], nbr, Cm, Minv, g, Gz, gprev, Gy, m_out, v_out, h_out, t != steps, B, N, K)
            ops.linear_bwd(m_out, None, None, 1.0, h_out, GC, dW=GC, scratch=scr(GC), scratch_stride=n_small)      # GC += mᵀ·h
            ops.linear_bwd(v_out, None, None, 1.0, g, GM, dW=GM, scratch=scr(GM), scratch_stride=n_small)          # GM += vᵀ·g
            g = gprev
        ops.grad_slots_reduce(wscr, small, 2 * F * F, n_small)    # fold the GC / GM partial slots
        Gc = zeros(F, F)
        aux = _aux_stream(dev)
        fork_aux, join_aux = torch.cuda.Event(), torch.cuda.Event()
        bscr = torch.empty(3 * F * F, dtype=torch.float64, device=dev)
        fork_aux.record(torch.cuda.current_stream(dev))
        aux.wait_event(fork_aux)
        with torch.cuda.stream(aux):                             # off the critical path: Gc is only needed when backward returns
            ops.crf_compat_bwd(cc, Minv, GC, GM, Gc, scratch=bscr)
            join_aux.record(aux)
        Gu = big.take(Mc, F)
        if steps > 0:
            ops.crf_upsample_bwd(Gz, g, up, Gu, B, N, Nc)      # dL/dz = Σ_t h^t + g^0
        else:
            ops.crf_upsample_bwd(g, None, up, Gu, B, N, Nc)
        # unary_nn — on the side stream, concurrently with the pairwise_nn chain below (buffers allocated here, on the main stream)
        dAu = torch.empty((Mc, F), dtype=torch.float32, device=dev)
        dU = torch.empty((Mc, Cu), dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        sums_2u, sums_1u = sums.take(ops.STAT_SLOTS * 2 * F), sums.take(ops.STAT_SLOTS * 2 * F)
        main, side = torch.cuda.current_stream(dev), _side_stream(dev)
        fork, join = torch.cuda.Event(), torch.cuda.Event()
        fork.record(main)
        side.wait_event(fork)
        with torch.cuda.stream(side):
            ops.bn_backward_prepare(Gu, H2u, s2u, 1.0, dg["2u"], db["2u"], sums=sums_2u)
            ops.linear_bwd(Gu, H2u, s2u, 1.0, H1u, W2u, scale1=s1u.scale, shift1=s1u.shift, slope1=sl[0], dX1=dAu, dW=dW["2u"], scratch=scr(dW["2u"]), scratch_stride=n_small)
            ops.bn_backward_prepare(dAu, H1u, s1u, sl[0], dg["1u"], db["1u"], sums=sums_1u)
            ops.linear_bwd(dAu, H1u, s1u, sl[0], U, W1u, dX1=dU, dW=dW["1u"], scratch=scr(dW["1u"]), scratch_stride=n_small)
            join.record(side)
        # pairwise_nn (its input gradient accumulates onto the fusion_nn branch)
        ops.bn_backward_prepare(Gy, H2p, s2p, 1.0, dg["2p"], db["2p"], sums=sums.take(ops.STAT_SLOTS * 2 * F))
        dA = torch.empty((M, F), dtype=torch.float32, device=dev)
        ops.linear_bwd(Gy, H2p, s2p, 1.0, H1p, W2p, scale1=s1p.scale, shift1=s1p.shift, slope1=sl[2], dX1=dA, dW=dW["2p"], scratch=scr(dW["2p"]), scratch_stride=n_small)
        ops.bn_backward_prepare(dA, H1p, s1p, sl[2], dg["1p"], db["1p"], sums=sums.take(ops.STAT_SLOTS * 2 * F))
        need_p = ctx.needs_input_grad[1]
        ops.linear_bwd(dA, H1p, s1p, sl[2], P, W1p, dX1=dP if need_p else None, acc1=True, dW=dW["1p"], scratch=scr(dW["1p"]), scratch_stride=n_small)

        main.wait_event(join)
        main.wait_event(join_aux)
        ops.grad_slots_reduce(wscr[2 * F * F:], small[2 * F * F:], n_small - 2 * F * F, n_small)   # all weight gradients, one launch
        grads = []
        for k in ("1u", "2u", "1p", "2p", "o", "f"):
            grads += [dW[k], dg[k], db[k]]
        return (dU.view(B, Nc, Cu) if dU is not None else None, dP.view(B, N, Cp) if need_p else None, None, None, None, None,
                None, None, *_param_grads(ctx.gbuf, [Gc, *grads]))


_THIRD = {}


def _third_stream(dev):
    """Fourth stream: in the fused backward the first layers' weight gradients (dW1 = dH1ᵀ·X) and input gradients (dX = dH1·W1)
    are independent kernels; the weight gradient runs here."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _THIRD:
        _THIRD[key] = torch.cuda.Stream(device=dev)
    return _THIRD[key]


def fused_eligible(unary, pairwise, neighbor_idx, steps, training, mods, F, Co):
    """The layer-specialised kernels (csrc/crf_fused.cu) cover the hot-path shape family: hidden width 16 (out_channels 64),
    16 neighbours, batch statistics in every BatchNorm, LeakyReLU-family activations in the reference's positions."""
    if F != 16 or Co != 64 or pairwise.shape[-1] != 64 or unary.shape[-1] not in (64, 128) or neighbor_idx.shape[-1] != 16 or steps < 1:
        return False
    if unary.dtype != torch.float32 or pairwise.dtype != torch.float32:
        return False
    for m in mods:
        bn = m.bn.batch_norm
        if not (training or not bn.track_running_stats) or bn.momentum is None:
            return False
    sl = [m.slope for m in mods]
    if any(v is None for v in sl) or sl[1] != 1.0 or sl[3] != 1.0 or not all(0.0 <= v <= 1.0 for v in sl):
        return False
    return True


class _CRFConvFusedFunction(torch.autograd.Function):
    """The same layer as _CRFConvFunction on the layer-specialised kernels: 13 launches forward, 14 backward for steps = 1
    (was 24 + 33), every BatchNorm finalize folded into the producing kernel, out_nn's backward reduced to one pass."""

    @staticmethod
    def forward(ctx, unary, pairwise, up_idx, neighbor_idx, steps, mods, gbuf, c, *params):
        if not (unary.is_cuda and pairwise.is_cuda):
            raise RuntimeError("crfconv_b200 layers run on CUDA tensors only (no CPU fallback)")
        ctx.gbuf = gbuf
        (W1u, _, _, W2u, _, _, W1p, _, _, W2p, _, _, Wo, _, _, Wf, _, _) = [p.detach().contiguous().float() for p in params]
        bns = [m.bn.batch_norm for m in mods]          # order: u0, u1, p0, p1, out, fusion
        sl = [m.slope for m in mods]
        B, Nc, Cu = unary.shape
        _, N, Cp = pairwise.shape
        K = neighbor_idx.shape[-1]
        dev = unary.device
        U, P = ops.as2d(unary), ops.as2d(pairwise)
        up = up_idx.detach().reshape(B, N).contiguous().to(torch.int64)
        nbr = neighbor_idx.detach().contiguous().to(torch.int64)
        Mc, M = B * Nc, B * N
        F, Co = 16, 64
        NP = ops.fused_part_floats()

        # one zero-filled allocation: [tcgen05 statistics slots of out_nn and fusion_nn | 8 counters]; partial-sum scratches need no init
        CI = ops.counter_ints()
        zf = ops.Flat(2 * ops.STAT_SLOTS * 2 * Co + 8 * CI, torch.float32, dev, scratch=True)
        st_o, st_f = zf.take(ops.STAT_SLOTS * 2 * Co), zf.take(ops.STAT_SLOTS * 2 * Co)
        cnt = zf.take(8 * CI).view(torch.int32).view(8, CI)
        parts = torch.empty((4, NP), dtype=torch.float32, device=dev)
        s1u, s2u, s1p, s2p = (ops.BN(F, dev, alloc_stats=False) for _ in range(4))
        so, sf = ops.BN(Co, dev, st_o), ops.BN(Co, dev, st_f)
        H1u, H2u = torch.empty((Mc, F), dtype=torch.float32, device=dev), torch.empty((Mc, F), dtype=torch.float32, device=dev)
        H1p, H2p = torch.empty((M, F), dtype=torch.float32, device=dev), torch.empty((M, F), dtype=torch.float32, device=dev)
        main, side, aux = torch.cuda.current_stream(dev), _side_stream(dev), _aux_stream(dev)
        fork, join, join_aux = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
        cc = c.detach().contiguous().float()
        Cm, Minv = torch.empty_like(cc), torch.empty_like(cc)
        cscr = torch.empty(3 * F * F, dtype=torch.float64, device=dev)
        fork.record(main)
        side.wait_event(fork)
        aux.wait_event(fork)
        with torch.cuda.stream(aux):
            ops.crf_compat_fwd(cc, out=(Cm, Minv), scratch=cscr)
            join_aux.record(aux)
        with torch.cuda.stream(side):                  # unary_nn (:58)
            ops.lin16_fwd(U, W1u, s1u, bns[0], parts[0], cnt[0], out=H1u)
            ops.lin16_fwd(H1u, W2u, s2u, bns[1], parts[1], cnt[1], pre=s1u, pslope=sl[0], out=H2u)
            join.record(side)
        ops.lin16_fwd(P, W1p, s1p, bns[2], parts[2], cnt[2], out=H1p)          # pairwise_nn (:59)
        ops.lin16_fwd(H1p, W2p, s2p, bns[3], parts[3], cnt[3], pre=s1p, pslope=sl[2], out=H2p)
        main.wait_event(join)
        main.wait_event(join_aux)
        z = ops.crf_upsample_fwd(H2u, s2u, up, B, N, Nc)                          # (:60)
        xs = [z]
        for _ in range(steps):                                                    # (:68-72)
            xs.append(ops.crf_step_fwd(H2p, s2p.scale, z, xs[-1], nbr, Cm, Minv, B, N, K))
        H3 = ops.up16_fwd(xs[-1], Wo, so, bns[4], cnt[4])                       # out_nn (:74)
        Hf = ops.linear_fwd_bn(H3, Wf, sf, bns[5], cnt[5], scale1=so.scale, shift1=so.shift, slope1=sl[4], X2=P)   # fusion_nn (:76)
        out = ops.bn_act_fwd(Hf, sf, sl[5])
        nbt = [b.num_batches_tracked for b in bns if b.track_running_stats and b.num_batches_tracked is not None]
        from . import common as _common
        if nbt and _common._NBT_DEFER is not None:
            _common._NBT_DEFER.extend(nbt)                # bumped once per step by the network's forward
        elif nbt:
            torch._foreach_add_(nbt, 1)

        ctx.dims = (B, N, Nc, K, F, Co, Cu, Cp, steps)
        ctx.bn = (s1u, s2u, s1p, s2p, so, sf)
        ctx.sl = sl
        ctx.gamma_y = bns[3].weight.detach() if bns[3].weight is not None else torch.ones(F, dtype=torch.float32, device=dev)
        ctx.save_for_backward(U, P, up, nbr, H1u, H2u, H1p, H2p, H3, Hf, Cm, Minv, cc, W1u, W2u, W1p, W2p, Wo, Wf, *xs)
        return out.view(B, N, Co)

    @staticmethod
    def backward(ctx, gout):
        (U, P, up, nbr, H1u, H2u, H1p, H2p, H3, Hf, Cm, Minv, cc, W1u, W2u, W1p, W2p, Wo, Wf, *xs) = ctx.saved_tensors
        B, N, Nc, K, F, Co, Cu, Cp, steps = ctx.dims
        s1u, s2u, s1p, s2p, so, sf = ctx.bn
        sl = ctx.sl
        dev = gout.device
        Mc, M = B * Nc, B * N
        z = xs[0]
        g2 = ops.as2d(gout)
        NP = ops.fused_part_floats()

        wl = (("1u", W1u), ("2u", W2u), ("1p", W1p), ("2p", W2p), ("o", Wo), ("f", Wf))
        cl = (("1u", F), ("2u", F), ("1p", F), ("2p", F), ("o", Co), ("f", Co))
        n_small = sum(w.numel() for _, w in wl) + 2 * sum(n for _, n in cl) + 3 * F * F
        n_out = ops.out_bwd_part_floats()
        n_big = (steps + 1) * M * F + Mc * F
        # ONE zero-filled allocation: [small grads | weight-grad partial slots | fusion BN Σ slots | out_nn partials | y sums | counters | scatter targets]
        CI = ops.counter_ints()
        flat = ops.Flat(n_small * (1 + ops.GRAD_SLOTS) + ops.STAT_SLOTS * 2 * Co + n_out + 128 + 8 * CI + n_big, torch.float32, dev)
        small = flat.take(n_small)
        wscr = flat.take(ops.GRAD_SLOTS * n_small)
        sums_f = flat.take(ops.STAT_SLOTS * 2 * Co)
        out_part = flat.take(n_out)
        ysum = flat.take(128)
        cnt = flat.take(8 * CI).view(torch.int32).view(8, CI)
        big = ops.Flat.__new__(ops.Flat); big.buf, big.off = flat.take(n_big), 0
        parts = torch.empty((3, NP), dtype=torch.float32, device=dev)
        cursor = [0]

        def take_small(*shape):
            n = 1
            for d in shape:
                n *= int(d)
            v = small[cursor[0]:cursor[0] + n].view(*shape)
            cursor[0] += n
            return v

        def scr(t):                                          # partial-slot region that mirrors the small-gradient view `t`
            return wscr[(t.data_ptr() - small.data_ptr()) // 4:]

        GC, GM = take_small(F, F), take_small(F, F)
        dW = {k: take_small(*w.shape) for k, w in wl}
        dg = {k: take_small(n) for k, n in cl}
        db = {k: take_small(n) for k, n in cl}
        # fusion_nn (:76): BatchNorm backward sums (+ finalize), input gradients dO | dP and weight gradient on tcgen05
        ops.bn_backward_prepare_fin(g2, Hf, sf, sl[5], dg["f"], db["f"], sums_f, cnt[0])
        dO = torch.empty((M, Co), dtype=torch.float32, device=dev)
        dP = torch.empty((M, Cp), dtype=torch.float32, device=dev)
        main = torch.cuda.current_stream(dev)
        # one pass over dY, Hf, H3 and P for both gradients (csrc/linear3b.cu)
        ops.linear_bwd(g2, Hf, sf, sl[5], H3, Wf, scale1=so.scale, shift1=so.shift, slope1=sl[4], X2=P, dX1=dO, dX2=dP, dW=dW["f"], scratch=scr(dW["f"]), scratch_stride=n_small)
        # out_nn (:74) in one pass over dO
        Q, a0 = torch.empty((F, F), dtype=torch.float32, device=dev), torch.empty(F, dtype=torch.float32, device=dev)
        T = ops.out16_bwd(dO, H3, so, sl[4], xs[-1], Wo, out_part, cnt[1], dg["o"], db["o"], dW["o"], Q, a0)
        # mean-field steps, last to first (:68-72)
        Gy = big.take(M, F)
        Gz = torch.empty((M, F), dtype=torch.float32, device=dev)
        g = T
        for t in range(steps, 0, -1):
            gprev = big.take(M, F)
            first = t == steps
            ops.crf_step_bwd_fused(H2p, s2p, z, xs[t - 1], nbr, Cm, Minv, g, xs[-1] if first else None, Q if first else None,
                                   a0 if first else None, Gz, not first, gprev, Gy, scr(GC), scr(GM), n_small, ysum, B, N, K,
                                   t == 1, cnt[2], ctx.gamma_y, dg["2p"], db["2p"])
            g = gprev
        Gc = take_small(F, F)
        aux = _aux_stream(dev)
        fork_aux, join_aux = torch.cuda.Event(), torch.cuda.Event()
        bscr = torch.empty(3 * F * F, dtype=torch.float64, device=dev)
        fork_aux.record(main)
        aux.wait_event(fork_aux)
        with torch.cuda.stream(aux):                             # off the critical path: Gc is only needed when backward returns
            ops.grad_slots_reduce(wscr, small, 2 * F * F, n_small)    # fold the GC / GM partial slots
            ops.crf_compat_bwd(cc, Minv, GC, GM, Gc, scratch=bscr)
            join_aux.record(aux)
        Gu = big.take(Mc, F)
        ops.crf_upsample_bwd_fused(Gz, g, up, H2u, s2u, Gu, B, N, Nc, parts[0], cnt[3], dg["2u"], db["2u"])   # dL/dz = Σ_t h^t + g^0
        need_u, need_p = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        dV1u = torch.empty((Mc, F), dtype=torch.float32, device=dev)
        dV1p = torch.empty((M, F), dtype=torch.float32, device=dev)
        dU = torch.empty((Mc, Cu), dtype=torch.float32, device=dev) if need_u else None
        side, third = _side_stream(dev), _third_stream(dev)
        fork, join, fork3, join3 = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
        fork.record(main)
        side.wait_event(fork)
        with torch.cuda.stream(side):                            # unary_nn
            ops.mid16_bwd(Gu, H2u, s2u, H1u, s1u, sl[0], W2u, scr(dW["2u"]), n_small, parts[1], cnt[4], dg["1u"], db["1u"], out=dV1u)
            ops.in16_wgrad(dV1u, H1u, s1u, U, scr(dW["1u"]), n_small)
            if need_u:
                ops.in16_dgrad(dV1u, H1u, s1u, W1u, dU, False)
            join.record(side)
        # pairwise_nn (its input gradient accumulates onto the fusion_nn branch)
        ops.mid16_bwd(Gy, H2p, s2p, H1p, s1p, sl[2], W2p, scr(dW["2p"]), n_small, parts[2], cnt[5], dg["1p"], db["1p"], out=dV1p)
        fork3.record(main)
        third.wait_event(fork3)
        with torch.cuda.stream(third):
            ops.in16_wgrad(dV1p, H1p, s1p, P, scr(dW["1p"]), n_small)
            join3.record(third)
        if need_p:
            ops.in16_dgrad(dV1p, H1p, s1p, W1p, dP, True)
        main.wait_event(join)
        main.wait_event(join3)
        main.wait_event(join_aux)
        ops.grad_slots_reduce(wscr[2 * F * F:], small[2 * F * F:], n_small - 2 * F * F, n_small)   # all weight gradients, one launch
        grads = []
        for k in ("1u", "2u", "1p", "2p", "o", "f"):
            grads += [dW[k], dg[k], db[k]]
        return (dU.view(B, Nc, Cu) if dU is not None else None, dP.view(B, N, Cp) if need_p else None, None, None, None, None,
                None, *_param_grads(ctx.gbuf, [Gc, *grads]))


class ContinuousGaussianCRFConv(nn.Module):
    def __init__(self, unary_channels, pairwise_channels, out_channels=None, steps=1):
        super(ContinuousGaussianCRFConv, self).__init__()
        self.unary_channels = unary_channels
        self.pairwise_channels = pairwise_channels
        self.out_channels = out_channels if out_channels is not None else pairwise_channels
        self.hidden_channels = self.out_channels // 4
        self.steps = steps

        act = lambda: nn.LeakyReLU(negative_slope=0.1)   # noqa: E731
        self.unary_nn = nn.Sequential(MLP(self.unary_channels, self.hidden_channels, activation=act()),
                                      MLP(self.hidden_channels, self.hidden_channels, activation=None))
        self.pairwise_nn = nn.Sequential(MLP(self.pairwise_channels, self.hidden_channels, activation=act()),
                                         MLP(self.hidden_channels, self.hidden_channels, activation=None))
        self.out_nn = MLP(self.hidden_channels, self.out_channels, activation=act())
        self.fusion_nn = MLP(self.out_channels * 2, self.out_channels, activation=act())
        self.c = nn.Parameter(torch.Tensor(self.hidden_channels, self.hidden_channels))
        self._reset_parameters()

    def _reset_parameters(self):
        nn.init.eye_(self.c)

    def forward(self, unary, pairwise, up_idx, neighbor_idx):
        if self.pairwise_channels != self.out_channels:
            # the reference's fusion_nn silently requires this too (continuous_crf_conv_big.py:29,76)
            raise RuntimeError("ContinuousGaussianCRFConv: fusion_nn needs pairwise_channels == out_channels")
        if self.hidden_channels not in (4, 8, 16, 32, 64):
            raise RuntimeError("ContinuousGaussianCRFConv: hidden channels (out_channels // 4) must be 4, 8, 16, 32 or 64")
        mods = (self.unary_nn[0], self.unary_nn[1], self.pairwise_nn[0], self.pairwise_nn[1], self.out_nn, self.fusion_nn)
        params = []
        for m in (self.unary_nn[0], self.unary_nn[1], self.pairwise_nn[0], self.pairwise_nn[1], self.out_nn, self.fusion_nn):
            params += list(_mlp_params(m))
        from .common import direct_grad_buffers
        gbuf = direct_grad_buffers(self.c, *params)
        if gbuf is not None and any(b is None for b in gbuf):
            gbuf = None
        if USE_FUSED and fused_eligible(unary, pairwise, neighbor_idx, self.steps, self.training, mods, self.hidden_channels, self.out_channels):
            return _CRFConvFusedFunction.apply(unary, pairwise, up_idx, neighbor_idx, self.steps, mods, gbuf, self.c, *params)
        return _CRFConvFunction.apply(unary, pairwise, up_idx, neighbor_idx, self.steps, self.training, mods, gbuf, self.c, *params)
