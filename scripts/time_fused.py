"""CUDA-event timing of every kernel of the fused CRF layer step in isolation (S1 shape, B clouds), with the generic kernels of the
same work beside them.  Each op runs `reps` times back to back on inputs that (together) exceed L2; prints us per call and GB/s of
the op's own algorithmic bytes.   python scripts/time_fused.py [B]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from crfconv_b200 import ops
from crfconv_b200.nearest_neighbors import knn_batch

B = int(sys.argv[1]) if len(sys.argv) > 1 else 6
dev = torch.device("cuda")
N, K, F, Co, Cu = bench.N_POINTS, 16, 16, 64, 128
Nc = N // 4
M, Mc = B * N, B * Nc
g = torch.Generator().manual_seed(0)
s = bench.make_inputs(torch, B, dev, seed=0)
P, U = s["pairwise"].reshape(M, Co).contiguous(), s["unary"].reshape(Mc, Cu).contiguous()
nbr, up = s["neighbor_idx"], s["up_idx"].reshape(B, N).contiguous()
rnd = lambda *sh: torch.randn(*sh, device=dev)
bnm16, bnm64 = torch.nn.BatchNorm1d(16).to(dev), torch.nn.BatchNorm1d(64).to(dev)
CI = ops.counter_ints()
cnt = torch.zeros(CI, dtype=torch.int32, device=dev)
part = torch.empty(ops.fused_part_floats(), device=dev)


def bn(C, H=None):
    st = ops.BN(C, dev)
    st.scale.fill_(1.0); st.shift.zero_(); st.mean.zero_(); st.invstd.fill_(1.0); st.k1.zero_(); st.k2.fill_(0.01)
    st.count, st.training = (H.shape[0] if H is not None else M), True
    return st


def timeit(name, fn, nbytes, reps=20):
    """`reps` back-to-back calls captured into ONE CUDA graph and replayed: no Python / ctypes launch overhead in the measurement."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / reps * 1e3
    print(f"{name:44s} {us:8.1f} us   {nbytes / us / 1e3:8.1f} GB/s   ({nbytes / 1e6:.0f} MB)", flush=True)


W1p, W1u, W2, Wo, Wf = rnd(16, Co) / 8, rnd(16, Cu) / 11, rnd(16, 16) / 4, rnd(Co, 16) / 4, rnd(Co, 2 * Co) / 11
H1p, H2p, H1u, H2u = rnd(M, F), rnd(M, F), rnd(Mc, F), rnd(Mc, F)
b1, b2, b3, bf = bn(F), bn(F), bn(Co), bn(Co)
fb = 4
print(f"S1 shape, {B} clouds: M = {M}, Mc = {Mc}")
timeit("lin16_fwd[64]  P -> H1p", lambda: ops.lin16_fwd(P, W1p, b1, bnm16, part, cnt, out=H1p), fb * M * (Co + F))
timeit("  generic linear_fwd[64->16]", lambda: ops.linear_fwd(P, W1p, stats=b1.stats, out=H1p), fb * M * (Co + F))
timeit("lin16_fwd[128] U -> H1u", lambda: ops.lin16_fwd(U, W1u, b1, bnm16, part, cnt, out=H1u), fb * Mc * (Cu + F))
timeit("  generic linear_fwd[128->16]", lambda: ops.linear_fwd(U, W1u, stats=b1.stats, out=H1u), fb * Mc * (Cu + F))
timeit("lin16_fwd[16]  H1p -> H2p", lambda: ops.lin16_fwd(H1p, W2, b2, bnm16, part, cnt, pre=b1, pslope=0.1, out=H2p), fb * M * 2 * F)
timeit("  generic linear_fwd[16->16]", lambda: ops.linear_fwd(H1p, W2, scale1=b1.scale, shift1=b1.shift, slope1=0.1, stats=b2.stats, out=H2p), fb * M * 2 * F)
z = ops.crf_upsample_fwd(H2u, b2, up, B, N, Nc)
timeit("crf_upsample_fwd", lambda: ops.crf_upsample_fwd(H2u, b2, up, B, N, Nc), fb * (Mc * F + M * F) + 8 * M)
c = torch.eye(F, device=dev) + 0.1 * rnd(F, F)
Cm, Minv = ops.crf_compat_fwd(c)
timeit("crf_step_fwd", lambda: ops.crf_step_fwd(H2p, b2.scale, z, z, nbr, Cm, Minv, B, N, K), fb * M * F * 3 + 8 * M * K)
x1 = ops.crf_step_fwd(H2p, b2.scale, z, z, nbr, Cm, Minv, B, N, K)
H3, Hf = torch.empty(M, Co, device=dev), torch.empty(M, Co, device=dev)
b3.stats.zero_(); bf.stats.zero_()
timeit("up16_fwd[64] (mma.sync + fin)", lambda: ops.up16_fwd(x1, Wo, b3, bnm64, cnt, out=H3), fb * M * (F + Co))
timeit("linear_fwd_bn[16->64] (tcgen05 + fin)", lambda: ops.linear_fwd_bn(x1, Wo, b3, bnm64, cnt, out=H3), fb * M * (F + Co))
timeit("  linear_fwd[16->64] (no fin)", lambda: ops.linear_fwd(x1, Wo, stats=b3.stats, out=H3), fb * M * (F + Co))
timeit("linear_fwd_bn[128->64] (tcgen05 + fin)", lambda: ops.linear_fwd_bn(H3, Wf, bf, bnm64, cnt, scale1=b3.scale, shift1=b3.shift, slope1=0.1, X2=P, out=Hf), fb * M * 3 * Co)
timeit("  linear_fwd[128->64] (no fin)", lambda: ops.linear_fwd(H3, Wf, scale1=b3.scale, shift1=b3.shift, slope1=0.1, X2=P, stats=bf.stats, out=Hf), fb * M * 3 * Co)
out = torch.empty(M, Co, device=dev)
timeit("bn_act_fwd[64]", lambda: ops.bn_act_fwd(Hf, bf, 0.1, out=out), fb * M * 2 * Co)
# ---- backward
g2 = rnd(M, Co)
dg, db = torch.zeros(Co, device=dev), torch.zeros(Co, device=dev)
sums = torch.zeros(ops.STAT_SLOTS * 2 * Co, device=dev)
timeit("bn_backward_prepare_fin[64]", lambda: ops.bn_backward_prepare_fin(g2, Hf, bf, 0.1, dg, db, sums, cnt), fb * M * 2 * Co)
timeit("  bn_backward_prepare[64] (2 launches)", lambda: ops.bn_backward_prepare(g2, Hf, bf, 0.1, dg, db, sums=sums), fb * M * 2 * Co)
dO, dP = torch.empty(M, Co, device=dev), torch.empty(M, Co, device=dev)
dWf = torch.zeros(Co, 2 * Co, device=dev)
scr = torch.zeros(ops.GRAD_SLOTS * 20000, device=dev)
timeit("linear_bwd[64<-128] one pass (bwd3)", lambda: ops.linear_bwd(g2, Hf, bf, 0.1, H3, Wf, scale1=b3.scale, shift1=b3.shift, slope1=0.1, X2=P, dX1=dO, dX2=dP, dW=dWf, scratch=scr, scratch_stride=20000), fb * M * (2 * Co + 2 * Co + 2 * Co))
timeit("  dgrad3 + wgrad3 (two calls)", lambda: (ops.linear_bwd(g2, Hf, bf, 0.1, H3, Wf, scale1=b3.scale, shift1=b3.shift, slope1=0.1, X2=P, dX1=dO, dX2=dP),
                                                ops.linear_bwd(g2, Hf, bf, 0.1, H3, Wf, scale1=b3.scale, shift1=b3.shift, slope1=0.1, X2=P, dW=dWf, scratch=scr, scratch_stride=20000)), fb * M * (2 * Co + 2 * Co + 2 * Co))
timeit("  dgrad only", lambda: ops.linear_bwd(g2, Hf, bf, 0.1, H3, Wf, scale1=b3.scale, shift1=b3.shift, slope1=0.1, X2=P, dX1=dO, dX2=dP), fb * M * 4 * Co)
timeit("  wgrad only", lambda: ops.linear_bwd(g2, Hf, bf, 0.1, H3, Wf, scale1=b3.scale, shift1=b3.shift, slope1=0.1, X2=P, dW=dWf, scratch=scr, scratch_stride=20000), fb * M * 4 * Co)
opart = torch.zeros(ops.out_bwd_part_floats(), device=dev)
dW3, Q, a0, T = torch.zeros(Co, F, device=dev), torch.empty(F, F, device=dev), torch.empty(F, device=dev), torch.empty(M, F, device=dev)
timeit("out16_bwd", lambda: ops.out16_bwd(dO, H3, b3, 0.1, x1, Wo, opart, cnt, dg, db, dW3, Q, a0, out=T), fb * M * (2 * Co + 2 * F))
dX1 = torch.empty(M, F, device=dev)
timeit("  generic out_nn bwd (reduce + dgrad + wgrad)", lambda: (ops.bn_backward_prepare(dO, H3, b3, 0.1, dg, db, sums=sums),
                                                                ops.linear_bwd(dO, H3, b3, 0.1, x1, Wo, dX1=dX1, dW=dW3, scratch=scr, scratch_stride=20000)), fb * M * (2 * Co + 2 * F))
Gz, gp, Gy = torch.empty(M, F, device=dev), torch.zeros(M, F, device=dev), torch.zeros(M, F, device=dev)
ysum = torch.zeros(128, device=dev)
gam = torch.ones(F, device=dev)
d16, e16 = torch.zeros(F, device=dev), torch.zeros(F, device=dev)
Q.copy_(0.01 * (Q.new_ones(F, F))); a0.zero_()
timeit("crf_step_bwd_fused", lambda: ops.crf_step_bwd_fused(H2p, b2, z, z, nbr, Cm, Minv, T, x1, Q, a0, Gz, False, gp, Gy, scr, scr[256:], 20000,
                                                             ysum, B, N, K, True, cnt, gam, d16, e16), fb * M * F * 7 + 8 * M * K)
mo, vo, ho = (torch.empty(M, F, device=dev) for _ in range(3))
cgrad, w2grad, w1grad = torch.zeros(F, F, device=dev), torch.zeros(F, F, device=dev), torch.zeros(16, Co, device=dev)
timeit("  generic crf_step_bwd + GC/GM GEMMs", lambda: (ops.crf_step_bwd(H2p, b2.scale, z, z, nbr, Cm, Minv, T, Gz, gp, Gy, mo, vo, ho, False, B, N, K),
                                                        ops.linear_bwd(mo, None, None, 1.0, ho, c, dW=cgrad, scratch=scr, scratch_stride=20000),
                                                        ops.linear_bwd(vo, None, None, 1.0, T, c, dW=cgrad, scratch=scr, scratch_stride=20000)), fb * M * F * 7 + 8 * M * K)
Gu = torch.zeros(Mc, F, device=dev)
timeit("crf_upsample_bwd_fused", lambda: ops.crf_upsample_bwd_fused(Gz, gp, up, H2u, b2, Gu, B, N, Nc, part, cnt, d16, e16), fb * (2 * M * F + Mc * F) + 8 * M)
dV1 = torch.empty(M, F, device=dev)
timeit("mid16_bwd (pairwise)", lambda: ops.mid16_bwd(Gy, H2p, b2, H1p, b1, 0.1, W2, scr, 20000, part, cnt, d16, e16, out=dV1), fb * M * F * 4)
timeit("  generic 16x16 bwd (reduce + narrow::bwd)", lambda: (ops.bn_backward_prepare(Gy, H2p, b2, 1.0, d16, e16, sums=sums[:ops.STAT_SLOTS * 32]),
                                                            ops.linear_bwd(Gy, H2p, b2, 1.0, H1p, W2, scale1=b1.scale, shift1=b1.shift, slope1=0.1, dX1=dV1, dW=w2grad, scratch=scr, scratch_stride=20000)), fb * M * F * 4)
timeit("in16_dgrad[64] (+=)", lambda: ops.in16_dgrad(dV1, H1p, b1, W1p, dP, True), fb * M * (2 * F + 2 * Co))
timeit("in16_wgrad[64]", lambda: ops.in16_wgrad(dV1, H1p, b1, P, scr, 20000), fb * M * (2 * F + Co))
timeit("  generic P-layer bwd (reduce + dgrad + wgrad)", lambda: (ops.bn_backward_prepare(dV1, H1p, b1, 0.1, d16, e16, sums=sums[:ops.STAT_SLOTS * 32]),
                                                                ops.linear_bwd(dV1, H1p, b1, 0.1, P, W1p, dX1=dP, acc1=True, dW=w1grad, scratch=scr, scratch_stride=20000)), fb * M * (4 * F + 3 * Co))
dV1u, dU = torch.empty(Mc, F, device=dev), torch.empty(Mc, Cu, device=dev)
timeit("in16_dgrad[128] (=)", lambda: ops.in16_dgrad(dV1u, H1u, b1, W1u, dU, False), fb * Mc * (2 * F + Cu))
timeit("in16_wgrad[128]", lambda: ops.in16_wgrad(dV1u, H1u, b1, U, scr, 20000), fb * Mc * (2 * F + Cu))
