"""GPU parity of the one-pass input + weight gradient kernel (csrc/linear3b.cu), which crfconv_linear_bwd takes when a call asks
for dW and dX1 / dX2 at 32 < Cout <= 64, 64 < C1 + C2 <= 128 and >= 8,192 rows.  References: an fp64 torch statement built from
the product's own forward output H (as in test_linear_ops_gpu.py), and the separate input-gradient-only and weight-gradient-only
calls, which keep the two-kernel path.  Tolerance relative to each tensor's max: 2e-5 (3xTF32)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 2e-5


@pytest.fixture(scope="module")
def ops():
    from crfconv_b200 import ops as o
    return o


def lrelu(v, s):
    return torch.where(v > 0, v, v * s)


def rel(a, b):
    b = b.double()
    return float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-30))


class Case:
    """Inputs of fusion_nn's backward (Linear [C1 | C2] -> Cout, BatchNorm + LeakyReLU(0.1)); bn=False: a plain Linear."""

    def __init__(self, ops, M, C1, C2, Cout, bn=True, seed=0):
        g = torch.Generator(device="cuda").manual_seed(seed + M + C1 + C2)
        rn = lambda *s: torch.randn(*s, generator=g, device="cuda")   # noqa: E731
        self.ops, self.M, self.C1, self.C2, self.Cout = ops, M, C1, C2, Cout
        self.X1, self.X2 = rn(M, C1), (rn(M, C2) if C2 else None)
        self.W = rn(Cout, C1 + C2) / (C1 + C2) ** 0.5
        self.sc1, self.sh1 = 1 + 0.2 * rn(C1), 0.2 * rn(C1)           # the BN3 + LeakyReLU(0.1) prologue of X1
        self.dY = rn(M, Cout)
        A = lrelu(self.X1.double() * self.sc1.double() + self.sh1.double(), 0.1)
        self.A = torch.cat([A, self.X2.double()], 1) if C2 else A
        self.bn = None
        if bn:
            gamma, beta = 1 + 0.2 * rn(Cout), 0.2 * rn(Cout)
            st = ops.BN(Cout, self.X1.device)
            self.H = ops.linear_fwd(self.X1, self.W, scale1=self.sc1, shift1=self.sh1, slope1=0.1, X2=self.X2, stats=st.stats)
            ops.bn_finalize_fwd(st, M, gamma, beta, 1e-5, 0.1, True, None, None)
            ops.bn_backward_prepare(self.dY, self.H, st, 0.1, torch.zeros(Cout, device="cuda"), torch.zeros(Cout, device="cuda"))
            self.bn = st
            Hd = self.H.double()
            mu, var = Hd.mean(0), Hd.var(0, unbiased=False)
            Hh = (Hd - mu) * (var + 1e-5).rsqrt()
            dV = torch.where(Hh * gamma.double() + beta.double() > 0, self.dY.double(), self.dY.double() * 0.1)
            self.dH = gamma.double() * (var + 1e-5).rsqrt() * (dV - dV.mean(0) - Hh * (dV * Hh).mean(0))
        else:
            self.H = None
            self.dH = self.dY.double()

    def call(self, dX1=None, dX2=None, dW=None, acc1=False, acc2=False, scratch=None, scratch_stride=0):
        self.ops.linear_bwd(self.dY, self.H, self.bn, 0.1 if self.bn else 1.0, self.X1, self.W, scale1=self.sc1, shift1=self.sh1,
                            slope1=0.1, X2=self.X2, dX1=dX1, acc1=acc1, dX2=dX2, acc2=acc2, dW=dW, scratch=scratch,
                            scratch_stride=scratch_stride)

    def ref(self):
        dA = self.dH @ self.W.double()
        return dA[:, :self.C1], dA[:, self.C1:], self.dH.t() @ self.A


def _launches(ops, fn):
    n0 = ops.COUNTERS["launches"]
    fn()
    return ops.COUNTERS["launches"] - n0


@pytest.mark.parametrize("M", [245760, 8193, 245759])
def test_fusion_nn_shape(ops, M):
    """S1 fusion_nn: C1 = 64 (BN3 + LeakyReLU prologue), C2 = 64, Cout = 64; ragged row counts around it."""
    c = Case(ops, M, 64, 64, 64)
    dX1, dX2, dW = torch.empty_like(c.X1), torch.empty_like(c.X2), torch.zeros_like(c.W)
    assert _launches(ops, lambda: c.call(dX1, dX2, dW)) == 1
    r1, r2, rw = c.ref()
    assert rel(dX1, r1) < TOL and rel(dX2, r2) < TOL and rel(dW, rw) < TOL
    # the input-gradient-only and weight-gradient-only calls take the two separate kernels
    e1, e2, ew = torch.empty_like(c.X1), torch.empty_like(c.X2), torch.zeros_like(c.W)
    assert _launches(ops, lambda: (c.call(e1, e2), c.call(dW=ew))) == 2
    assert rel(dX1, e1) < TOL and rel(dX2, e2) < TOL and rel(dW, ew) < TOL


def test_slotted_weight_gradient(ops):
    """dW through the caller's partial slots (the fused CRF layer's flat gradient layout) and its reduce."""
    c = Case(ops, 40960, 64, 64, 64)
    n = c.W.numel()
    stride = n + 100
    scratch = torch.zeros(ops.GRAD_SLOTS * stride, device="cuda")
    dX1, dX2, dW = torch.empty_like(c.X1), torch.empty_like(c.X2), torch.zeros_like(c.W)
    assert _launches(ops, lambda: c.call(dX1, dX2, dW, scratch=scratch, scratch_stride=stride)) == 1
    ops.grad_slots_reduce(scratch, dW.view(-1), n, stride)
    r1, r2, rw = c.ref()
    assert rel(dX1, r1) < TOL and rel(dX2, r2) < TOL and rel(dW, rw) < TOL


@pytest.mark.parametrize("M,C1,C2,Cout,bn", [
    (20000, 128, 0, 64, True),      # one input segment of 128 channels
    (20000, 64, 64, 64, False),     # plain Linear: dH = dY
    (9001, 96, 0, 48, False),       # three input blocks, Cout padded to 64
    (9001, 36, 44, 40, False),      # blocks with channel padding in both segments
])
def test_variants(ops, M, C1, C2, Cout, bn):
    c = Case(ops, M, C1, C2, Cout, bn=bn)
    dX1, dX2, dW = torch.empty_like(c.X1), (torch.empty_like(c.X2) if C2 else None), torch.zeros_like(c.W)
    assert _launches(ops, lambda: c.call(dX1, dX2, dW)) == 1
    r1, r2, rw = c.ref()
    assert rel(dX1, r1) < TOL and rel(dW, rw) < TOL
    if C2:
        assert rel(dX2, r2) < TOL


def test_accumulate_and_missing_destination(ops):
    c = Case(ops, 30000, 64, 64, 64, seed=5)
    r1, r2, rw = c.ref()
    b1, b2 = torch.randn_like(c.X1), torch.randn_like(c.X2)
    dX1, dX2, dW = b1.clone(), b2.clone(), torch.zeros_like(c.W)
    c.call(dX1, dX2, dW, acc1=True, acc2=True)
    assert rel(dX1, r1 + b1.double()) < TOL and rel(dX2, r2 + b2.double()) < TOL and rel(dW, rw) < TOL
    # dX1 = None: only dX2 is written (the rows of a frozen first input)
    dX2, dW = torch.empty_like(c.X2), torch.zeros_like(c.W)
    assert _launches(ops, lambda: c.call(None, dX2, dW)) == 1
    assert rel(dX2, r2) < TOL and rel(dW, rw) < TOL


def test_cuda_graph_replay(ops):
    c = Case(ops, 245760, 64, 64, 64, seed=9)
    dX1, dX2, dW = torch.empty_like(c.X1), torch.empty_like(c.X2), torch.zeros_like(c.W)
    c.call(dX1, dX2, dW)
    torch.cuda.synchronize()
    eager = (dX1.clone(), dX2.clone(), dW.clone())
    gX1, gX2, gW = torch.empty_like(c.X1), torch.empty_like(c.X2), torch.zeros_like(c.W)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        c.call(gX1, gX2, gW)                 # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gW.zero_()
        c.call(gX1, gX2, gW)
    for _ in range(2):
        gX1.zero_(); gX2.zero_()
        graph.replay()
    torch.cuda.synchronize()
    assert rel(gX1, eager[0]) < 1e-6 and rel(gX2, eager[1]) < 1e-6 and rel(gW, eager[2]) < TOL
