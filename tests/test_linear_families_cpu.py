"""Every GEMM kernel of the Linear families (csrc/linear*.cu) has at least one case in tests/test_linear_families_gpu.py that
asserts, through the profiler, that the kernel ran.  A kernel added without such a case fails here, on a machine without a GPU."""
import os
import re

from tests import test_linear_families_gpu as families

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "crfconv_b200", "csrc")

# Kernels that are not GEMMs and have no dispatch of their own: the BatchNorm bookkeeping around a Linear and the reduce of
# weight-gradient partial slots.
EXCLUDED = {
    "lin::bn_finalize_fwd_kernel": "BatchNorm statistics → scale/shift; run by crfconv_bn_finalize_fwd and after linear_fwd_bn's two-launch path",
    "lin::bn_act_fwd_kernel": "elementwise BatchNorm affine + LeakyReLU, no contraction",
    "lin::bn_bwd_reduce_kernel": "BatchNorm-backward column sums (k1 / k2), no contraction",
    "lin::bn_finalize_bwd_kernel": "BatchNorm-backward finalize of the column sums",
    "lin::grad_slots_reduce_kernel": "folds weight-gradient partial slots; checked through the slotted cases of the GPU file",
}

_OPEN = re.compile(r"^\s*namespace\s+(\w+)\s*\{")
_CLOSE = re.compile(r"^\s*\}\s*//\s*namespace\s+(\w+)")
_KERNEL = re.compile(r"__global__\s+void\s+(?:__launch_bounds__\((?:[^()]|\([^()]*\))*\)\s+)?(\w+)\s*\(")


def global_kernels():
    """{'lin2::fwd2t_kernel', ...}: the __global__ functions of csrc/linear*.cu, qualified below namespace crf."""
    found = set()
    for fn in sorted(os.listdir(CSRC)):
        if not (fn.startswith("linear") and fn.endswith(".cu")):
            continue
        stack = []
        with open(os.path.join(CSRC, fn)) as f:
            for line in f:
                m = _OPEN.match(line)
                if m:
                    stack.append(m.group(1))
                    continue
                m = _CLOSE.match(line)
                if m:
                    assert stack and stack[-1] == m.group(1), f"{fn}: unbalanced namespace {m.group(1)}"
                    stack.pop()
                    continue
                if "__global__" in line:
                    k = _KERNEL.search(line)
                    assert k, f"{fn}: cannot parse kernel declaration: {line.strip()}"
                    assert stack[:1] == ["crf"], f"{fn}: kernel {k.group(1)} outside namespace crf"
                    found.add("::".join(stack[1:] + [k.group(1)]))
        assert not stack, f"{fn}: namespaces left open: {stack}"
    return found


def test_every_linear_gemm_kernel_has_a_case():
    kernels = global_kernels()
    assert set(EXCLUDED) <= kernels, f"excluded kernels that no longer exist: {set(EXCLUDED) - kernels}"
    gemm = kernels - set(EXCLUDED)
    covered = {k for c in families.CASES for k in c.kernels}
    assert gemm - covered == set(), f"GEMM kernels without a case in test_linear_families_gpu.py: {sorted(gemm - covered)}"
    assert set(families.GEMM_KERNELS) == gemm, f"the GPU file's kernel list is stale: {set(families.GEMM_KERNELS) ^ gemm}"
    assert covered - gemm <= set(families.UTILITY_KERNELS), f"cases name unknown kernels: {covered - gemm}"


def test_profiler_names_map_to_source_names():
    """The profiler reports demangled (or, without a demangler, mangled) names; both map to the qualified source name."""
    q = families._qualified
    assert q("void crf::lin2::dgrad2_kernel<128, true, false>(crf::lin::DgradArgs, int)") == "lin2::dgrad2_kernel"
    assert q("void crf::lin::sm::fwd_small_kernel<64>(crf::lin::FwdArgs)") == "lin::sm::fwd_small_kernel"
    assert q("_ZN3crf3lin2dw19wgrad_direct_kernelILi1ELi1EEEvNS0_9WgradArgsE") == "lin::dw::wgrad_direct_kernel"
    assert q("void at::native::vectorized_elementwise_kernel<4>(int)") is None
