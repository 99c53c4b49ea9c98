"""Every ``__global__`` instantiation in ``libb200fe.so`` is claimed by a case of the kernel-coverage table
(``tests/kernel_cases.py``, run on the GPU by ``tests/test_gpu_kernel_coverage.py``) or by an allowlist entry naming
the existing test that runs it.  A new template instantiation without a case fails here, on a machine without a GPU.
The table's own claims that can be checked on the host (resolved variant, FFT tile width, the generic tail's size
limit) are checked here too."""
import ast
import os
import shutil
import subprocess

import pytest

from helpers import ROOT
from kernel_cases import ALLOWLIST, CASES, claims, fft_pick_ft, generic_tail_smem_bytes, kernel_name, make_engine

LIB = os.path.join(ROOT, "audio-deepfake-detection-fmsl_b200", "lib", "libb200fe.so")


def _library_kernels():
    if shutil.which("cuobjdump") is None and not os.path.exists("/usr/local/cuda/bin/cuobjdump"):
        pytest.skip("cuobjdump not found")
    if shutil.which("c++filt") is None:
        pytest.skip("c++filt not found")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    elf = subprocess.run([cuobjdump, "-elf", LIB], capture_output=True, text=True, check=True).stdout
    mangled = sorted({tok[len(".text."):] for tok in elf.split() if tok.startswith(".text._Z")})
    assert mangled, "no kernel symbols found in " + LIB
    demangled = subprocess.run(["c++filt"], input="\n".join(mangled), capture_output=True, text=True,
                               check=True).stdout.splitlines()
    return sorted({kernel_name(d) for d in demangled})


def test_every_kernel_instantiation_is_claimed():
    kernels = _library_kernels()
    assert len(kernels) >= 60, kernels
    patterns = [p for c in CASES for p in c.kernels]
    unclaimed = [k for k in kernels if k not in ALLOWLIST and not any(claims(p, k) for p in patterns)]
    assert not unclaimed, f"kernel instantiations without a coverage case or allowlist entry: {unclaimed}"
    # every pattern of the table names a kernel that exists (a renamed kernel must not leave a dead case behind)
    dead = sorted({p for p in patterns if not any(claims(p, k) for k in kernels)})
    assert not dead, f"coverage cases name kernels the library does not have: {dead}"
    assert set(ALLOWLIST) <= set(kernels)


def test_allowlist_names_existing_tests():
    for kernel, ref in ALLOWLIST.items():
        module, name = ref.split("::")
        with open(os.path.join(ROOT, "tests", module + ".py")) as fh:
            tree = ast.parse(fh.read())
        names = {n.name for n in ast.walk(tree) if isinstance(n, ast.FunctionDef)}
        assert name in names, f"{kernel}: {ref} does not exist"


def test_case_ids_are_unique():
    ids = [c.id for c in CASES]
    assert len(ids) == len(set(ids))


@pytest.mark.parametrize("case", [c for c in CASES if c.kind != "deltas"], ids=lambda c: c.id)
def test_case_configuration_packs_and_resolves(fe, case):
    """Every case's tables pack, and AUTO (or the case's explicit request) resolves to the variant it names."""
    eng = make_engine(fe, case)
    assert eng.resolved_variant() == case.variant
    if case.request == "auto" and case.variant == "fft" and case.kind != "spectrogram":
        with pytest.raises(NotImplementedError):   # AUTO took the FFT variant because the tensor cores refuse it
            make_engine(fe, case, request="dft_gemm")
    if case.ft:
        mode = 0 if case.kind == "spectrogram" else 1
        n_ch = case.n_fft // 2 + 1 if mode == 0 else case.n_filter
        assert fft_pick_ft(case.n_fft, case.hop, n_ch, mode) == case.ft


def test_generic_tail_limit_cases_straddle_the_check():
    by_id = {c.id: c for c in CASES}
    ok, rejected = by_id["generic_largest"], by_id["generic_rejected"]
    nF = 1 + ok.T // ok.hop
    assert generic_tail_smem_bytes(ok.n_filter, ok.n_coef, ok.deltas, ok.delta_win, nF) <= 200 * 1024
    assert generic_tail_smem_bytes(rejected.n_filter, rejected.n_coef, rejected.deltas, rejected.delta_win,
                                   nF) > 200 * 1024
    assert rejected.n_filter == ok.n_filter + 1
