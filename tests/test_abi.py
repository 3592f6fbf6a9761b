"""No-GPU checks of the drop-in boundary: the C-ABI library loads, exports every symbol include/afcrypto.h
declares, refuses to run without a device (no CPU fallback), and the product never touches oracle/."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "afcrypto.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(afc_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from agentfield_b200 import _abi
    lib = _abi.load()
    names = _declared()
    assert len(names) >= 38
    for n in names:
        assert hasattr(lib, n), "libafcrypto.so does not export %s" % n
    assert set(names) == set(_abi.SYMBOLS), "ctypes table and header disagree: %s" % (set(names) ^ set(_abi.SYMBOLS))
    assert b"sm_100a" in lib.afc_version()
    assert lib.afc_strerror(-2).startswith(b"CUDA")


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the refusal path needs a CPU-only box")
    import agentfield_b200 as afb
    with pytest.raises(afb.AfcError) as ei:
        afb.Context(0)
    assert ei.value.rc == afb._abi.AFC_ECUDA
    lib = afb._abi.load()
    out = (C.c_uint8 * 32)()
    off = (C.c_uint64 * 2)(0, 0)
    assert lib.afc_sha256_batch(None, None, off, 1, out) == afb._abi.AFC_EINVAL     # NULL ctx: nothing computes


def test_product_never_imports_or_links_the_oracle():
    """The oracle is test infrastructure: nothing under agentfield_b200/ may import, include or link it (or the CPU build of
    the kernel logic under tests/hostsim), and the shared object must carry no oracle / OpenSSL code."""
    import subprocess
    pkg = os.path.join(ROOT, "agentfield_b200")
    pat = re.compile(r"^\s*(from|import)\s+oracle\b|^\s*from\s+\.\.?oracle\b|#include\s*[\"<][^\">]*oracle|c_oracle|libafc_oracle|libafc_hostsim|libafc_openssl")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".inc")) or f == "Makefile":
                for ln in open(os.path.join(d, f), errors="ignore"):
                    assert not pat.search(ln), (os.path.join(d, f), ln.strip())
    so = os.path.join(pkg, "libafcrypto.so")
    syms = subprocess.check_output(["nm", "-D", so]).decode()
    assert "afo_" not in syms and "afx_" not in syms and "EVP_" not in syms and "hs_verify" not in syms
    ldd = subprocess.check_output(["ldd", so]).decode()
    assert "libcrypto" not in ldd and "libafc_oracle" not in ldd


def test_kernels_are_sm100a_sass():
    import shutil
    import subprocess
    so = os.path.join(ROOT, "agentfield_b200", "libafcrypto.so")
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    out = subprocess.check_output([cuobjdump, "-lelf", so]).decode()
    assert "sm_100a" in out and "sm_90" not in out and "sm_80" not in out


def _build_c_harness():
    import subprocess
    d = os.path.join(ROOT, "tests", "c_abi")
    subprocess.check_call(["make", "-s", "-C", d])
    return os.path.join(d, "harness")


def test_plain_c_caller_compiles_and_fails_loudly_without_a_gpu():
    """tests/c_abi/harness.c is what a cgo binding amounts to: a C99 translation unit that sees only include/afcrypto.h and links
    libafcrypto.so.  It must build with -Wall -Wextra -pedantic, and on a box without a GPU report AFC_ECUDA (exit code 77) instead
    of computing anything on the CPU."""
    import subprocess
    import torch
    exe = _build_c_harness()
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the harness is run by the gpu-marked test")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 77 and "no CPU path" in r.stdout, (r.returncode, r.stdout, r.stderr)


@pytest.mark.gpu
def test_plain_c_caller_passes_its_known_answer_checks():
    """The same program on the GPU box: RFC 8032 TEST 1-3 (sign, public key, verify, a corrupted signature reported as ok = 0),
    RFC 4231 case 2, SHA-256 one-shot and streaming, the first Certificate-Transparency roots — through the C ABI from C."""
    import subprocess
    r = subprocess.run([_build_c_harness()], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "c_abi harness ok" in r.stdout, (r.returncode, r.stdout, r.stderr)
