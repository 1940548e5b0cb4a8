"""The C-ABI shared library: it loads, exports every symbol the headers in include/ declare, reports its ABI
version, and refuses to run without a CUDA device (no CPU fallback).  No GPU needed."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest
import torch

import coverm_b200
from case_runner import ROOT


def _build_nvcc():
    """The nvcc coverm_b200/csrc/Makefile compiles with: $NVCC, else the Makefile's default."""
    mk = open(os.path.join(ROOT, "coverm_b200", "csrc", "Makefile")).read()
    nvcc = os.environ.get("NVCC") or re.search(r"^NVCC \?= *(\S+)", mk, re.M).group(1)
    return shutil.which(nvcc) or nvcc


# the toolkit that built the library disassembles it
CUOBJDUMP = os.path.join(os.path.dirname(_build_nvcc()), "cuobjdump")


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(coverm_b200.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return coverm_b200.load_library()


def declared_functions(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cmbh?_[a-z_0-9]+)\s*\(", text)))


def test_exports_every_declared_symbol(lib):
    names = declared_functions("coverm_b200.h") + declared_functions("coverm_b200_host.h")
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/ but not exported by libcoverm_b200.so"
    assert set(coverm_b200.DEVICE_SYMBOLS + coverm_b200.HOST_SYMBOLS) == set(names)


def test_abi_version_and_struct_sizes(lib):
    assert lib.cmb_abi_version() == 3
    assert ctypes.sizeof(coverm_b200.ContigStats) == 144
    assert ctypes.sizeof(coverm_b200.Params) == 56
    assert ctypes.sizeof(coverm_b200.ReadBatch) == 8 + 13 * 8


def test_kernels_are_sm_100a_with_tma(lib):
    out = subprocess.run([CUOBJDUMP, "-sass", coverm_b200.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "UTMALDG" in out, "K2 must stage its tiles with TMA (cp.async.bulk.tensor)"
    for k in ("k1_filter_accumulate", "k1b_local", "k1b_apply", "k2_scan_reduce", "k3_finalize", "kd_inflate", "kd_inflate_g8", "kd_guess", "kd_walk",
              "kd_extract"):
        assert k in out


# any visible CUDA device: its device node need not be /dev/nvidia0
@pytest.mark.skipif(torch.cuda.is_available(), reason="a CUDA device is visible")
def test_fails_loudly_without_a_gpu(lib):
    h = ctypes.c_void_p()
    cfg = coverm_b200.DeviceCfg(0, 1024, 2048, 2)
    rc = lib.cmb_create(ctypes.byref(cfg), ctypes.byref(h))
    assert rc != 0 and not h.value
    assert b"no CPU fallback" in lib.cmb_last_error(None)
    p = subprocess.run([coverm_b200.COVERM_BIN, "contig", "-b", os.path.join(ROOT, "tests/golden/data/tpm_test.bam")],
                       capture_output=True, text=True)
    assert p.returncode != 0 and "CUDA" in p.stderr


def test_product_does_not_link_the_oracle():
    """libcoverm_b200.so / coverm must not contain anything from oracle/ (the device emulator is test-only)."""
    mk = open(os.path.join(ROOT, "coverm_b200", "csrc", "Makefile")).read()
    assert "oracle" not in mk
    for root, _, files in os.walk(os.path.join(ROOT, "coverm_b200", "csrc")):
        for f in files:
            if f.endswith((".cu", ".cpp", ".hpp", ".h")):
                assert "oracle/" not in open(os.path.join(root, f)).read(), f
