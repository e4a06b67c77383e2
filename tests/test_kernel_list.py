"""The kernels compiled into libcapycrypt_gpu.so are exactly the ones tests/test_dispatch_matrix_gpu.py lists in KERNELS.

That file runs every kernel of KERNELS under a bit-exact oracle check; this test makes sure the list stays complete, so a
new kernel or template instantiation cannot land without a row in that matrix.  No GPU needed: the kernel names come from
the ELF sections of the device code (cuobjdump), demangled with cu++filt.
"""
import importlib.util
import os
import re
import shutil
import subprocess

import pytest

from capycrypt_b200 import _binding

HERE = os.path.dirname(os.path.abspath(__file__))


def _matrix():
    spec = importlib.util.spec_from_file_location("dispatch_matrix", os.path.join(HERE, "test_dispatch_matrix_gpu.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _cuda_tool(name):
    """a CUDA binary tool: on PATH, next to the nvcc the build uses, or under CUDA_HOME"""
    nvcc = shutil.which(os.environ.get("NVCC", "nvcc"))
    for p in (shutil.which(name), nvcc and os.path.join(os.path.dirname(nvcc), name),
              os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", name)):
        if p and os.path.exists(p):
            return p
    pytest.fail(f"{name} not found (it ships with the CUDA toolkit that builds the library)")


def compiled_kernels(lib_path):
    elf = subprocess.run([_cuda_tool("cuobjdump"), "-elf", lib_path], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(re.findall(r"\.text\.([A-Za-z_$][\w$]*)", elf)))
    assert mangled, "no device code sections in the library"
    out = subprocess.run([_cuda_tool("cu++filt")], input="\n".join(mangled) + "\n", capture_output=True, text=True,
                         check=True).stdout
    return out.split("\n")[:len(mangled)]


def test_normalise_kernel_names():
    m = _matrix()
    assert m.normalise_kernel("void capy::sha3_short_kernel<(int)17, (int)2>(const uint4 *, unsigned long)") == \
        "sha3_short_kernel<17,2>"
    assert m.normalise_kernel("void capy::sponge_tiered_kernel<19>(capy::SpongeJob, capy::SpongeTiers)") == \
        "sponge_tiered_kernel<19>"
    assert m.normalise_kernel("capy::len_scan_kernel(unsigned int *, unsigned int *)") == "len_scan_kernel"


def test_library_kernels_equal_the_matrix_list():
    assert os.path.exists(_binding.LIB_PATH), "build the library first (python -m capycrypt_b200.build)"
    m = _matrix()
    got = {m.normalise_kernel(k) for k in compiled_kernels(_binding.LIB_PATH)}
    assert len(m.KERNELS) == 53
    assert not got - m.KERNELS, f"kernels without a row in the dispatch matrix: {sorted(got - m.KERNELS)}"
    assert not m.KERNELS - got, f"KERNELS names kernels the library does not have: {sorted(m.KERNELS - got)}"
