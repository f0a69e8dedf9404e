import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


# the CPU oracle runs small ops: dozens of OpenMP threads only add spin-wait overhead, and the GPU box reports
# 128 logical CPUs while its cgroup grants 16 (cpu.max)
def _usable_cpus():
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


torch.set_num_threads(max(1, min(16, _usable_cpus())))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "ref: needs the live reference tree at /root/reference (build container)")


def pytest_collection_modifyitems(config, items):
    has_gpu = torch.cuda.is_available()
    from oracle import ref_shims
    has_ref = ref_shims.reference_available()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "ref" in item.keywords and not has_ref:
            item.add_marker(pytest.mark.skip(reason="reference tree not present"))


def load_golden(name):
    """Fixture arrays by name; a uniform(-0.5, 0.5) input stored as `key/seed` + `key/shape` (oracle/gen_golden.py:
    seeded_input) comes back regenerated under `key`."""
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    out = {k: (torch.from_numpy(z[k]) if z[k].dtype.kind == "f" else z[k]) for k in z.files}
    for k in [k[:-len("/seed")] for k in z.files if k.endswith("/seed")]:
        g = torch.Generator().manual_seed(int(z[k + "/seed"]))
        out[k] = torch.rand(tuple(int(s) for s in z[k + "/shape"]), generator=g) - 0.5
    return out


def assert_golden_close(got, z, key, rel, floor):
    """||got - golden|| <= rel * ||golden|| + floor * sqrt(numel) over the elements the fixture stores for `key`: the whole
    tensor, or the seeded sample of a large one (oracle/gen_golden.py:store_sampled), whose whole-tensor norm must then
    lie within the same bound of the stored norm."""
    got = got.detach().cpu().double()
    if key in z:
        ref = z[key].double()
    else:
        norm = float(z[key + "/norm"])
        bound = rel * norm + floor * got.numel() ** 0.5
        assert abs(float(got.norm()) - norm) <= bound, (key, float(got.norm()), norm)
        got, ref = got.reshape(-1)[torch.from_numpy(z[key + "/idx"]).long()], z[key + "/samp"].double()
    err = float((got - ref).norm())
    assert err <= rel * float(ref.norm()) + floor * ref.numel() ** 0.5, (key, err)


@pytest.fixture
def golden():
    return load_golden


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


# ---------------------------------------------------------------------------------------------------------------
# host emulation of the plain SIMT kernels (tests/emu/): the product's .cu sources compiled with g++ -DPN_EMULATE
# ---------------------------------------------------------------------------------------------------------------
EMU_DIR = os.path.join(ROOT, "tests", "emu")
EMU_SO = os.path.join(EMU_DIR, "_build", "libpacknet_emu.so")


def _emu_sources():
    csrc = os.path.join(ROOT, "packnet_sfm_b200", "csrc")
    return [os.path.join(EMU_DIR, "emu_kernels.cpp"), os.path.join(EMU_DIR, "cuda_emu.h"),
            os.path.join(ROOT, "include", "packnet_b200.h")] + \
           [os.path.join(csrc, f) for f in ("common.cuh", "fold_kernels.cu", "frame_kernels.cu", "layer_kernels.cu", "loss_kernels.cu", "loss_group_kernel.cuh", "pack_kernels.cu", "optim_kernels.cu")]


@pytest.fixture(scope="session")
def emu_lib():
    """libpacknet_emu.so: fold / frame / layer / loss kernels from their real source, built for the host
    (-ffp-contract=off: every float operation rounds once, as the __f*_rn chains of the loss kernel require)."""
    import ctypes
    import subprocess
    from packnet_sfm_b200 import _lib, _lib_conv
    src = _emu_sources()
    os.makedirs(os.path.dirname(EMU_SO), exist_ok=True)
    if not os.path.exists(EMU_SO) or any(os.path.getmtime(f) > os.path.getmtime(EMU_SO) for f in src):
        cmd = ["g++", "-std=c++20", "-O1", "-ffp-contract=off", "-shared", "-fPIC", "-pthread", "-DPN_EMULATE", "-x", "c++",
               "-Wno-unknown-pragmas", "-I", EMU_DIR, "-I", os.path.join(ROOT, "include"),
               "-I", os.path.join(ROOT, "packnet_sfm_b200", "csrc"), src[0], "-o", EMU_SO]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 0, r.stdout
    lib = ctypes.CDLL(EMU_SO)
    _lib._declare(lib)
    _lib_conv.declare(lib)
    return lib


@pytest.fixture
def emulated_kernels(emu_lib, monkeypatch):
    """Route the product's Python layer (packnet_sfm_b200._lib) to the emulated library; CPU tensors pass as device memory."""
    from packnet_sfm_b200 import _lib, folded
    monkeypatch.setattr(_lib, "lib", lambda: emu_lib)
    monkeypatch.setattr(_lib, "require_cuda", lambda *a: None)
    monkeypatch.setattr(_lib, "current_stream", lambda: None)
    monkeypatch.setattr(folded, "_use_kernels", lambda t: True)
    return emu_lib
