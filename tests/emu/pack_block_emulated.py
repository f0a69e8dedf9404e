"""PackLayerConv3d (networks.py) with the FOLDED path, forward and backward, on the CPU: fold / frame / GroupNorm+ELU kernels
from their real source under the host emulation, PyTorch's conv2d (with autograd) in place of the tcgen05 engine, against
the golden vectors the live reference produced for the block (tests/golden/blocks.npz: output, input gradient and all six
parameter gradients).  TEST INFRASTRUCTURE; not collected by pytest (minutes of CPU: the fold kernels' shuffle reductions
are slow to emulate):   python tests/emu/pack_block_emulated.py"""
import ctypes, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch
import torch.nn.functional as F
from conftest import assert_golden_close, load_golden, rel_l2
from oracle import packnet_oracle as PO
from packnet_sfm_b200 import _lib, _lib_conv, folded, functional as PF

lib = ctypes.CDLL(os.path.join(ROOT, 'tests', 'emu', '_build', 'libpacknet_emu.so'))
_lib._declare(lib); _lib_conv.declare(lib)
_lib.lib = lambda: lib; _lib.require_cuda = lambda *a: None; _lib.current_stream = lambda: None
folded._use_kernels = lambda t: True
PF.conv2d = lambda x, w, b=None: F.conv2d(x.permute(0, 3, 1, 2), w, b, padding=w.shape[-1] // 2).permute(0, 2, 3, 1).contiguous()
from packnet_sfm_b200 import networks as N   # noqa: E402

PF.set_pack_fold(True, min_pixels=0)
z = load_golden("blocks")
for tag, cin, k, seed in (("pack_k5", 16, 5, 22), ("pack_k3", 32, 3, 21)):
    t0 = time.time()
    mod = N.PackLayerConv3d(cin, k)
    mod.load_state_dict(PO.block_state_dict("pack", cin, k=k, seed=seed), strict=True)
    x = z[tag + "_x"].permute(0, 2, 3, 1).contiguous().requires_grad_(True)
    y = mod(x)
    y.backward(z[tag + "_gy"].permute(0, 2, 3, 1).contiguous())
    ey = rel_l2(y.permute(0, 3, 1, 2), z[tag + "_y"])
    ex = rel_l2(x.grad.permute(0, 3, 1, 2), z[tag + "_gx"])
    print("%s: y %.2e  gx %.2e  (%.0f s)" % (tag, ey, ex, time.time() - t0), flush=True)
    assert ey < 1e-5 and ex < 1e-4
    for name, p in mod.named_parameters():
        # same criterion as tests/test_layers_gpu.py: the convolution bias in front of a GroupNorm has a gradient that is
        # zero up to cancellation (|g| ~ 1e-6), hence the absolute floor
        assert_golden_close(p.grad, z, tag + "_g_" + name, 1e-3, 5e-5)
        print("   g %-24s ok" % name, flush=True)
print("ok")
