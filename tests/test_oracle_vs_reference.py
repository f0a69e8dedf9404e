"""CPU: the oracle restatement against what the unmodified reference's own module and loss class computed
(oracle/gen_golden.py: restatement_case, loss_restatement_case)."""
import torch

from conftest import load_golden


def test_packnet01_restatement_matches_reference_module():
    """Same parameter names, order and shapes as the reference's PackNet01, and its depth maps for the same weights.  The
    oracle runs the reference's ops in the reference's order, so with the CPU convolution kernels that produced the fixture
    the maps are bit-identical; a host whose oneDNN picks other kernels (AVX2 instead of AVX-512) sums in another order,
    which moves them by up to 4e-5 relative."""
    from oracle import packnet_oracle as PO
    z = load_golden("packnet01_restatement_64x96")
    sd = PO.packnet01_state_dict()
    assert list(sd) == list(z["keys"])
    assert all(tuple(sd[k].shape) == tuple(int(s) for s in z["shape/" + k]) for k in sd)
    with torch.no_grad():
        mine = PO.packnet01_forward(z["rgb"], sd)
    for i, a in enumerate(mine):
        b = z["disp%d" % (i + 1)]
        assert a.shape == b.shape
        assert float(((a - b).abs() / b.abs()).max()) < 1e-4, i


def test_loss_restatement_matches_reference_class():
    """Same ops in the same order as the reference's MultiViewPhotometricLoss: bit-identical on the host that produced the
    fixture; 1e-6 leaves room for another host's CPU kernels (as tests/test_oracle_golden.py)."""
    from oracle import loss_oracle as LO
    z = load_golden("loss_restatement_2x24x48")
    inv = [z["inv%d" % i] for i in range(4)]
    out = LO.multiview_photometric_loss(z["rgb"], [z["ctx0"], z["ctx1"]], inv, z["K"], z["K"], [z["pose0"], z["pose1"]])
    assert abs(float(out["loss"]) - float(z["loss"])) <= 1e-6 * abs(float(z["loss"]))
