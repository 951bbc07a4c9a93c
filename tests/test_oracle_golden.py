"""The oracle restatement (oracle/w2l_oracle.py) against the committed outputs of the REAL
reference modules (tests/golden/*.npz, made by tests/golden/make_golden.py)."""
import os

import numpy as np
import torch

from oracle import w2l_oracle as O

TOL = 2e-5  # fp32 CPU conv summation-order noise between runs/threads; values are O(1..30)


def _fp(t):
    f = t.detach().double().flatten()
    return np.concatenate([[f.sum().item(), f.abs().sum().item(), f.abs().max().item()],
                           f[:32].numpy(), f[-32:].numpy()])


def _check_fp(name, got, want):
    scale = max(1.0, abs(want[1]))
    assert abs(got[0] - want[0]) <= 1e-5 * scale, name
    assert abs(got[1] - want[1]) <= 1e-5 * scale, name
    np.testing.assert_allclose(got[3:], want[3:], rtol=1e-4, atol=1e-4, err_msg=name)


def test_macs_match_survey():
    assert O.macs_per_unit("generator") == 3966984192
    assert O.macs_per_unit("syncnet") == 1210281984
    assert O.macs_per_unit("disc") == 1255850496


def test_generator_oracle_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "generator.npz"))
    sd = O.make_state_dict("generator", 0)
    assert len(sd) == 352
    chk = sum(v.double().abs().sum().item() for v in sd.values() if v.dtype.is_floating_point)
    assert abs(chk - float(g["gen_sd_checksum"])) <= 1e-9 * chk, "seeded weights drifted (torch RNG changed?)"
    mel, face = O.make_generator_inputs(2, 0)
    np.testing.assert_allclose([mel.double().abs().sum().item(), face.double().abs().sum().item()],
                               g["gen4_in_checksum"], rtol=1e-12)
    taps = {}
    with torch.no_grad():
        logits = O.generator_forward(sd, mel, face, taps, return_logits=True)
    np.testing.assert_allclose(logits.numpy(), g["gen4_logits"], atol=2e-4, rtol=0)
    np.testing.assert_allclose(torch.sigmoid(logits).numpy(), g["gen4_out"], atol=TOL, rtol=0)
    for name, _ in O.generator_layers():
        _check_fp(name, _fp(taps[name]), g["gen4_fp/" + name])


def test_generator_oracle_5d_and_odd_batch(golden_dir):
    g = np.load(os.path.join(golden_dir, "generator.npz"))
    sd = O.make_state_dict("generator", 0)
    mel5, face5 = O.make_generator_inputs(2, seed=1, t=5)
    with torch.no_grad():
        y5 = O.generator_forward(sd, mel5, face5)
    assert tuple(y5.shape) == (2, 3, 5, 96, 96)
    np.testing.assert_allclose(y5.numpy(), g["gen5_out"], atol=TOL, rtol=0)
    mel3, face3 = O.make_generator_inputs(3, seed=2)
    with torch.no_grad():
        y3 = O.generator_forward(sd, mel3, face3)
    np.testing.assert_allclose(y3.numpy(), g["gen4n3_out"], atol=TOL, rtol=0)


def test_syncnet_oracle_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "syncnet.npz"))
    sd = O.make_state_dict("syncnet", 0)
    mel, face = O.make_syncnet_inputs(3, 0)
    taps = {}
    with torch.no_grad():
        a, v = O.syncnet_forward(sd, mel, face, taps)
    np.testing.assert_allclose(a.numpy(), g["sync_a"], atol=TOL, rtol=0)
    np.testing.assert_allclose(v.numpy(), g["sync_v"], atol=TOL, rtol=0)
    np.testing.assert_allclose(a.norm(dim=1).numpy(), 1.0, atol=1e-5)
    for name, _ in O.syncnet_layers():
        _check_fp(name, _fp(taps[name]), g["sync_fp/" + name])


def test_disc_oracle_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "disc.npz"))
    sd = O.make_state_dict("disc", 0)
    frames = O.make_disc_inputs(2, 5, 0)
    taps = {}
    with torch.no_grad():
        lo = O.disc_forward(sd, frames, taps, return_logits=True)
    assert tuple(lo.shape) == (10, 1)
    np.testing.assert_allclose(lo.numpy(), g["disc_logits"], atol=2e-4, rtol=1e-4)
    np.testing.assert_allclose(torch.sigmoid(lo).numpy(), g["disc_out"], atol=TOL, rtol=0)
    for name, _ in O.disc_layers():
        _check_fp(name, _fp(taps[name]), g["disc_fp/" + name])


def test_oracle_vs_live_reference(golden_dir):
    """A second weight and input seed against the full outputs of the reference modules
    (tests/golden/reference_seed3.npz, made by make_golden.py)."""
    g = np.load(os.path.join(golden_dir, "reference_seed3.npz"))
    sd = O.make_state_dict("generator", 3)
    chk = sum(v.double().abs().sum().item() for v in sd.values() if v.dtype.is_floating_point)
    assert abs(chk - float(g["gen_sd_checksum"])) <= 1e-9 * chk, "seeded weights drifted (torch RNG changed?)"
    mel, face = O.make_generator_inputs(1, 5)
    np.testing.assert_allclose([mel.double().abs().sum().item(), face.double().abs().sum().item()],
                               g["gen_in_checksum"], rtol=1e-12)
    with torch.no_grad():
        np.testing.assert_allclose(O.generator_forward(sd, mel, face).numpy(), g["gen_out"], atol=TOL)
    sd = O.make_state_dict("syncnet", 3)
    mel, face = O.make_syncnet_inputs(2, 5)
    with torch.no_grad():
        a1, v1 = O.syncnet_forward(sd, mel, face)
    np.testing.assert_allclose(a1.numpy(), g["sync_a"], atol=TOL)
    np.testing.assert_allclose(v1.numpy(), g["sync_v"], atol=TOL)
    sd = O.make_state_dict("disc", 3)
    fr = O.make_disc_inputs(1, 5, 5)
    with torch.no_grad():
        np.testing.assert_allclose(O.disc_forward(sd, fr).numpy(), g["disc_out"], atol=TOL)
