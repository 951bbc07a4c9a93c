"""Scope row f4 (S3FD face detector), CPU part: the restatement oracle/s3fd_oracle.py against vectors produced by the REAL
reference modules (tests/golden/s3fd.npz, s3fd_seed3.npz <- tests/golden/make_golden_s3fd.py), and the product's
host-side post-processing (wav2lip_b200/face_detection/detection/sfd/sfd_detector.py: vectorised NumPy) against the
reference's own candidate array and NMS keep lists."""
import os

import numpy as np
import pytest
import torch

from oracle import s3fd_oracle as S


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "s3fd.npz"))


def test_oracle_network_matches_reference_golden(gold):
    sd = S.make_state_dict(0)
    with torch.no_grad():
        olist = S.forward(sd, S.preprocess(S.make_images(2, 96, 128, seed=1)))
    assert len(olist) == 12
    for i, o in enumerate(olist):
        ref = gold[f"o{i}"]
        assert tuple(o.shape) == ref.shape
        assert np.abs(o.numpy() - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max()), i
    with torch.no_grad():
        o2 = S.forward(sd, S.preprocess(S.make_images(1, 150, 210, seed=2)))
    assert [list(o.shape) for o in o2] == gold["big_shapes"].tolist()       # odd sizes: floor pools, fc6 (+4), stride-2 tails
    for i, o in enumerate(o2):
        f = o.double().flatten()
        assert abs(f.abs().sum().item() - gold["big_fp"][i][1]) <= 1e-4 * gold["big_fp"][i][1]


def test_oracle_candidates_and_nms_match_reference_golden(gold):
    olist = [torch.from_numpy(gold[f"o{i}"]) for i in range(12)]
    cand = S.batch_candidates(olist)
    assert cand.shape == gold["candidates"].shape
    np.testing.assert_allclose(cand, gold["candidates"], rtol=1e-5, atol=1e-4)
    for i in range(cand.shape[1]):
        assert np.array_equal(np.array(S.nms(gold["candidates"][:, i, :], 0.3)), gold[f"keep{i}"])


def test_product_postprocessing_matches_reference_golden(gold):
    """decode_candidates / nms of the product's detector are host-side NumPy: checked here without a GPU."""
    from wav2lip_b200.face_detection.detection.sfd import sfd_detector as D
    cand = D.decode_candidates([gold[f"o{i}"] for i in range(12)])
    assert cand.shape == gold["candidates"].shape
    np.testing.assert_allclose(cand, gold["candidates"], rtol=1e-5, atol=1e-3)
    for i in range(cand.shape[1]):
        assert np.array_equal(np.array(D.nms(gold["candidates"][:, i, :], 0.3)), gold[f"keep{i}"])
    # no hit anywhere -> the reference's (1, B, 5) zero array
    quiet = [np.zeros_like(gold[f"o{i}"]) for i in range(12)]
    for i in range(6):
        quiet[2 * i][:, 0] = 10.0
    assert D.decode_candidates(quiet).shape == (1, 2, 5)


def test_mirror_state_dict_is_the_references():
    from wav2lip_b200.face_detection.detection.sfd.net_s3fd import s3fd
    m = s3fd()
    sd = S.make_state_dict(0)
    assert list(m.state_dict().keys()) == list(sd.keys())
    m.load_state_dict(sd, strict=True)
    with pytest.raises(Exception):
        m(torch.zeros(1, 3, 64, 64))          # CPU tensor: no fallback


def test_oracle_against_live_reference(golden_dir):
    """A second weight seed and frame size against the reference module's 12 output maps
    (tests/golden/s3fd_seed3.npz, made by make_golden_s3fd.py)."""
    g = np.load(os.path.join(golden_dir, "s3fd_seed3.npz"))
    sd = S.make_state_dict(3)
    imgs = S.make_images(1, 70, 90, seed=5)
    with torch.no_grad():
        b = S.forward(sd, S.preprocess(imgs))
    assert len(b) == 12
    for i, y in enumerate(b):
        x = torch.from_numpy(g[f"o{i}"])
        assert x.shape == y.shape, i
        assert torch.allclose(x, y, rtol=1e-4, atol=1e-5), i
