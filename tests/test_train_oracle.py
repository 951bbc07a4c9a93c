"""Pins oracle/train_oracle.py (the restatement of one wav2lip_train.py / color_syncnet_train.py optimisation step —
oracle for the NEXT scope row, no product code behind it yet) against tests/golden/train.npz, which was produced by the
REAL reference modules + torch.optim.Adam (tests/golden/make_golden_train.py).  Same torch build, same CPU ops, same
thread count: agreement is to rounding (different autograd graph shapes reorder a few fp32 sums)."""
import os

import numpy as np
import pytest
import torch

from oracle import train_oracle as T
from oracle import w2l_oracle as O

GOLDEN_THREADS = 8  # tests/golden/make_golden_train.py


def fp3(t):
    f = t.detach().double().flatten()
    return np.array([f.sum().item(), f.abs().sum().item(), f.abs().max().item()])


def close(a, b, rel):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.all(np.abs(a - b) <= rel * np.maximum(np.abs(b), 1e-12) + 1e-12)


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "train.npz"))


@pytest.fixture(autouse=True)
def golden_threads():
    """torch's CPU ops split their sums by thread, and the expert's train-mode BatchNorm over two windows followed by
    Adam amplifies a different rounding far past these tolerances: run with the thread count train.npz was made with."""
    old = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(old)


def _train_inputs(B, seed):
    g = torch.Generator().manual_seed(seed)
    indiv_mels, x = O.make_generator_inputs(B, seed=seed, t=5)
    mel = torch.rand((B, 1, 80, 16), generator=g) * 8 - 4
    gt = torch.rand((B, 3, 5, 96, 96), generator=g)
    return x, indiv_mels, mel, gt


def test_generator_training_step_matches_reference(gold):
    gen_sd = O.make_state_dict("generator", 0, init="default")
    sync_sd = O.make_state_dict("syncnet", 1, init="default")
    x, indiv_mels, mel, gt = _train_inputs(2, seed=7)
    state = None
    for step in range(2):
        r = T.wav2lip_train_step(gen_sd, sync_sd, x, indiv_mels, mel, gt, syncnet_wt=0.03, lr=1e-4, state=state)
        state = r["state"]
        losses = np.array([r["loss"].item(), r["sync_loss"].item(), r["l1"].item()])
        assert close(losses, gold[f"gen{step}_losses"], 1e-5), (step, losses, gold[f"gen{step}_losses"])
        assert close(fp3(r["g"]), gold[f"gen{step}_g_fp"], 1e-5)
        names = list(gold[f"gen{step}_grad_names"])
        assert names == list(r["grads"].keys())                     # same parameter set and order as named_parameters()
        got = np.stack([fp3(r["grads"][n]) for n in names])
        ref = gold[f"gen{step}_grad_fp"]
        # abs-sum and max-abs of every gradient tensor to 1e-3 relative (sums of ~1e6 fp32 terms, order differs);
        # the plain sum cancels and is compared against the abs-sum scale
        assert close(got[:, 1], ref[:, 1], 1e-3), np.abs(got[:, 1] / ref[:, 1] - 1).max()
        assert close(got[:, 2], ref[:, 2], 1e-3)
        assert np.all(np.abs(got[:, 0] - ref[:, 0]) <= 1e-3 * ref[:, 1] + 1e-12)
        assert np.allclose(r["grads"]["output_block.1.weight"].flatten().numpy(), gold[f"gen{step}_grad_head_w"], rtol=1e-3, atol=1e-7)
        assert np.allclose(r["grads"]["face_encoder_blocks.0.0.conv_block.0.weight"].flatten()[:64].numpy(),
                           gold[f"gen{step}_grad_first_w"], rtol=2e-3, atol=1e-7)
        assert np.allclose(r["grads"]["face_decoder_blocks.6.0.conv_block.0.weight"].flatten()[:64].numpy(),
                           gold[f"gen{step}_grad_dec60_w"], rtol=2e-3, atol=1e-7)
        # post-step state: parameters moved by Adam (|delta| = lr on the first step), BatchNorm buffers by the forward
        sd_names = list(gold[f"gen{step}_sd_names"])
        assert sd_names == list(gen_sd.keys())
        got_sd = np.stack([fp3(gen_sd[n]) for n in sd_names])
        assert close(got_sd[:, 1], gold[f"gen{step}_sd_fp"][:, 1], 1e-5)
        assert close(got_sd[:, 2], gold[f"gen{step}_sd_fp"][:, 2], 1e-5)
        exp = np.stack([fp3(v) for k, v in sync_sd.items() if "running" in k or "num_batches" in k])
        assert close(exp[:, 1], gold[f"gen{step}_expert_buf_fp"][:, 1], 1e-5)   # the expert's BN buffers move too (train mode)


def test_first_adam_step_moves_every_weight_by_lr(gold):
    """Sanity of the Adam restatement: after step 1, |delta| == lr * |g| / (|g| + eps*sqrt(1-b2)) ~ lr wherever g != 0."""
    gen_sd = O.make_state_dict("generator", 0, init="default")
    before = {k: v.clone() for k, v in gen_sd.items()}
    sync_sd = O.make_state_dict("syncnet", 1, init="default")
    x, indiv_mels, mel, gt = _train_inputs(2, seed=7)
    r = T.wav2lip_train_step(gen_sd, sync_sd, x, indiv_mels, mel, gt, syncnet_wt=0.03, lr=1e-4)
    k = "output_block.1.weight"
    d = (gen_sd[k] - before[k]).abs()
    g = r["grads"][k].abs()
    assert torch.allclose(d[g > 1e-6], torch.full_like(d[g > 1e-6], 1e-4), rtol=2e-2)


def test_syncnet_training_step_matches_reference(gold):
    sd = O.make_state_dict("syncnet", 2, init="default")
    mel, face = O.make_syncnet_inputs(4, seed=5)
    y = torch.tensor([[1.0], [0.0], [1.0], [0.0]])
    state = None
    for step in range(2):
        r = T.syncnet_train_step(sd, face, mel, y, lr=1e-4, state=state)
        state = r["state"]
        assert close([r["loss"].item()], gold[f"sync{step}_loss"], 1e-5)
        names = list(gold[f"sync{step}_grad_names"])
        assert names == list(r["grads"].keys())
        got = np.stack([fp3(r["grads"][n]) for n in names])
        ref = gold[f"sync{step}_grad_fp"]
        assert close(got[:, 1], ref[:, 1], 1e-3) and close(got[:, 2], ref[:, 2], 1e-3)
        sd_names = list(gold[f"sync{step}_sd_names"])
        assert sd_names == list(sd.keys())
        got_sd = np.stack([fp3(sd[n]) for n in sd_names])
        assert close(got_sd[:, 1], gold[f"sync{step}_sd_fp"][:, 1], 1e-5)


def test_hq_training_step_matches_reference(gold):
    """hq_wav2lip_train.py:213-255: generator step with sync + perceptual + L1, then the discriminator's real/fake step."""
    gen_sd = O.make_state_dict("generator", 0, init="default")
    disc_sd = O.make_state_dict("disc", 3, init="default")
    sync_sd = O.make_state_dict("syncnet", 1, init="default")
    x, indiv_mels, mel, gt = _train_inputs(2, seed=8)
    states = None
    for step in range(2):
        r = T.hq_train_step(gen_sd, disc_sd, sync_sd, x, indiv_mels, mel, gt, syncnet_wt=0.03, disc_wt=0.07, states=states)
        states = r["states"]
        losses = np.array([r[k].item() for k in ("loss", "sync_loss", "perceptual", "l1", "disc_real", "disc_fake")])
        assert close(losses, gold[f"hq{step}_losses"], 2e-5), (step, losses, gold[f"hq{step}_losses"])
        for who, grads in (("gen", r["gen_grads"]), ("disc", r["disc_grads"])):
            names = list(gold[f"hq{step}_{who}_grad_names"])
            assert names == list(grads.keys())
            got = np.stack([fp3(grads[n]) for n in names])
            ref = gold[f"hq{step}_{who}_grad_fp"]
            assert close(got[:, 1], ref[:, 1], 2e-3), (who, np.abs(got[:, 1] / ref[:, 1] - 1).max())
            assert close(got[:, 2], ref[:, 2], 2e-3)
        got_sd = np.stack([fp3(v) for v in gen_sd.values()])
        assert close(got_sd[:, 1], gold[f"hq{step}_gen_sd_fp"][:, 1], 1e-5)
        got_dsd = np.stack([fp3(v) for v in disc_sd.values()])
        assert close(got_dsd[:, 1], gold[f"hq{step}_disc_sd_fp"][:, 1], 1e-5)
