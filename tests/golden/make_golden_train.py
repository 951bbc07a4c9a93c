"""Generate tests/golden/train.npz by running ONE optimisation step of the REAL reference modules (build container
only; /root/reference is not on the GPU box):

    python tests/golden/make_golden_train.py

The training scripts parse argv and touch the dataset on import, so the step is driven from here with their own
statements (cited): wav2lip_train.py:178-198 (losses), :210-231 (the step), :357-360 (Adam over the generator's
parameters, lr = hparams.initial_learning_rate = 1e-4), color_syncnet_train.py:146-163 and hq_wav2lip_train.py:213-255
(generator + quality discriminator, Adam betas (0.5, 0.999)).  The expert SyncNet is left in
its constructor's train mode, as the scripts leave it (wav2lip_train.py:187-189).

Stored: loss values, per-parameter gradient fingerprints (sum, abs-sum, max-abs), a few raw gradient slices, the
post-step parameter / BatchNorm-buffer fingerprints.  Weights and inputs are regenerated from seeds by the tests.
"""
import os
import sys

import numpy as np
import torch
from torch import nn, optim

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")

from models import Wav2Lip, SyncNet_color, Wav2Lip_disc_qual  # noqa: E402  (the reference)
from oracle import w2l_oracle as O  # noqa: E402

syncnet_T = 5           # hparams.py
LR = 1e-4               # hparams.initial_learning_rate / syncnet_lr
SYNCNET_WT = 0.03       # hparams.py comment: "will be set automatically to 0.03 later"


def fp3(t):
    f = t.detach().double().flatten()
    return np.array([f.sum().item(), f.abs().sum().item(), f.abs().max().item()])


def train_inputs(B, seed):
    """x (B,6,T,96,96), indiv_mels (B,T,1,80,16), mel (B,1,80,16), gt (B,3,T,96,96) as the Dataset builds them
    (wav2lip_train.py:153-163): values in [0,1] / [-4,4]."""
    g = torch.Generator().manual_seed(seed)
    indiv_mels, x = O.make_generator_inputs(B, seed=seed, t=syncnet_T)
    mel = torch.rand((B, 1, 80, 16), generator=g) * 8 - 4
    gt = torch.rand((B, 3, syncnet_T, 96, 96), generator=g)
    return x, indiv_mels, mel, gt


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)   # the fp32 sums depend on the thread count: tests/test_train_oracle.py runs with 8 too
    out = {}
    B = 2

    # ---------------- wav2lip_train.py step ----------------
    model = Wav2Lip()
    model.load_state_dict(O.make_state_dict("generator", 0, init="default"), strict=True)
    syncnet = SyncNet_color()                                     # wav2lip_train.py:187: stays in train mode
    syncnet.load_state_dict(O.make_state_dict("syncnet", 1, init="default"), strict=True)
    for p in syncnet.parameters():                                # :188-189
        p.requires_grad = False
    optimizer = optim.Adam([p for p in model.parameters() if p.requires_grad], lr=LR)   # :357-360

    logloss = nn.BCELoss()                                        # :178

    def cosine_loss(a, v, y):                                     # :179-183
        d = nn.functional.cosine_similarity(a, v)
        return logloss(d.unsqueeze(1), y)

    recon_loss = nn.L1Loss()                                      # :191

    def get_sync_loss(mel, g):                                    # :192-198
        g = g[:, :, :, g.size(3) // 2:]
        g = torch.cat([g[:, :, i] for i in range(syncnet_T)], dim=1)
        a, v = syncnet(mel, g)
        y = torch.ones(g.size(0), 1).float()
        return cosine_loss(a, v, y)

    x, indiv_mels, mel, gt = train_inputs(B, seed=7)
    for step in range(2):                                         # two steps: the second sees Adam state + moved BN stats
        model.train()                                             # :211
        optimizer.zero_grad()                                     # :212
        g = model(indiv_mels, x)                                  # :220
        sync_loss = get_sync_loss(mel, g)                         # :223
        l1loss = recon_loss(g, gt)                                # :227
        loss = SYNCNET_WT * sync_loss + (1 - SYNCNET_WT) * l1loss  # :229
        loss.backward()                                           # :230
        grads = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
        optimizer.step()                                          # :231
        out[f"gen{step}_losses"] = np.array([loss.item(), sync_loss.item(), l1loss.item()])
        out[f"gen{step}_g_fp"] = fp3(g)
        out[f"gen{step}_grad_names"] = np.array(list(grads.keys()))
        out[f"gen{step}_grad_fp"] = np.stack([fp3(v) for v in grads.values()])
        out[f"gen{step}_grad_head_w"] = grads["output_block.1.weight"].flatten().numpy()
        out[f"gen{step}_grad_first_w"] = grads["face_encoder_blocks.0.0.conv_block.0.weight"].flatten()[:64].numpy()
        out[f"gen{step}_grad_dec60_w"] = grads["face_decoder_blocks.6.0.conv_block.0.weight"].flatten()[:64].numpy()
        sd = model.state_dict()
        out[f"gen{step}_sd_names"] = np.array(list(sd.keys()))
        out[f"gen{step}_sd_fp"] = np.stack([fp3(v) for v in sd.values()])
        ssd = syncnet.state_dict()
        out[f"gen{step}_expert_buf_fp"] = np.stack([fp3(v) for k, v in ssd.items() if "running" in k or "num_batches" in k])

    # ---------------- color_syncnet_train.py step ----------------
    s = SyncNet_color()
    s.load_state_dict(O.make_state_dict("syncnet", 2, init="default"), strict=True)
    opt = optim.Adam([p for p in s.parameters() if p.requires_grad], lr=LR)     # color_syncnet_train.py:262-263
    mel_s, face_s = O.make_syncnet_inputs(4, seed=5)
    y = torch.tensor([[1.0], [0.0], [1.0], [0.0]])
    for step in range(2):
        s.train()                                                 # :146
        opt.zero_grad()
        a, v = s(mel_s, face_s)                                   # :154
        loss = cosine_loss(a, v, y)                               # :157
        loss.backward()
        grads = {n: p.grad.detach().clone() for n, p in s.named_parameters()}
        opt.step()
        out[f"sync{step}_loss"] = np.array([loss.item()])
        out[f"sync{step}_grad_names"] = np.array(list(grads.keys()))
        out[f"sync{step}_grad_fp"] = np.stack([fp3(v) for v in grads.values()])
        sd = s.state_dict()
        out[f"sync{step}_sd_names"] = np.array(list(sd.keys()))
        out[f"sync{step}_sd_fp"] = np.stack([fp3(v) for v in sd.values()])

    # ---------------- hq_wav2lip_train.py step ----------------
    import torch.nn.functional as F
    DISC_WT = 0.07                                                # hparams.disc_wt
    model = Wav2Lip()
    model.load_state_dict(O.make_state_dict("generator", 0, init="default"), strict=True)
    disc = Wav2Lip_disc_qual()
    disc.load_state_dict(O.make_state_dict("disc", 3, init="default"), strict=True)
    syncnet = SyncNet_color()
    syncnet.load_state_dict(O.make_state_dict("syncnet", 1, init="default"), strict=True)
    for p in syncnet.parameters():
        p.requires_grad = False
    optimizer = optim.Adam([p for p in model.parameters() if p.requires_grad], lr=LR, betas=(0.5, 0.999))       # :418-419
    disc_optimizer = optim.Adam([p for p in disc.parameters() if p.requires_grad], lr=LR, betas=(0.5, 0.999))   # :420-421
    x, indiv_mels, mel, gt = train_inputs(B, seed=8)
    for step in range(2):
        disc.train(); model.train()                               # :213-214
        optimizer.zero_grad(); disc_optimizer.zero_grad()         # :222-223
        g = model(indiv_mels, x)                                  # :225
        sync_loss = get_sync_loss(mel, g)                         # :228
        # disc.perceptual_forward(g) (:233) moves its target with .cuda() (wav2lip.py:172) and cannot run on this CPU box;
        # its arithmetic is forward() + BCE against ones (wav2lip.py:163-174 vs :176-184):
        perceptual_loss = F.binary_cross_entropy(disc(g), torch.ones((g.size(0) * syncnet_T, 1)))
        l1loss = recon_loss(g, gt)                                # :237
        loss = SYNCNET_WT * sync_loss + DISC_WT * perceptual_loss + (1. - SYNCNET_WT - DISC_WT) * l1loss   # :239-240
        loss.backward()                                           # :242
        ggrads = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
        optimizer.step()                                          # :243
        disc_optimizer.zero_grad()                                # :246
        pred = disc(gt)                                           # :248
        disc_real_loss = F.binary_cross_entropy(pred, torch.ones((len(pred), 1)))
        disc_real_loss.backward()
        pred = disc(g.detach())                                   # :252
        disc_fake_loss = F.binary_cross_entropy(pred, torch.zeros((len(pred), 1)))
        disc_fake_loss.backward()
        dgrads = {n: p.grad.detach().clone() for n, p in disc.named_parameters()}
        disc_optimizer.step()                                     # :255
        out[f"hq{step}_losses"] = np.array([loss.item(), sync_loss.item(), perceptual_loss.item(), l1loss.item(),
                                            disc_real_loss.item(), disc_fake_loss.item()])
        out[f"hq{step}_gen_grad_names"] = np.array(list(ggrads.keys()))
        out[f"hq{step}_gen_grad_fp"] = np.stack([fp3(v) for v in ggrads.values()])
        out[f"hq{step}_disc_grad_names"] = np.array(list(dgrads.keys()))
        out[f"hq{step}_disc_grad_fp"] = np.stack([fp3(v) for v in dgrads.values()])
        out[f"hq{step}_gen_sd_fp"] = np.stack([fp3(v) for v in model.state_dict().values()])
        out[f"hq{step}_disc_sd_fp"] = np.stack([fp3(v) for v in disc.state_dict().values()])

    np.savez_compressed(os.path.join(HERE, "train.npz"), **out)
    print("wrote train.npz:", {k: getattr(v, "shape", None) for k, v in out.items() if "names" not in k})
    print("generator losses", out["gen0_losses"], out["gen1_losses"], "syncnet", out["sync0_loss"], out["sync1_loss"])


if __name__ == "__main__":
    main()
