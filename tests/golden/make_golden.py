"""Generate tests/golden/*.npz by running the REAL reference modules (build container only).

    python tests/golden/make_golden.py

Imports `models` from /root/reference (read-only mount, not present on the GPU box), loads the
seeded weights from oracle.w2l_oracle.make_state_dict() with strict=True (which also proves the
key sets are identical), runs the reference forward on the seeded inputs and stores the outputs
plus per-block fingerprints.  Weights and inputs are NOT stored (145 MB): they are regenerated
from the seed by the same CPU torch.Generator calls; an input/weight checksum is stored so RNG
drift is detected instead of silently passing.

The mel vectors are produced by oracle/mel_oracle.py itself (librosa is not installable here —
"parity unpinned" at the librosa boundary, see that file's header); they pin the oracle against
accidental edits and feed the GPU tests.
"""
import os
import sys

import numpy as np
import torch

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")

from models import Wav2Lip, SyncNet_color, Wav2Lip_disc_qual  # noqa: E402  (the reference)
from oracle import w2l_oracle as O  # noqa: E402
from oracle import mel_oracle as M  # noqa: E402


def fingerprint(t: torch.Tensor) -> np.ndarray:
    """[sum, abs-sum, max-abs] in float64 + the first 32 and the last 32 flattened values."""
    f = t.detach().double().flatten()
    head = f[:32].numpy()
    tail = f[-32:].numpy()
    return np.concatenate([[f.sum().item(), f.abs().sum().item(), f.abs().max().item()], head, tail])


def checksum_sd(sd) -> float:
    return float(sum(v.double().abs().sum().item() for v in sd.values() if v.dtype.is_floating_point))


def hook_blocks(model, names, store):
    mods = dict(model.named_modules())
    handles = []
    for n in names:
        handles.append(mods[n].register_forward_hook(
            lambda _m, _i, o, n=n: store.__setitem__(n, fingerprint(o))))
    return handles


def main():
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count() or 1)
    out = {}

    # ---------------- generator ----------------
    sd = O.make_state_dict("generator", seed=0)
    g = Wav2Lip()
    g.load_state_dict(sd, strict=True)
    g.eval()
    names = [n for n, _ in O.generator_layers()]
    fps = {}
    logits = {}
    hs = hook_blocks(g, names, fps)
    hs.append(g.output_block[1].register_forward_hook(lambda _m, _i, o: logits.__setitem__("l", o.detach().clone())))
    mel, face = O.make_generator_inputs(2, seed=0)
    with torch.no_grad():
        y = g(mel, face)
    out["gen4_out"] = y.numpy()
    out["gen4_logits"] = logits["l"].numpy()
    for n in names:
        out["gen4_fp/" + n] = fps[n]
    out["gen_sd_checksum"] = np.float64(checksum_sd(sd))
    out["gen4_in_checksum"] = np.array([mel.double().abs().sum().item(), face.double().abs().sum().item()])
    mel5, face5 = O.make_generator_inputs(2, seed=1, t=5)
    with torch.no_grad():
        y5 = g(mel5, face5)
    out["gen5_out"] = y5.numpy()
    out["gen5_in_checksum"] = np.array([mel5.double().abs().sum().item(), face5.double().abs().sum().item()])
    # odd batch size (exercises partial tiles): N = 3
    mel3, face3 = O.make_generator_inputs(3, seed=2)
    with torch.no_grad():
        y3 = g(mel3, face3)
    out["gen4n3_out"] = y3.numpy()
    for h in hs:
        h.remove()
    # the reference's own initialisation statistics ("random weights" of BASELINE.json configs[0..1])
    sdd = O.make_state_dict("generator", seed=0, init="default")
    gd = Wav2Lip()
    gd.load_state_dict(sdd, strict=True)
    gd.eval()
    lg = {}
    hd = gd.output_block[1].register_forward_hook(lambda _m, _i, o: lg.__setitem__("l", o.detach().clone()))
    with torch.no_grad():
        yd = gd(mel, face)
    hd.remove()
    out["gen4_default_out"] = yd.numpy()
    out["gen4_default_logits"] = lg["l"].numpy()
    out["gen_default_sd_checksum"] = np.float64(checksum_sd(sdd))
    np.savez_compressed(os.path.join(HERE, "generator.npz"), **out)

    # ---------------- syncnet ----------------
    out = {}
    sd = O.make_state_dict("syncnet", seed=0)
    s = SyncNet_color()
    s.load_state_dict(sd, strict=True)
    s.eval()
    names = [n for n, _ in O.syncnet_layers()]
    fps = {}
    hs = hook_blocks(s, names, fps)
    mel, face = O.make_syncnet_inputs(3, seed=0)
    with torch.no_grad():
        a, v = s(mel, face)
    out["sync_a"] = a.numpy()
    out["sync_v"] = v.numpy()
    for n in names:
        out["sync_fp/" + n] = fps[n]
    out["sync_sd_checksum"] = np.float64(checksum_sd(sd))
    out["sync_in_checksum"] = np.array([mel.double().abs().sum().item(), face.double().abs().sum().item()])
    for h in hs:
        h.remove()
    np.savez_compressed(os.path.join(HERE, "syncnet.npz"), **out)

    # ---------------- disc ----------------
    out = {}
    sd = O.make_state_dict("disc", seed=0)
    d = Wav2Lip_disc_qual()
    d.load_state_dict(sd, strict=True)
    d.eval()
    names = [n for n, _ in O.disc_layers()]
    fps = {}
    logits = {}
    hs = hook_blocks(d, names, fps)
    hs.append(d.binary_pred[0].register_forward_hook(lambda _m, _i, o: logits.__setitem__("l", o.detach().clone())))
    frames = O.make_disc_inputs(2, t=5, seed=0)
    with torch.no_grad():
        p = d(frames)
    out["disc_out"] = p.numpy()
    out["disc_logits"] = logits["l"].reshape(-1, 1).numpy()
    for n in names:
        out["disc_fp/" + n] = fps[n]
    out["disc_sd_checksum"] = np.float64(checksum_sd(sd))
    out["disc_in_checksum"] = np.float64(frames.double().abs().sum().item())
    for h in hs:
        h.remove()
    np.savez_compressed(os.path.join(HERE, "disc.npz"), **out)

    # ---------------- mel (oracle-generated; parity unpinned at the librosa boundary) ----------------
    out = {}
    for kind in ("noise", "sweep", "mix"):
        wav = M.make_wav(48000 + 137, seed=7, kind=kind)  # non-multiple of hop
        out["mel_" + kind] = M.melspectrogram(wav)
        out["wav_checksum_" + kind] = np.float64(np.abs(wav.astype(np.float64)).sum())
    out["mel_basis"] = M.mel_basis()
    np.savez_compressed(os.path.join(HERE, "mel.npz"), **out)
    reference_seed3()
    for f in ("generator", "syncnet", "disc", "mel", "reference_seed3"):
        print(f, os.path.getsize(os.path.join(HERE, f + ".npz")) // 1024, "KiB")


def reference_seed3():
    """Full outputs of the three reference networks on a second weight seed (3) and input seed (5), for
    tests/test_oracle_golden.py::test_oracle_vs_live_reference."""
    out = {}
    sd = O.make_state_dict("generator", 3)
    m = Wav2Lip()
    m.load_state_dict(sd, strict=True)
    m.eval()
    mel, face = O.make_generator_inputs(1, 5)
    with torch.no_grad():
        out["gen_out"] = m(mel, face).numpy()
    out["gen_sd_checksum"] = np.float64(checksum_sd(sd))
    out["gen_in_checksum"] = np.array([mel.double().abs().sum().item(), face.double().abs().sum().item()])
    sd = O.make_state_dict("syncnet", 3)
    s = SyncNet_color()
    s.load_state_dict(sd, strict=True)
    s.eval()
    mel, face = O.make_syncnet_inputs(2, 5)
    with torch.no_grad():
        a, v = s(mel, face)
    out["sync_a"], out["sync_v"] = a.numpy(), v.numpy()
    sd = O.make_state_dict("disc", 3)
    d = Wav2Lip_disc_qual()
    d.load_state_dict(sd, strict=True)
    d.eval()
    with torch.no_grad():
        out["disc_out"] = d(O.make_disc_inputs(1, 5, 5)).numpy()
    np.savez_compressed(os.path.join(HERE, "reference_seed3.npz"), **out)


if __name__ == "__main__":
    main()
