"""Golden vectors for scope row f4 from the REAL reference: /root/reference/face_detection/detection/sfd/{net_s3fd,detect,
bbox}.py are loaded by path (they need torch, numpy, cv2, scipy only), seeded weights from oracle/s3fd_oracle.make_state_dict
are loaded with strict=True, and the module's 12 output maps (fingerprints + a slice each), the batch_detect candidate array
and the NMS keep lists are stored.  Run in the build container:  python tests/golden/make_golden_s3fd.py"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from oracle import s3fd_oracle as S  # noqa: E402

REF = "/root/reference/face_detection/detection/sfd"


def load_reference():
    pkg = types.ModuleType("refsfd")
    pkg.__path__ = [REF]
    sys.modules["refsfd"] = pkg
    mods = {}
    for name in ("net_s3fd", "bbox", "detect"):
        spec = importlib.util.spec_from_file_location("refsfd." + name, os.path.join(REF, name + ".py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules["refsfd." + name] = m
        spec.loader.exec_module(m)
        mods[name] = m
    return mods


def fp(t):
    f = t.detach().double().flatten()
    return np.array([f.sum().item(), f.abs().sum().item(), f.abs().max().item()])


def main():
    ref = load_reference()
    sd = S.make_state_dict(0)
    net = ref["net_s3fd"].s3fd()
    net.load_state_dict(sd, strict=True)
    net.eval()
    imgs = S.make_images(2, 96, 128, seed=1)
    out = {}
    with torch.no_grad():
        olist = net(S.preprocess(imgs))
    for i, o in enumerate(olist):
        out[f"o{i}"] = o.numpy()
        out[f"o{i}_fp"] = fp(o)
    cand = ref["detect"].batch_detect(net, imgs, device="cpu")
    out["candidates"] = cand.astype(np.float32)
    keeps = [np.array(ref["bbox"].nms(cand[:, i, :], 0.3), dtype=np.int64) for i in range(cand.shape[1])]
    for i, k in enumerate(keeps):
        out[f"keep{i}"] = k
    # a larger, odd-sized frame: fingerprints only
    imgs2 = S.make_images(1, 150, 210, seed=2)
    with torch.no_grad():
        o2 = net(S.preprocess(imgs2))
    out["big_fp"] = np.stack([fp(o) for o in o2])
    out["big_shapes"] = np.array([list(o.shape) for o in o2], dtype=np.int32)
    np.savez_compressed(os.path.join(HERE, "s3fd.npz"), **out)
    print("wrote s3fd.npz:", cand.shape, [len(k) for k in keeps], [tuple(o.shape) for o in olist])
    seed3(ref)


def seed3(ref):
    """The 12 output maps at a second weight seed (3) on a 70x90 frame (seed 5), for
    tests/test_s3fd_oracle.py::test_oracle_against_live_reference."""
    net = ref["net_s3fd"].s3fd()
    net.load_state_dict(S.make_state_dict(3), strict=True)
    net.eval()
    with torch.no_grad():
        olist = net(S.preprocess(S.make_images(1, 70, 90, seed=5)))
    np.savez_compressed(os.path.join(HERE, "s3fd_seed3.npz"), **{f"o{i}": o.numpy() for i, o in enumerate(olist)})
    print("wrote s3fd_seed3.npz:", [tuple(o.shape) for o in olist])


if __name__ == "__main__":
    main()
