"""Write tests/golden/reference_py_lines.json: every .py file of the original Wav2Lip checkout (path relative to its
root) with its number of lines, so that tests/test_abi.py can check the file:line citations of include/w2l.h without
the checkout.

    python tests/golden/make_golden_citations.py <Wav2Lip checkout>
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def main(ref):
    lines = {}
    for dp, _dn, fn in os.walk(ref):
        for f in fn:
            if f.endswith(".py"):
                p = os.path.join(dp, f)
                lines[os.path.relpath(p, ref)] = sum(1 for _ in open(p, errors="replace"))
    with open(os.path.join(HERE, "reference_py_lines.json"), "w") as f:
        json.dump(dict(sorted(lines.items())), f, indent=1)
        f.write("\n")
    print(len(lines), "files")


if __name__ == "__main__":
    main(sys.argv[1])
