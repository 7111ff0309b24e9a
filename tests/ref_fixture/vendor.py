"""Copy the reference's caller scripts, model classes and training utilities VERBATIM into tests/ref_fixture/.

    python tests/ref_fixture/vendor.py            # in the build container, where /root/reference exists

TEST INFRASTRUCTURE ONLY.  These files are the unmodified MIT-licensed sources of usc-sail/speech-emotion-privacy-trust
(LICENSE copied next to them).  They exist in this repository for one purpose: north_star requires that the reference's
own train() / test() functions "run unchanged" against the drop-in modules, and the GPU box that runs the parity tests
has no /root/reference.  Nothing in the product package imports, reads or executes anything under tests/ref_fixture/;
tests/ref_harness.py drives them.  `--check` verifies the committed copies still equal the reference byte for byte.
Copying also records the SHA-256 of every copied file in tests/golden/ref_fixture_sha256.json, so the test suite can
check the copies against the reference without a checkout of it; `--check` verifies that file against the reference too.
"""
from __future__ import annotations

import hashlib
import json
import shutil
import sys
from pathlib import Path

REF = Path("/root/reference")
HERE = Path(__file__).resolve().parent
DIGESTS = HERE.parent / "golden" / "ref_fixture_sha256.json"
FILES = [
    "LICENSE",
    "training/training_cloak_with_grl.py",
    "training/training_cloak.py",
    "training/adversary_cloak_evaluation.py",
    "training/training_adversary_baselines.py",
    "utils/training_tools.py",
    "model/baseline_models.py",
    "model/cloak_models.py",
    "model/reversal_gradient.py",
]


def main(check: bool) -> int:
    bad = 0
    for rel in FILES:
        src, dst = REF / rel, HERE / rel
        if check:
            same = dst.exists() and dst.read_bytes() == src.read_bytes()
            print(("ok      " if same else "DIFFERS ") + rel)
            bad += not same
        else:
            dst.parent.mkdir(parents=True, exist_ok=True)
            shutil.copyfile(src, dst)
            print("copied", rel)
    digests = {rel: hashlib.sha256((REF / rel).read_bytes()).hexdigest() for rel in FILES}
    if check:
        same = DIGESTS.exists() and json.loads(DIGESTS.read_text()) == digests
        print(("ok      " if same else "DIFFERS ") + str(DIGESTS.relative_to(HERE.parent.parent)))
        bad += not same
    else:
        DIGESTS.write_text(json.dumps(digests, indent=1) + "\n")
    return bad


if __name__ == "__main__":
    sys.exit(main("--check" in sys.argv))
