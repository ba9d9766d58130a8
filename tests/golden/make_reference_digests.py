#!/usr/bin/env python
"""Record tests/golden/reference_digests.json: the sha256 digests (and status codes) of the reference library's
results for the cases of tests/test_oracle.py section (b), so that the oracle is held to them in every checkout.

    python tests/golden/make_reference_digests.py                 # from the reference (oracle/_ref/libvvdsp_ref.so)
    python tests/golden/make_reference_digests.py --from-oracle   # from the oracle restatement

--from-oracle is valid only while the oracle is bit-identical to the reference on these cases; the same tests
check that live wherever oracle/_ref is built.
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]
import test_oracle as t  # noqa: E402
from oracle.oracle import Oracle, Reference  # noqa: E402

SOURCES = {
    "reference": "the reference library, oracle/_ref/libvvdsp_ref.so",
    "oracle": "the oracle restatement (oracle/vvdsp_oracle.c, oracle/driver.c), which the live comparison against the "
              "reference library found bit-identical on every one of these cases",
}


def main():
    from_oracle = "--from-oracle" in sys.argv[1:]
    oracle = Oracle()
    impl = oracle if from_oracle else Reference()
    digests = {}
    with tempfile.TemporaryDirectory() as tmp:
        cases = [c for nfft, hop, win in t.LIVE_STFT for c in t.stft_cases(oracle, nfft, hop, win)]
        cases += [*t.status_cases(oracle), *t.mel_cases(oracle), *t.mfcc_cases(oracle), *t.pcm_cases(oracle, tmp)]
        for key, mine, theirs in cases:
            assert key not in digests, key
            digests[key] = t.bits((mine if from_oracle else theirs)(impl))
    out = os.path.join(HERE, "reference_digests.json")
    with open(out, "w") as f:
        json.dump(dict(generator="tests/golden/make_reference_digests.py", source=SOURCES["oracle" if from_oracle else "reference"],
                       digests=digests), f, indent=1)
        f.write("\n")
    print(f"{len(digests)} digests -> {out}")


if __name__ == "__main__":
    main()
