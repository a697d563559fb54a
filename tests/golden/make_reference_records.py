"""Records what the reference itself computes in the scenarios of tests/test_oracle_vs_ref.py and of
test_gpu_parity.test_cuda_path_against_the_reference_itself:  python tests/golden/make_reference_records.py [name ...]

Needs oracle/_ref/libgg_ref.so (oracle/build_ref.py, from the reference sources).  Each scenario is run on the
reference and its answers are written to tests/golden/ref_<name>.npz as digests and value samples
(tests/golden_util.ReferenceRecord); the tests then run the same scenario on the oracle port or the CUDA path and
compare check by check.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import test_gpu_parity  # noqa: E402
import test_oracle_vs_ref  # noqa: E402
from golden_util import ReferenceRecord  # noqa: E402
from oracle import ref as refmod  # noqa: E402

SCENARIOS = {name: (fn, test_oracle_vs_ref.Reference) for name, fn in test_oracle_vs_ref.SCENARIOS.items()}
SCENARIOS.update({f"cuda_{cfg}": (lambda rec, make, cfg=cfg: test_gpu_parity.full_size_stream(rec, make, cfg), test_gpu_parity.Reference)
                  for cfg in test_gpu_parity.REFERENCE_CFGS})


def main(names):
    if not refmod.available():
        raise SystemExit("oracle/_ref/libgg_ref.so is missing: build it with oracle/build_ref.py first")
    for name in names or SCENARIOS:
        fn, make = SCENARIOS[name]
        rec = ReferenceRecord(name, record=True)
        fn(rec, make)
        rec.finish()
        print(name, len(rec.keys), "checks", os.path.getsize(rec.path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1:])
