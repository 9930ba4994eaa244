"""Child process of tests/test_gpu_spanning_regions.py: the ps_create_multi handle against the single-GPU handle
(tests/multi_worker.py) on scenes whose reduced regions cross the cuts.  usage: python spanning_multi_worker.py <case> <ndev>"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import multi_worker  # noqa: E402
import spanning_cases  # noqa: E402

for name in ("span_blob64_notile", "span_blob64_tile8_pad0", "span_s3_128_notile", "span_bodies_notile"):
    multi_worker.CASES[name] = (lambda n: lambda: spanning_cases.CASES[n]()[0])(name)

if __name__ == "__main__":
    multi_worker.main(sys.argv[1], int(sys.argv[2]))
