"""Regenerates tests/golden/denoise_cornell_4096spp.npz, the 4096-spp oracle render test_denoise's quality test measures
against (run from the repo root: python tests/golden/make_denoise_golden.py; about 40 s on 8 host threads)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle as O  # noqa: E402
from yuki_b200 import transforms as xf  # noqa: E402
import test_denoise as TD  # noqa: E402

TD.make_golden(xf, O)
print("wrote", TD.GOLDEN_REF)
