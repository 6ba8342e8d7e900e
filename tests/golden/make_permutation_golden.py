"""Golden arrays of SURVEY 8a row E6 from the UNMODIFIED reference (azchess/encoding.py:310-386), needs the reference tree:
    python tests/golden/make_permutation_golden.py  ->  tests/golden/permutations_golden.json"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import refload  # noqa: E402

enc = refload.load_reference("encoding")
out = {"horizontal_flip": [int(v) for v in enc.build_horizontal_flip_permutation()],
       "rotate180": [int(v) for v in enc.build_rotate180_permutation()]}
with open(os.path.join(HERE, "permutations_golden.json"), "w") as f:
    json.dump(out, f)
print({k: len(v) for k, v in out.items()})
