"""Writes tests/golden/table_lack_resized.npz: Sawyer + table_lack_0825 composed from the MJCF asset tree (FURNITURE_ASSETS) at the
furn_size_rand factor tests/test_reset_rng.py draws (seed 77, furn_size_rand 0.1).  A resized scene can only be composed from the
asset tree; the stored scene lets that test run where the tree is absent."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from furniture_b200 import mjcf  # noqa: E402

if mjcf.default_assets_root() is None:
    sys.exit("set FURNITURE_ASSETS to the reference's furniture/env/models/assets")
factor = 1 + np.random.RandomState(77).uniform(-0.1, 0.1, 1)[0]
mjcf.load_scene("Sawyer", "table_lack_0825", resize_factor=factor).save(os.path.join(ROOT, "tests", "golden", "table_lack_resized.npz"))
