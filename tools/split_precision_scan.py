"""Parity margin of the split-integer mode for several digit counts S: full fits against the golden vectors of the
reference's float64 path.  Prints max-norm relative errors of ws / TCs and whether the iteration count matched."""
import os
import sys

import numpy as np

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
sys.path.insert(0, "oracle")
from conftest import load_golden  # noqa: E402
from linearcorex_b200 import Corex  # noqa: E402

CASES = ["readme_demo_f64", "big5_l0_f64", "syn_400x300x10_f64", "syn_60x400x8_f64", "outliers_missing_f64",
         "standard_missing_f64", "adni_l1_f64", "syn_4000x2000x20_f64", "adni_l0_f64"]
for S in (6, 5, 4):
    os.environ["LCX_SPLIT_DIGITS"] = str(S)
    worst = 0.0
    for name in CASES:
        z, kw, x = load_golden(name)
        mdl = Corex(precision="fp64_split", **kw)
        if name.startswith("readme_demo"):
            x = np.random.random((100, 50))
        mdl.fit(x)
        ew = np.abs(mdl.ws - z["ws"]).max() / np.abs(z["ws"]).max() if mdl.ws.shape == z["ws"].shape else np.nan
        et = np.abs(mdl.tcs - z["m_TCs"]).max() / np.abs(z["m_TCs"]).max()
        same = len(mdl.history["TC"]) == len(z["history_TC"])
        worst = max(worst, ew if same else 1.0)
        print("S=%d %-26s it %5d/%5d  |dW|=%.2e  |dTCs|=%.2e" % (S, name, len(mdl.history["TC"]), len(z["history_TC"]), ew, et),
              flush=True)
    print("S=%d WORST %.2e" % (S, worst), flush=True)
