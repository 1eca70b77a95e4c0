"""DEV TOOL: small solves with grad_eps for compute-sanitizer memcheck, one case per arithmetic kind of the gradient kernels:
c1_64 (real), c3_96 (complex vectors, real coefficient fields: PML), lossy_48 (complex fields)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.golden.cases import CASES  # noqa: E402
from tidy3d_b200 import compute_modes_batch  # noqa: E402

for name in sys.argv[1:] or ["c1_64", "c3_96", "lossy_48"]:
    fac, kw, _ = CASES[name]
    wl = fac()
    p = dict(eps_cross=wl.eps_cross, coords=wl.coords, freq=wl.freqs[0], mode_spec=wl.mode_spec, **kw)
    out, infos = compute_modes_batch([p, p], want_fields=False, return_info=True, grad_eps=[True, False])
    g = infos[0]["grad_eps"]
    print(name, "complex" if infos[0]["is_complex"] else "real", "max|dn/deps|", float(np.abs(g).max()), "finite", bool(np.isfinite(g).all()), flush=True)
