"""Cost of the permittivity gradient (grad_eps) at the headline shape: 512^2, 4 modes, one device batch of 64 distinct problems,
want_fields=False.  Needs a GPU; prints one JSON line and writes it to --out.

* device time of the whole call with and without grad_eps, alternated in one process (b200ms_stats.device_ms);
* the two gradient kernels alone by CUDA events (b200ms_bench_stencil mode 3, 64 device-resident problems, L2 not flushed:
  the 3.2 GB the kernels write exceed the 126 MB L2 anyway);
* their achieved bytes/s against the algorithmic bytes below, and the card name and power limit read in the same call.

Algorithmic bytes per problem (csrc/sensitivity.cuh): the scan pass and the write pass each read the two in-plane E values
(s_v bytes each) and exx, eyy, iez (s_c bytes each) of every cell and mode; the write pass also writes 3 complex128 values:
    bytes = N * M * (2 * (2 * s_v + 3 * s_c) + 3 * 16)
(s_v = 8 or 16 for real or complex arithmetic; s_c = 8 for the lossless headline media.)
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tidy3d_b200 import _cabi  # noqa: E402
from tidy3d_b200 import workloads as W  # noqa: E402
from tidy3d_b200.solver import compute_modes_batch  # noqa: E402


def algorithmic_bytes(n_cells, modes, batch, s_v, s_c):
    return float(n_cells) * modes * batch * (2 * (2 * s_v + 3 * s_c) + 3 * 16)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--nrep", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    probs = []
    for i in range(a.batch):  # distinct media: core width 0.40 .. 0.71 um
        wl = W.si_strip(a.n, 4, w=0.40 + 0.31 * i / max(1, a.batch - 1))
        probs.append(dict(eps_cross=wl.eps_cross, coords=wl.coords, freq=float(wl.freqs[0]), mode_spec=wl.mode_spec))
    h = _cabi.Handle()
    h.set_options(max_batch=a.batch)
    times = {"plain": [], "grad": []}
    n_ref, is_complex = None, False
    compute_modes_batch(probs, want_fields=False, handle=h)  # warm-up
    for _ in range(a.rounds):
        for key in ("plain", "grad"):
            out, infos = compute_modes_batch(probs, want_fields=False, handle=h, grad_eps=(key == "grad"), return_info=True)
            is_complex = infos[0]["is_complex"]
            st = h.last_stats()
            assert st["device_batches"] == 1
            times[key].append(st["device_ms"])
            n = np.stack([o[1] for o in out])
            n_ref = n if n_ref is None else n_ref
            assert np.array_equal(n, n_ref), "n_complex changed between calls"
    pk = _cabi.PackedProblem(probs[0]["eps_cross"], probs[0]["coords"], probs[0]["freq"], probs[0]["mode_spec"])
    ms, nbytes = C.c_double(), C.c_double()
    rc = _cabi.lib().b200ms_bench_stencil(h._h, C.byref(pk.struct), a.batch, 3, a.nrep, 0, None, None, C.byref(ms), C.byref(nbytes))
    assert rc == _cabi.OK, h.last_error()
    formula = algorithmic_bytes(a.n * a.n, 4, a.batch, 16 if is_complex else 8, 8)
    assert abs(formula - nbytes.value) < 1e-6 * formula, (formula, nbytes.value)
    rec = dict(
        shape=f"{a.n}x{a.n}", modes=4, batch=a.batch, card=card(),
        device_ms_plain=times["plain"], device_ms_grad=times["grad"],
        grad_overhead_ms=float(np.median(times["grad"]) - np.median(times["plain"])),
        kernel_ms=ms.value, algorithmic_bytes=formula, achieved_tb_s=formula / (ms.value * 1e-3) / 1e12,
    )  # fmt: skip
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
