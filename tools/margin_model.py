"""CPU model of the prefilter margin: how wide is 2*eps against the spread of the scores, per shadow format?

The engine is exact whatever the prefilter format; the format only decides how many rows fall within the error
margin of the k-th score (survivors the candidate lists must hold, rows finalize_kernel rescores in fp64).  This
script re-derives the AUTO threshold of the int8 shadow (median 2 eps8 / sigma <= 1.2, b2f_api.cu choose_format):

    python tools/margin_model.py [--rows 100000] [--total 38636520] [--k 100]

Method: the project's synthetic generator (isotropic rows and rows with a common mean), the exact eps formulas of
pass_init_kernel (mode 2 bf16, mode 4 int8 with one scale per 32-row tile and per query), the k-th score at the
full size from a Gaussian tail fit to the sampled scores.  "survivors" = rows with s~ >= s_k - 2 eps,
"window" = rows within eps of s_k (what the second rescoring round reads).
"""
import argparse
import os
import sys

import numpy as np
from scipy.stats import norm as N

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from convdr_b200 import synth  # noqa: E402


def bf16(x):
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32).astype(np.float64)


def int8_tiles(x, rows=32):
    out = np.empty_like(x)
    for t in range(0, len(x), rows):
        blk = x[t:t + rows]
        s = np.abs(blk).max() / 127.0
        out[t:t + rows] = np.clip(np.rint(blk / s), -127, 127) * s if s > 0 else 0.0
    return out


def int8_rows(x):
    s = np.abs(x).max(axis=1, keepdims=True) / 127.0
    return np.clip(np.rint(x / np.where(s > 0, s, 1)), -127, 127) * s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000)
    ap.add_argument("--total", type=int, default=38_636_520)
    ap.add_argument("--nq", type=int, default=173)
    ap.add_argument("--k", type=int, default=100)
    a = ap.parse_args()
    z = N.isf(a.k / a.total)
    for name, nrm, ms in (("iso", 1.0, 0), ("aniso", 28.0, 443)):
        P = synth.block(0, a.rows, seed=0, stream=0, norm=nrm, mean_shift=ms).astype(np.float64)
        Q = synth.block(0, a.nq, seed=0, stream=1, norm=nrm, mean_shift=ms).astype(np.float64)
        pc = P - P[:65536].mean(0)
        Pm = np.linalg.norm(pc, axis=1).max()
        qn = np.linalg.norm(Q, axis=1)
        sd = (Q @ pc.T).std(1)
        E16 = np.linalg.norm(pc - bf16(pc), axis=1).max()
        eq16 = np.linalg.norm(Q - bf16(Q), axis=1)
        eps16 = qn * E16 * (1 + 2**-8) + eq16 * Pm + 1.1e-4 * qn * Pm
        E8 = np.linalg.norm(pc - int8_tiles(pc), axis=1).max()
        eq8 = np.linalg.norm(Q - int8_rows(Q), axis=1)
        eps8 = (qn + eq8) * E8 + eq8 * Pm + (qn + eq8) * (Pm + E8) * 2**-21
        for tag, eps in (("bf16", eps16), ("int8", eps8)):
            r = 2 * eps / sd
            surv = a.total * N.sf(z - r)
            win = a.total * N.sf(z - eps / sd) - a.k
            print(f"{name:5s} {tag:4s} 2eps/sigma median {np.median(r):.3f} max {r.max():.3f} | survivors/query "
                  f"median {np.median(surv):9.0f} max {surv.max():9.0f} | window median {np.median(win):7.0f}")


if __name__ == "__main__":
    main()
