"""Host-only estimate of the pair kernel's tile skip (DESIGN.md section 4.1).

The pair kernel skips a 128-event tile for a warp of 32 chains when every event
of the tile is above the mass cut (500) for every parameter point in the box
spanned by those chains.  This script builds the bench's synthetic sample,
lays it out as the engine does -- (class, mass band, separation or mass) --
and counts the fraction of pairs that fall in such tiles for a box
p in [-r, r] in each parameter, for a given table of band edges.  FP64, no
error margin: an estimate, not the kernel's rule.

  python scripts/skip_fraction.py [--events N] [--box R] [--edges 450,550,600,700,900]
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "root-simple-mcmc_b200"))
sys.path.insert(0, ROOT)

TILE = 128


def prepared(ev):
    nom = np.log(ev["TrueMass"])
    d = np.log(ev["Mass"]) - nom
    ls = d / (np.log(ev["TrueMass"] + ev["TrueMassSigma"]) - nom)
    cls = np.where(ev["Type"] == 0, 0, 2) + (ev["MuDk"] > 0)
    return nom, d, ls, cls


def min_log_mass(nom, d, ls, r):
    """Smallest corrected log-mass over the box p2, p3, p4 in [-r, r] (the corner rule)."""
    from scipy.special import erf
    sk_lo, sk_hi = 0.3 * erf(-r / 10.0), 0.3 * erf(r / 10.0)
    w_lo, w_hi = np.exp(-r / 10.0), np.exp(r / 10.0)
    sk = np.where((d >= 0) == (ls >= 0), sk_lo, sk_hi)
    w = np.where(d >= 0, w_lo, w_hi)
    return nom + w * d * np.exp(ls * sk) - r / 10.0


def skip_fraction(ev, r, edges):
    nom, d, ls, cls = prepared(ev)
    cut = min_log_mass(nom, d, ls, r) >= np.log(500.0)
    band = np.searchsorted(np.asarray(edges, float), ev["Mass"], side="right")
    skipped = banded = 0
    for c in range(4):
        sel = np.nonzero(cls == c)[0]
        second = ev["Separation"][sel] if c in (0, 2) else ev["Mass"][sel]
        order = sel[np.lexsort((second, band[sel]))]
        flags = cut[order]
        n = len(flags)
        padded = np.concatenate([flags, np.ones((-n) % TILE, bool)]).reshape(-1, TILE)
        whole = padded.all(axis=1)
        real = np.minimum(TILE, n - TILE * np.arange(len(whole)))
        skipped += int(real[whole].sum())
        banded += int(np.count_nonzero(flags))
    total = len(ev)
    return skipped / total, banded / total


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--events", type=int, default=1_000_000)
    ap.add_argument("--box", type=float, nargs="+", default=[0.5, 1.0, 2.0])
    ap.add_argument("--edges", default="450,550,600,700,900")
    args = ap.parse_args()
    import bench
    ev, _ = bench.workload_inputs(args.events)
    edges = [float(v) for v in args.edges.split(",")]
    for r in args.box:
        tiles, events = skip_fraction(ev, r, edges)
        print("box +-%.2f  edges %s  pairs in skipped tiles %.1f %%  (upper bound, per event %.1f %%)"
              % (r, args.edges, 100 * tiles, 100 * events))


if __name__ == "__main__":
    main()
