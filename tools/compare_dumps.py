"""Compare two `bench.py --dump-outputs` directories (no GPU needed).

Usage: compare_dumps.py A B [--json OUT]

Both dumps must come from runs with identical arguments (the rows of a dump are a seeded sample).  For every block (raw,
smooth) and feature it reports the largest absolute difference, the largest relative difference |a - b| / max (1, |a|) (the
measure the parity tests use) and the number of rows whose non-finite class differs (finite / +inf / -inf / NaN).  The dumps
do not carry the pitch lag; the frame's f0 is sr / (2 lag) or -sr, a function of the lag alone, so rows whose raw f0 differs are
the rows whose lag differs, and they are counted and listed.  Exits 1 when the row sets differ."""
import argparse
import json
import os
import sys

import numpy as np

FEATURES = ("onset", "rms", "f0", "centroid", "spread", "flatness", "ler", "flux", "slope", "her", "oer", "inharm")


def load(d, name):
    return np.load(os.path.join(d, name + ".npy")), np.load(os.path.join(d, name + "_nonfinite.npy"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--json", help="also write the report as JSON")
    args = ap.parse_args()

    ra, rb = np.load(os.path.join(args.a, "rows.npy")), np.load(os.path.join(args.b, "rows.npy"))
    if not np.array_equal(ra, rb):
        print("the dumps hold different rows: compare runs with identical arguments")
        return 1
    report = {"rows": int(len(ra))}
    for block in ("raw", "smooth"):
        va, ca = load(args.a, block)
        vb, cb = load(args.b, block)
        both = (ca == 0) & (cb == 0)
        feats = {}
        for i, name in enumerate(FEATURES):
            m = both[:, i]
            d = np.abs(va[m, i].astype(np.float64) - vb[m, i].astype(np.float64))
            rel = d / np.maximum(1.0, np.abs(va[m, i].astype(np.float64)))
            feats[name] = {
                "max_abs": float(d.max()) if d.size else 0.0,
                "max_rel": float(rel.max()) if rel.size else 0.0,
                "differ": int((d > 0).sum()),
                "nonfinite_class_differs": int((ca[:, i] != cb[:, i]).sum()),
            }
        report[block] = feats
    va, ca = load(args.a, "raw")
    vb, cb = load(args.b, "raw")
    f0 = FEATURES.index("f0")
    lag_rows = np.nonzero((va[:, f0] != vb[:, f0]) | (ca[:, f0] != cb[:, f0]))[0]
    report["lag_differs"] = int(len(lag_rows))
    report["lag_differs_rows"] = [int(ra[r]) for r in lag_rows[:50]]

    print(f"{report['rows']} rows")
    for block in ("raw", "smooth"):
        print(f"{block}:  {'feature':9s} {'max abs':>10s} {'max rel':>10s} {'rows differ':>12s} {'class differs':>14s}")
        for name, f in report[block].items():
            print(f"        {name:9s} {f['max_abs']:10.3g} {f['max_rel']:10.3g} {f['differ']:12d} {f['nonfinite_class_differs']:14d}")
    print(f"rows whose lag differs (raw f0 differs): {report['lag_differs']}" + (f"  first rows (t * F + f): {report['lag_differs_rows'][:10]}" if report["lag_differs"] else ""))
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(report, fh, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
