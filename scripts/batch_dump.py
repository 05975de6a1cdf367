"""Dumps what the uniform batch and single fits compute, to compare two builds byte for byte.

`dump` runs, from the package tree at --root, fit_cnmf_batch with an integer K (cmf_create_batch) for R in {1, 8, 64} and
single fit_cnmf fits, fp64 and fp32, at the config-1 shape (N=500, T=2000, K=5, L=10), 100 iterations without early stop,
and writes every W, H and loss_hist as .npy under --out.  `compare` reads two such directories and reports, per array,
whether the bytes are equal.  Run `dump` once per build (e.g. a change and its parent) on the same machine, then `compare`."""
import argparse
import json
import os
import sys

import numpy as np

N, T, K, L, ITR = 500, 2000, 5, 10, 100
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dump(root, out):
    sys.path.insert(0, os.path.abspath(root))            # the package (built already) of the tree under test
    sys.path.append(REPO)                                  # the data generator
    import cmf_jl_b200 as cmf
    from oracle import cnmf_oracle as po

    assert os.path.dirname(os.path.abspath(cmf.__file__)).startswith(os.path.abspath(root)), cmf.__file__
    X, _, _ = po.synthetic_sequences(K=3, N=N, L=20, T=T, rng=np.random.default_rng(1234))
    os.makedirs(out, exist_ok=True)
    kw = dict(L=L, K=K, max_itr=ITR, check_convergence=False, layout="KNL")
    for dtype in ("f64", "f32"):
        for R in (1, 8, 64):
            for r, res in enumerate(cmf.fit_cnmf_batch(X, seeds=list(range(R)), dtype=dtype, **kw)):
                for name in ("W", "H", "loss_hist"):
                    np.save(os.path.join(out, f"batch_{dtype}_R{R}_r{r}_{name}.npy"), np.asarray(getattr(res, name)))
        for seed in range(4):
            res = cmf.fit_cnmf(X, seed=seed, dtype=dtype, **kw)
            for name in ("W", "H", "loss_hist"):
                np.save(os.path.join(out, f"single_{dtype}_s{seed}_{name}.npy"), np.asarray(getattr(res, name)))


def compare(a, b):
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b)), "the two dumps hold different arrays"
    differ = [n for n in names if np.load(os.path.join(a, n)).tobytes() != np.load(os.path.join(b, n)).tobytes()]
    return {"arrays": len(names), "identical": len(names) - len(differ), "differ": differ}


def main():
    ap = argparse.ArgumentParser()
    sub = ap.add_subparsers(dest="cmd", required=True)
    d = sub.add_parser("dump")
    d.add_argument("--root", default=REPO)
    d.add_argument("--out", required=True)
    c = sub.add_parser("compare")
    c.add_argument("a")
    c.add_argument("b")
    c.add_argument("--json", help="also write the result here")
    args = ap.parse_args()
    if args.cmd == "dump":
        dump(args.root, args.out)
        return
    res = compare(args.a, args.b)
    print(json.dumps(res))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    sys.exit(0 if not res["differ"] else 1)


if __name__ == "__main__":
    main()
