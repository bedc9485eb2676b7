"""Developer aid for A/B runs of the force kernel: the first forces after upload of bench.py's N = 3500 state, and their comparison.

  python scripts/first_forces.py OUT.npy        forces of the library MDQT_LIB_PATH (default: the tree's) -> OUT.npy
  python scripts/first_forces.py --compare DIR  DIR/F_parent.npy against DIR/F_new.npy, per ion against tests/pair_reference.py's
                                                S (sum of |terms|), and bench.py's dumps DIR/dump_{parent,new}_{1,20}"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(HERE), os.path.join(os.path.dirname(HERE), "tests")]
N = 3500


def state():
    from mdqtplasmasims_b200 import su_params, synthetic
    p = su_params(n_ions=N, N0=N)
    return p, synthetic.random_positions(N, p.L, seed=12345)  # bench.py's synthetic_state, job 0


def forces(out):
    from mdqtplasmasims_b200 import Engine
    p, R = state()
    e = Engine(p)
    e.upload(R=R)
    e.forces()
    np.save(out, e.download_forces())
    e.close()


def compare(d):
    import pair_reference as pr
    p, R = state()
    Fp, Fn = np.load(os.path.join(d, "F_parent.npy")), np.load(os.path.join(d, "F_new.npy"))
    s = pr.ion_sums(R, p.L, p.kappa, p.rcut)
    print("first forces, N = %d: max |F_new - F_parent| / S = %.3e, identical components %d of %d; max error / bound: parent %.3e, new %.3e" % (
        N, float((np.abs(Fn - Fp) / s["SF"]).max()), int((Fn == Fp).sum()), Fn.size,
        *[float((np.abs(F - s["F"]) / pr.bound(s["SF"], s["QF"], pr.chain(64, 55, N), N, p.kappa * p.rcut)).max()) for F in (Fp, Fn)]))
    for steps in (1, 20):
        a, b = (os.path.join(d, "dump_%s_%d" % (k, steps)) for k in ("parent", "new"))
        if not (os.path.isdir(a) and os.path.isdir(b)):
            continue
        rel = {}
        for k in ("R", "V", "psi", "F"):
            x, y = np.load(os.path.join(a, k + ".npy")), np.load(os.path.join(b, k + ".npy"))
            rel[k] = float(np.abs(x - y).max() / np.abs(x).max())
        ta, tb = np.load(os.path.join(a, "tPart.npy")), np.load(os.path.join(b, "tPart.npy"))
        print("after %d bench steps (%d MD steps): largest |difference| / max |value|: %s; ions whose tPart differs (a quantum jump "
              "in one build only): %d" % (steps, 40 * steps, " ".join("%s %.3e" % kv for kv in rel.items()), int((ta != tb).sum())))


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        compare(sys.argv[2])
    else:
        forces(sys.argv[1])
