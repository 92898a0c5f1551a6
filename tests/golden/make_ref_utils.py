"""Golden vectors from the reference's own Python helpers (swarm_localization/scripts/utils.py): `quat2eulers` -- the Euler
convention the C++ side shares through swarm_msgs, which is not in the tree -- and `wrap_pi`.  The two functions are
executed where they lie under /root/reference (their module imports the `transformations` package, which is not installed
here, so only these function definitions are compiled); nothing is copied into the repository.

    python tests/golden/make_ref_utils.py        -> tests/golden/ref_utils.npz
    python tests/golden/make_ref_utils.py --check   compare the committed fixture with the functions instead of writing it
"""
import ast
import math
import os
import sys

import numpy as np

SRC = "/root/reference/swarm_localization/scripts/utils.py"
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_utils.npz")


def reference_functions(names=("quat2eulers", "wrap_pi")):
    tree = ast.parse(open(SRC).read(), SRC)
    keep = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in names]
    assert len(keep) == len(names)
    ns = {"np": np}
    ns.update({k: getattr(math, k) for k in ("atan2", "asin", "pi")})
    exec(compile(ast.Module(body=keep, type_ignores=[]), SRC, "exec"), ns)
    return [ns[n] for n in names]


def main(check=False):
    quat2eulers, wrap_pi = reference_functions()
    rng = np.random.default_rng(0)
    q = rng.standard_normal((200, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)                     # wxyz
    ypr = np.array([quat2eulers(*row) for row in q])                  # the reference returns (yaw, pitch, roll)
    a = rng.uniform(-20, 20, 200)
    out = dict(quat_wxyz=q, ypr=ypr, angle=a, wrapped=wrap_pi(a))
    if check:
        z = np.load(OUT)
        assert sorted(z.files) == sorted(out) and all(np.array_equal(z[k], v) for k, v in out.items()), \
            "tests/golden/ref_utils.npz differs from the reference's functions"
        print("ref_utils.npz matches the reference's functions")
        return
    np.savez(OUT, **out)
    print("wrote", OUT)


if __name__ == "__main__":
    main(check="--check" in sys.argv[1:])
