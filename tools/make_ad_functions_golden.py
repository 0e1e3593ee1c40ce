"""Generate the reference's results of the AD tests, from the unmodified reference's ``AdArray``:

* tests/golden/ad_functions.npz: value and Jacobian of ``pp.ad.functions`` (and ``AdArray.__pow__``) on the random
  ``AdArray``s ``cases()`` of tests/test_ad_functions.py, one entry per check of ``run_checks`` there;
* tests/golden/ad_adarray.npz: the expression of tests/test_zz_ad_gpu.py on ``adarray_case()``.

Run where the reference is importable:  python tools/make_ad_functions_golden.py"""
from __future__ import annotations

import os
import sys

import numpy as np
import scipy.sparse as sps

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (HERE, ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
from ref_loader import load_porepy  # noqa: E402
from make_mdflow_golden import put_csr  # noqa: E402
from test_ad_functions import GOLDEN, cases  # noqa: E402
from test_zz_ad_gpu import GOLDEN_ADARRAY, adarray_case  # noqa: E402

pp = load_porepy()


def main():
    f, A = pp.ad.functions, pp.ad.AdArray
    cs = cases()
    x = {k: A(v.copy(), j.copy()) for k, (v, j) in cs.items()}
    l2 = f.l2_norm(3, x["c"])
    results = {
        "exp": f.exp(x["a"]), "log": f.log(x["pos"]), "abs": f.abs(x["a"]), "sin": f.sin(x["a"]),
        "cos": f.cos(x["a"]), "tanh": f.tanh(x["a"]), "pow": x["pos"] ** 2.5, "sqrt": x["pos"] ** 0.5,
        "heaviside": f.heaviside(0.5, x["c"]), "heaviside_smooth": f.heaviside_smooth(x["a"], 1e-2),
        "characteristic": f.characteristic_function(1e-10, x["c"]),
        "maximum_ad_ad": f.maximum(x["a"], x["b"]), "maximum_ad_array": f.maximum(x["a"], cs["b"][0]),
        "maximum_array_ad": f.maximum(cs["b"][0], x["a"]), "maximum_ad_scalar": f.maximum(x["a"], 0.1),
        "l2_norm": l2, "l2_norm_dim1": f.l2_norm(1, x["a"]),
        # compositions of the kind the friction law uses: b (f_max - ||t||) clipped at zero
        "composition": f.maximum(x["pos"] - l2.val.mean(), 0.0) * f.exp(x["a"]),
    }
    d = {}
    for label, r in results.items():
        if isinstance(r, A):
            d[label + "__val"] = np.asarray(r.val, dtype=np.float64)
            put_csr(d, label + "__jac", r.jac)
        else:
            d[label + "__val"] = np.asarray(r, dtype=np.float64)
    np.savez_compressed(GOLDEN, **d)
    print(GOLDEN, len(results), "checks")

    v1, v2, M, N, w = adarray_case()
    n1, n2 = v1.size, v2.size
    h1 = A(v1, sps.hstack([sps.identity(n1), sps.csr_matrix((n1, n2))]).tocsr())
    h2 = A(v2, sps.hstack([sps.csr_matrix((n2, n1)), sps.identity(n2)]).tocsr())
    ref = (M @ h1) * (N @ h2) + 3.0 * (M @ h1) - (N @ h2) * w + 2.5
    ref = -ref + (M @ h1) * (M @ h1)
    d = {"val": np.asarray(ref.val, dtype=np.float64)}
    put_csr(d, "jac", ref.jac)
    np.savez_compressed(GOLDEN_ADARRAY, **d)
    print(GOLDEN_ADARRAY)


if __name__ == "__main__":
    main()
