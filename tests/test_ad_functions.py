"""``porepy_b200.ad_functions`` against the reference's ``pp.ad.functions`` / ``AdArray.__pow__`` on random ``AdArray``s
(value and Jacobian), incl. the tie rule of ``maximum`` and the zero-vector rule of ``l2_norm``.  The reference's results
are stored in tests/golden/ad_functions.npz (tools/make_ad_functions_golden.py).
CPU: the scipy stand-in for the device sparse algebra; GPU leg at the end of the suite."""
import os

import numpy as np
import scipy.sparse as sps

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ad_functions.npz")


def cases(n=24, m=40, seed=0):
    rng = np.random.default_rng(seed)

    def jac():
        return sps.random(n, m, 0.2, format="csr", random_state=int(rng.integers(1 << 30)), data_rvs=rng.standard_normal)
    a, b = rng.standard_normal(n), rng.standard_normal(n)
    b[:4] = a[:4]                                      # ties: maximum takes the first argument
    c = rng.standard_normal(n)
    c[3:6] = 0.0                                       # one vanishing 3-vector for l2_norm
    pos = 0.5 + rng.random(n)
    return dict(a=(a, jac()), b=(b, jac()), c=(c, jac()), pos=(pos, jac()))


def reference_results():
    """label -> (value, Jacobian or None) of the reference on ``cases()``."""
    d = np.load(GOLDEN)
    out = {}
    for key in d.files:
        if key.endswith("__val"):
            j = key[:-5] + "__jac"
            out[key[:-5]] = (d[key], sps.csr_matrix((d[j + "__data"], d[j + "__indices"], d[j + "__indptr"]),
                                                    shape=tuple(d[j + "__shape"])) if j + "__data" in d.files else None)
    return out


def run_checks(make, fn, to_host):
    """``make(val, jac)`` builds the device array; ``fn`` is porepy_b200.ad_functions."""
    ref = reference_results()
    cs = cases()
    dev = {k: make(v, j) for k, (v, j) in cs.items()}
    checked = set()

    def same(what, g):
        rv, rj = ref[what]
        gv, gj = to_host(g)
        assert np.allclose(gv, rv, rtol=1e-13, atol=1e-13), what
        if rj is not None:
            d = abs(rj - sps.csr_matrix(gj))
            assert (d.max() if d.nnz else 0.0) <= 1e-12 * max(abs(rj).max(), 1.0), what
        checked.add(what)
    same("exp", fn.exp(dev["a"]))
    same("log", fn.log(dev["pos"]))
    same("abs", fn.abs(dev["a"]))
    same("sin", fn.sin(dev["a"]))
    same("cos", fn.cos(dev["a"]))
    same("tanh", fn.tanh(dev["a"]))
    same("pow", fn.power(dev["pos"], 2.5))
    same("sqrt", fn.sqrt(dev["pos"]))
    same("heaviside", fn.heaviside(0.5, dev["c"]))
    same("heaviside_smooth", fn.heaviside_smooth(dev["a"], 1e-2))
    same("characteristic", fn.characteristic_function(1e-10, dev["c"]))
    same("maximum_ad_ad", fn.maximum(dev["a"], dev["b"]))
    same("maximum_ad_array", fn.maximum(dev["a"], cs["b"][0]))
    same("maximum_array_ad", fn.maximum(cs["b"][0], dev["a"]))
    same("maximum_ad_scalar", fn.maximum(dev["a"], 0.1))
    same("l2_norm", fn.l2_norm(3, dev["c"]))
    same("l2_norm_dim1", fn.l2_norm(1, dev["a"]))
    # compositions of the kind the friction law uses: b (f_max - ||t||) clipped at zero
    g = fn.maximum(dev["pos"] - float(ref["l2_norm"][0].mean()), 0.0) * fn.exp(dev["a"])
    same("composition", g)
    assert checked == set(ref)


def test_functions_match_the_reference_host_build(monkeypatch):
    import torch
    import emu_sparse
    from porepy_b200 import ad, ad_functions
    emu_sparse.install(monkeypatch)

    def make(v, j):
        return ad.DeviceAdArray(torch.as_tensor(v.copy()), emu_sparse.HostCsr(j))

    def to_host(g):
        if isinstance(g, ad.DeviceAdArray):
            return g.val.numpy(), g.jac.to_scipy()
        return g.numpy(), None
    run_checks(make, ad_functions, to_host)
