"""CPU-side checks of the reference's solver steps update_u, update_alpha and frank_wolfe_nmf in the drop-in module: they are
exported with the reference's positional arity, and without a GPU they refuse instead of computing on the host."""
import inspect

import numpy as np
import pytest

ARITY = {"update_u": 11, "update_alpha": 9, "frank_wolfe_nmf": 8}


def test_steps_are_exported_with_reference_arity():
    from demethify_b200 import deconvolution as dec
    for name, n in ARITY.items():
        assert name in dec.__all__
        params = inspect.signature(getattr(dec, name)).parameters.values()
        assert len(params) == n and all(p.default is p.empty and p.kind == p.POSITIONAL_OR_KEYWORD for p in params)


def _inputs():
    rs = np.random.RandomState(0)
    M, N, K, n_u = 8, 3, 2, 1
    X, D = rs.uniform(size=(M, N)), np.ones((M, N))
    Rk, u = rs.uniform(size=(M, K)), rs.uniform(size=(M, n_u))
    A = rs.dirichlet(np.ones(K + n_u), N).T
    return X, D, Rk, u, A, n_u


def test_steps_raise_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from demethify_b200 import _lib
    from demethify_b200 import deconvolution as dec
    X, D, Rk, u, A, n_u = _inputs()
    with pytest.raises(_lib.DmfError):
        dec.update_u(u, A, 2, 1.0, 1.0, 1.0, u, X, Rk, n_u, D)
    with pytest.raises(_lib.DmfError):
        dec.update_alpha(2, A, 1.0, 1.0, 1.0, A, np.c_[Rk, u], D, X)
    with pytest.raises(_lib.DmfError):
        dec.frank_wolfe_nmf(Rk, u, X, A[:-n_u], A[-n_u:], np.full(X.shape[1], 0.5), 2, D)
