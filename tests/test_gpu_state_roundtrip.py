"""erirt_set_state -> erirt_get_state, field by field: the person vectors, the N x J tiles (omega, CrossQr's nu) and the item /
structural parameters come back as set, in the storage precision of each."""
import ctypes as C

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]

N, J, F = 300, 13, 2
# one model of each family: item response only, regression, Latent, Cross (the two Qr models also carry nu)
FAMILY_MODELS = ["MlIrt", "RtIrt", "RtIrtLatentQr", "RtIrtCrossQr"]


@pytest.fixture(scope="module")
def E():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import erirt_b200
    erirt_b200._lib.load()
    return erirt_b200


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("model", FAMILY_MODELS)
def test_set_state_get_state_roundtrip(E, model, dtype):
    rng = np.random.default_rng(41)
    eng = E.Engine(model, N, J, F, n_iter=2, dtype=dtype, use_graph=False)
    cell = model == "RtIrtCrossQr"
    nb = {"MlIrt": F + 1, "RtIrt": 2 * (F + 1), "RtIrtLatentQr": F + 2}.get(model, 0)
    person = {"theta": (N,), "zeta": (N,), "nu": (N, J) if cell else (N,), "omega": (N, J)}
    params = {"a": J, "b": J, "lambda": J, "sigma2": J, "rho": J, "Sigma": 4}
    if nb:
        params["beta"] = nb
    want = {k: rng.normal(size=s) for k, s in person.items()}
    want.update({k: rng.normal(size=n) for k, n in params.items()})
    want["Sigma"] = want["Sigma"].reshape(2, 2)
    eng.set_state(**want)
    for k, v in want.items():
        got = eng.get_state(k)
        assert got.shape == v.shape, k
        if k in person and dtype == "f32":  # person and tile fields are stored in the engine's precision
            v = v.astype(np.float32).astype(np.float64)
        assert np.array_equal(got, v), f"{model} {dtype}: {k} does not come back as set"
    # a wrong length is refused in both directions
    lib, fields = eng.lib, E._lib.FIELDS
    for k, v in want.items():
        buf = np.zeros(v.size + 1)
        p = buf.ctypes.data_as(C.POINTER(C.c_double))
        assert lib.erirt_set_state(eng.h, fields[k], p, v.size + 1) == -1, k
        assert lib.erirt_get_state(eng.h, fields[k], p, v.size - 1) == -1, k
    eng.close()
