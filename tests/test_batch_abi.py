"""CPU tests of replica batches (erirt_create_batch): the entry point is declared and exported, and its argument checks and the
unsupported configurations are refused before any CUDA call."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from erirt_b200 import _lib
    return _lib.load()


def _cfg(model="RtIrt", person_trace=0):
    from erirt_b200 import _lib
    c = _lib.Config()
    c.abi_version = _lib.ABI_VERSION
    c.model = _lib.MODELS[model]
    c.n_subj = c.n_subj_total = 10
    c.n_item, c.n_feat, c.n_iter, c.n_chain, c.n_burnin = 3, 1, 4, 1, 2
    c.q_rt, c.dtype, c.person_trace = 0.5, _lib.F64, person_trace
    return c


def _create(lib, cfg, n_batch):
    h = ctypes.c_void_p()
    rc = lib.erirt_create_batch(ctypes.byref(cfg), n_batch, ctypes.byref(h))
    assert not h.value
    return rc, lib.erirt_last_error().decode()


def test_create_batch_is_declared_exported_and_bound(lib):
    from erirt_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "erirt_b200.h")).read()
    assert re.search(r"int erirt_create_batch\(const erirt_config\* cfg, int32_t n_batch, erirt_handle\*\* out\);", hdr)
    assert hasattr(lib, "erirt_create_batch")
    assert "erirt_create_batch" in _lib.EXPORTED


@pytest.mark.parametrize("n_batch", [0, -1, 65536])
def test_n_batch_out_of_range_is_an_argument_error(lib, n_batch):
    rc, msg = _create(lib, _cfg(), n_batch)
    assert rc == -1 and "n_batch" in msg


@pytest.mark.parametrize("model", ["RtIrtCross", "RtIrtCrossQr"])
def test_cross_family_batches_are_unsupported_before_cuda(lib, model):
    rc, msg = _create(lib, _cfg(model), 2)
    assert rc == -5 and "Cross" in msg


def test_person_trace_batches_are_unsupported_before_cuda(lib):
    rc, msg = _create(lib, _cfg(person_trace=1), 3)
    assert rc == -5 and "person_trace" in msg


def _models(kind, n, data=None, **cond):
    from erirt_b200 import api, structs
    C = structs.setCond(**{**dict(nSubj=20, nItem=4, nFeat=1, nIter=10, nChain=1), **cond})
    out = []
    for r in range(n):
        rng = np.random.default_rng(r)
        D = data if data is not None else structs.InputData(Y=rng.random((20, 4)) < 0.5, X=rng.normal(size=(20, 1)),
                                                            T=np.exp(rng.normal(size=(20, 4))))
        out.append(getattr(api, kind)(C, Data=D, rng=r))
    return out


def test_sample_batch_rejects_mixed_inputs_before_the_gpu(lib):
    from erirt_b200 import api, simulate, structs
    with pytest.raises(ValueError, match="one type"):
        api.sampleBatch(_models("GibbsRtIrt", 1) + _models("GibbsRtIrtNull", 1))
    with pytest.raises(ValueError, match="equal Cond"):
        api.sampleBatch(_models("GibbsRtIrt", 1) + _models("GibbsRtIrt", 1, nIter=12))
    with pytest.raises(ValueError, match="Cross"):
        api.sampleBatch(_models("GibbsRtIrtCross", 2))
    with pytest.raises(ValueError, match="person_trace"):
        api.sampleBatch(_models("GibbsRtIrt", 2), person_trace=True)
    with pytest.raises(ValueError, match="at least one"):
        api.sampleBatch([])
    mixed = _models("GibbsRtIrt", 2)
    mixed[1].Data = simulate.DeviceData(structs.InputPara(), None, "tnorm", 5)
    with pytest.raises(ValueError, match="mixed host and device"):
        api.sampleBatch(mixed)


@pytest.mark.parametrize("kw", [{}, {"person_trace": True}, {"person_trace": None}])
def test_batched_run_simulation_needs_person_trace_off_before_the_gpu(lib, kw):
    """A batch keeps no person trace, which changes the Diag counts and D-hat of runSimulation: batch=k with the default (or any
    other) person_trace is refused before any GPU work instead of returning a different Dict."""
    from erirt_b200 import simtools, simulate, structs
    C = structs.setCond(nSubj=20, nItem=4, nFeat=1, nIter=10, nChain=1, nRep=2)
    with pytest.raises(ValueError, match="person_trace=False"):
        simtools.runSimulation(C, simulate.setTrueParaRtIrt(C, rng=1), batch=2, rank=0, world=1, device=0, **kw)
