"""Thin object wrapper over the C ABI: one Engine == one erirt_handle (one chain, one person shard of a chain, or a batch of
n_batch independent replicas of one configuration, erirt_create_batch)."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import ErirtError, check  # noqa: F401


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class Engine:
    def __init__(self, model, n_subj, n_item, n_feat=0, *, n_iter=5000, n_chain=1, n_burnin=None, q_rt=0.5,
                 intercept=False, itemtype="2pl", cov2one=True, dtype="f32", seed=1234, chain=0, compat=0,
                 person_trace=False, device=0, use_graph=True, n_subj_total=None, subj_offset=0, time_kernels=False,
                 nu_cell_moments=False, n_batch=1):
        """n_batch > 1: a replica batch (include/erirt_b200.h, erirt_create_batch).  Inputs stack the replicas (person matrices as
        n_batch * n_subj rows, or arrays with a leading replica axis) and the getters return arrays with a leading replica axis;
        replica r samples the chain of a standalone engine with seed + r."""
        if itemtype not in ("1pl", "2pl"):
            # same text as the reference's sample! (src/GibbsRtIrt.pl.jl:212-214)
            raise ValueError("Invalid input: the item type must be '1pl' or '2pl'.")
        L = _lib.load()
        self.lib = L
        mid = _lib.MODELS[model] if isinstance(model, str) else int(model)
        cfg = _lib.Config()
        cfg.abi_version = _lib.ABI_VERSION
        cfg.model = mid
        cfg.n_subj = n_subj
        cfg.n_subj_total = n_subj if n_subj_total is None else n_subj_total
        cfg.subj_offset = subj_offset
        cfg.n_item, cfg.n_feat = n_item, n_feat
        cfg.n_iter, cfg.n_chain = n_iter, n_chain
        cfg.n_burnin = int(round(n_iter / 2)) if n_burnin is None else n_burnin
        cfg.q_rt = q_rt
        cfg.intercept, cfg.itemtype_1pl, cfg.cov2one = int(intercept), int(itemtype == "1pl"), int(cov2one)
        cfg.dtype = {"f32": _lib.F32, "f64": _lib.F64}[dtype]
        cfg.seed, cfg.chain, cfg.compat = seed, chain, compat
        cfg.person_trace, cfg.device, cfg.use_graph = int(person_trace), device, int(use_graph)
        cfg.time_kernels = int(time_kernels)
        cfg.nu_cell_moments = int(nu_cell_moments)
        self.cfg = cfg
        self.model = mid
        self.N, self.J, self.F = n_subj, n_item, n_feat
        self.B = int(n_batch)
        self.h = C.c_void_p()
        if self.B == 1:
            check(L.erirt_create(C.byref(cfg), C.byref(self.h)))
        else:
            check(L.erirt_create_batch(C.byref(cfg), self.B, C.byref(self.h)))

    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            self.lib.erirt_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- data / state ----
    def set_data(self, Y, logT=None, X=None):
        """Host matrices as Julia holds them.  A bool / uint8 Y (Julia's Matrix{Bool}) goes through erirt_set_data_y8 as it
        lies in memory; anything else is passed as column-major float64."""
        Y = self._rows(Y)
        y8 = Y.dtype in (np.bool_, np.uint8)
        Y = np.asfortranarray(Y, dtype=np.uint8 if y8 else np.float64)
        assert Y.shape == (self.B * self.N, self.J), Y.shape
        T = np.asfortranarray(self._rows(logT), dtype=np.float64) if logT is not None else None
        Xf = np.asfortranarray(self._rows(X), dtype=np.float64) if (X is not None and self.F > 0) else None
        fn = self.lib.erirt_set_data_y8 if y8 else self.lib.erirt_set_data
        check(fn(self.h, Y.ctypes.data, Y.shape[0], T.ctypes.data if T is not None else None,
                 T.shape[0] if T is not None else 0, Xf.ctypes.data if Xf is not None else None,
                 Xf.shape[0] if Xf is not None else 0))

    def _rows(self, M):
        """A batch's person matrix: (n_batch, N, ...) stacked to (n_batch * N, ...) rows; anything else as given."""
        M = np.asarray(M)
        return M.reshape((-1,) + M.shape[2:]) if (self.B > 1 and M.ndim == 3) else M

    def generate_data(self, theta, a, b, zeta=None, lambda_=None, sigma2=None, rho=None, X=None, error="unit", seed=1234):
        """The N x J part of setData* (src/SimTools.jl:117-368) on the device, straight into the packed layout (erirt_generate_data).
        error: "tnorm" (Null / RtIrt), "unit" (Latent*), "norm" / "tail" / "skew" (Cross).  A batch takes n_batch * N person values
        and n_batch * J item values (or arrays with a leading replica axis); replica r uses data seed seed + r."""
        def vec(v, n):
            if v is None:
                return None
            v = np.ascontiguousarray(np.asarray(v, dtype=np.float64).ravel())
            assert v.size == n, (v.size, n)
            return v
        th, ze = vec(theta, self.B * self.N), vec(zeta, self.B * self.N)
        av, bv, lv, sv, rv = (vec(v, self.B * self.J) for v in (a, b, lambda_, sigma2, rho))
        Xf = np.asfortranarray(self._rows(X), dtype=np.float64) if (X is not None and self.F > 0) else None
        p = lambda v: _dp(v) if v is not None else None  # noqa: E731
        check(self.lib.erirt_generate_data(self.h, p(th), p(ze), p(av), p(bv), p(lv), p(sv), p(rv), p(Xf), Xf.shape[0] if Xf is not None else 0,
                                           _lib.ERROR_TYPES[error], seed))

    def get_data(self):
        """(Y, logT) held by the engine, column-major float64 (logT is None for MlIrt); a batch: (n_batch, N, J) each."""
        n = self.B * self.N
        Y = np.empty((n, self.J), dtype=np.float64, order="F")
        T = np.empty((n, self.J), dtype=np.float64, order="F") if self.model != 0 else None
        check(self.lib.erirt_get_data(self.h, _dp(Y), n, _dp(T) if T is not None else None, n))
        if self.B > 1:
            return Y.reshape(self.B, self.N, self.J), (T.reshape(self.B, self.N, self.J) if T is not None else None)
        return Y, T

    def set_data_device(self, dY_ptr, ldY, dlogT_ptr, ldT, dX_ptr, ldX):
        """Column-major float64 buffers already on this engine's device (e.g. torch tensors' data_ptr())."""
        check(self.lib.erirt_set_data_device(self.h, dY_ptr, ldY, dlogT_ptr, ldT, dX_ptr, ldX))

    _PERSON = ("theta", "zeta", "nu", "omega")

    def set_state(self, **fields):
        """A batch takes each field in one form only: a sequence (or an array with a leading axis) of n_batch per-replica values,
        each in its standalone form."""
        for k, v in fields.items():
            if v is None:
                continue
            if self.B > 1:
                if np.ndim(v) < 1 or len(v) != self.B:
                    raise ValueError(f"set_state({k}=...) of a batch of {self.B}: pass one value per replica (leading axis of length {self.B})")
                if k.rstrip("_") in self._PERSON:  # n_batch * N rows, column-major
                    v = np.concatenate([np.asarray(x, dtype=np.float64).reshape(self.N, -1, order="F") for x in v], axis=0)
                else:  # n_batch consecutive blocks of the standalone layout
                    v = np.concatenate([np.asarray(x, dtype=np.float64).ravel(order="F") for x in v])
            a = np.ascontiguousarray(np.asarray(v, dtype=np.float64).ravel(order="F"))
            check(self.lib.erirt_set_state(self.h, _lib.FIELDS[k.rstrip("_")], _dp(a), a.size))

    def get_state(self, name):
        fid = _lib.FIELDS[name]
        n = {"theta": self.N, "zeta": self.N, "nu": self.N * self.J if self.model == 4 else self.N, "omega": self.N * self.J, "a": self.J, "b": self.J,
             "lambda": self.J, "sigma2": self.J, "rho": self.J, "Sigma": 4,
             "beta": {0: self.F + 1, 1: 2 * (self.F + 1), 2: 2 * (self.F + 1), 5: self.F + 2, 6: self.F + 2}.get(self.model, 0)}[name]
        B = self.B
        out = np.empty(n * B, dtype=np.float64)
        check(self.lib.erirt_get_state(self.h, fid, _dp(out), n * B))
        if B > 1:
            if name == "omega":
                return out.reshape((B * self.N, self.J), order="F").reshape(B, self.N, self.J)
            if name in self._PERSON:
                return out.reshape(B, self.N)
            return out.reshape(B, 2, 2).transpose(0, 2, 1) if name == "Sigma" else out.reshape(B, n)
        if name == "omega" or (name == "nu" and self.model == 4):
            return out.reshape((self.N, self.J), order="F")
        if name == "Sigma":
            return out.reshape((2, 2), order="F")
        return out

    # ---- sampling ----
    def sample(self, n_sweeps):
        check(self.lib.erirt_sample(self.h, int(n_sweeps)))

    def loglik_current(self):
        """getLogLikelihood* of the state currently held by the engine (no draws); a batch: (n_batch,) values."""
        out = np.empty(self.B, dtype=np.float64)
        check(self.lib.erirt_loglik_current(self.h, _dp(out)))
        return out if self.B > 1 else float(out[0])

    def trace_width(self, which):
        return int(self.lib.erirt_trace_width(self.h, _lib.TRACES[which]))

    def get_trace(self, which, first_col=0, n_cols=None):
        """Julia-layout array (nIter, n_cols, nChain) of Post.<which>[:, first_col:first_col+n_cols, :]; a batch: (n_batch, nIter,
        n_cols, nChain)."""
        W = self.trace_width(which)
        if n_cols is None:
            n_cols = W - first_col
        shape = (self.cfg.n_iter, n_cols, self.cfg.n_chain) + ((self.B,) if self.B > 1 else ())
        out = np.empty(shape, dtype=np.float64, order="F")
        check(self.lib.erirt_get_trace(self.h, _lib.TRACES[which], first_col, n_cols, _dp(out)))
        return np.moveaxis(out, 3, 0) if self.B > 1 else out

    def get_moments(self, name, out=None):
        """Post-burn-in mean and SD of theta / zeta / nu.  out: optional (mean, sd) float64 arrays to fill (e.g. views of pinned memory)."""
        cell = name == "nu" and self.model == 4  # CrossQr: N x J weights (needs nu_cell_moments=True)
        n = (self.N * self.J if cell else self.N) * self.B
        mean, sd = out if out is not None else (np.empty(n), np.empty(n))
        assert mean.dtype == np.float64 and sd.dtype == np.float64 and mean.size == n and sd.size == n
        check(self.lib.erirt_get_moments(self.h, _lib.FIELDS[name], _dp(mean), _dp(sd), n))
        if self.B > 1 and out is None:  # (n_batch, N)
            return mean.reshape(self.B, self.N), sd.reshape(self.B, self.N)
        if cell and out is None:
            return mean.reshape((self.N, self.J), order="F"), sd.reshape((self.N, self.J), order="F")
        return mean, sd

    def trace_ess_rhat(self, which, first_col=0, n_cols=None, skip=0):
        """Rank-normalised split bulk ESS and R-hat of columns [first_col, first_col + n_cols) of Post.<which>, iterations after the
        first `skip` (checkConvergence, src/SimTools.jl:419-443), computed by a CUDA kernel on the traces where they lie
        (erirt_trace_ess_rhat, csrc/diagnostics.cuh).  Returns (ess, rhat), NaN for constant columns."""
        w = int(self.lib.erirt_trace_width(self.h, _lib.TRACES[which]))
        if n_cols is None:
            n_cols = w - first_col
        ess, rhat = np.empty(n_cols * self.B), np.empty(n_cols * self.B)
        check(self.lib.erirt_trace_ess_rhat(self.h, _lib.TRACES[which], first_col, n_cols, skip, _dp(ess), _dp(rhat)))
        if self.B > 1:  # (n_batch, n_cols)
            return ess.reshape(self.B, n_cols), rhat.reshape(self.B, n_cols)
        return ess, rhat

    # ---- checkpoint / resume ----
    def checkpoint(self) -> np.ndarray:
        """State, auxiliaries, Philox sweep counter, running moments and traces of the chain as one byte array."""
        n = int(self.lib.erirt_checkpoint_size(self.h))
        if n < 0:
            check(n)  # the size call returns the error code
        buf = np.empty(n, dtype=np.uint8)
        check(self.lib.erirt_checkpoint_save(self.h, buf.ctypes.data, n))
        return buf

    def restore(self, buf):
        """Continue the chain a checkpoint() was taken from (same configuration; call set_data first)."""
        buf = np.ascontiguousarray(np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf)
        check(self.lib.erirt_checkpoint_load(self.h, buf.ctypes.data, buf.size))

    def stats(self):
        s = _lib.Stats()
        check(self.lib.erirt_get_stats(self.h, C.byref(s)))
        return {f[0]: getattr(s, f[0]) for f in _lib.Stats._fields_}

    def check_guards(self) -> int:
        """Guard bytes overwritten since erirt_create (handles created with ERIRT_GUARDS=1 in the environment); -1 without guards."""
        return int(self.lib.erirt_debug_check_guards(self.h))

    # ---- multi-GPU ----
    def comm_init(self, rank, world, unique_id=None):
        """unique_id: 128 bytes of an NCCL id (ncclAllReduce exchange), or None when the peer exchange is attached next."""
        buf = C.create_string_buffer(unique_id, 128) if unique_id is not None else None
        check(self.lib.erirt_comm_init(self.h, rank, world, buf))

    def peer_export(self) -> bytes:
        """Allocate this GPU's exchange buffer of the fused one-shot all-reduce and return its 64-byte CUDA IPC handle."""
        buf = C.create_string_buffer(64)
        check(self.lib.erirt_peer_export(self.h, buf))
        return buf.raw

    def peer_detach(self):
        """Unmap the peers' exchange buffers (all ranks, then a host barrier, then close())."""
        check(self.lib.erirt_peer_detach(self.h))

    def peer_attach(self, handles: bytes):
        """Map the peers' exchange buffers (world x 64 bytes of IPC handles, in rank order)."""
        buf = C.create_string_buffer(handles, len(handles))
        check(self.lib.erirt_peer_attach(self.h, buf))


def trim_pool(device=0):
    """Return the device memory the library's stream-ordered pool kept from destroyed engines to the driver."""
    check(_lib.load().erirt_trim_pool(device))


def nccl_unique_id() -> bytes:
    L = _lib.load()
    buf = C.create_string_buffer(128)
    check(L.erirt_nccl_unique_id(buf))
    return buf.raw


# ---- parity entry points ----
def k_pg(z, seed=1234, chain=0, sweep=1, row0=0, dtype="f64", device=0):
    L = _lib.load()
    z = np.ascontiguousarray(z, dtype=np.float64)
    rows, cols = z.shape
    out = np.empty_like(z)
    check(L.erirt_k_pg(_dp(z), rows, cols, row0, seed, chain, sweep, {"f32": 0, "f64": 1}[dtype], device, _dp(out)))
    return out


def k_nu_person(mu, lam, seed=1234, chain=0, sweep=1, row0=0, dtype="f64", device=0):
    L = _lib.load()
    mu = np.ascontiguousarray(mu, dtype=np.float64)
    out = np.empty_like(mu)
    check(L.erirt_k_nu_person(_dp(mu), lam, mu.size, row0, seed, chain, sweep, {"f32": 0, "f64": 1}[dtype], device,
                              _dp(out)))
    return out


def k_philox(ctr, key, device=0):
    L = _lib.load()
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    check(L.erirt_k_philox(c, k, device, o))
    return [int(v) for v in o]
