"""`Corex`: the sklearn-style Linear CorEx model of gregversteeg/LinearCorex, B200-native.

Drop-in for `linearcorex.Corex` (reference linearcorex/linearcorex.py:22-455): same constructor
keywords and defaults (:72-74), `fit` / `fit_transform` / `transform` / `predict` / `invert` /
`get_covariance` / `clusters()` / `tc` / `tcs` / `mis`, attributes `ws`, `moments`, `theta`,
`history`, `eps`, `m`, `n_samples`, `nv`, `n_obs`, global-RNG seeding (:89, :116) and warm start
(:114).  This file is host control flow only: every array operation runs in liblcx_b200.so
(hand-written sm_100a CUDA behind the C ABI of include/lcx_b200.h); torch owns the device
buffers and, for multi-GPU runs, supplies `torch.distributed`.  Only O(1) scalars (TC, max uj,
update_tangent) cross to the host inside the loop, at the points where the reference branches
on them (:250, :306, :327, :144, :152).

There is no CPU fallback.  If the CUDA library or a CUDA device is missing, construction of the
device session raises.

Extensions over the reference signature (all keyword-only in spirit, defaults keep reference
behaviour):
  eliminate_synergy   README/docstring name of `discourage_overlap` (README.md:32)
  precision           'fp64': all arithmetic binary64 (DMMA tensor-core contractions), parity target = the
                      reference's numpy float64 path.
                      'fp64_split' (default): the two X contractions run as exact int8 digit products on tcgen05
                      (6 radix-254 digits = 48 bits below max |X~| for the data -- one exponent for all of X~, which is
                      standardised -- and below each row / column maximum for W, grad and Y; truncation at the level of
                      binary64 rounding, measured parity 1e-11), everything else binary64.
                      'fp64_split5': 5 digits (40 bits), 30 % faster, parity 1e-9 on fits up to ~700 iterations.
                      'fp64_split7': 7 digits (56 bits, finer than binary64's significand), ~1.4x the cost of the
                      default; for ill-conditioned fits (pure-noise data, extreme outliers) that amplify the 48-bit
                      mode's perturbation past 1e-9.
                      'fast': 3 digits (24 bits, fp32-equivalent products; opt-in, 1e-4 tolerance).
                      'auto' (default): 'fp64_split', except for problems so small (N n m < 3e7: the README demo, big5,
                      adni) that an iteration is launch-bound -- there 'fp64' (DMMA) has fewer launches and is
                      10-50 % quicker (tools/small_configs.py) -- and except with gaussianize='none', where columns keep
                      their own scales and the single exponent of X~ would short-change small ones (also 'fp64').
                      Both are FP64-faithful; `precision_used` tells which ran.
  algorithm           'stream': every pass pair reads X~ (Y = X~ A^T, then X~^T Y), the reference's own formulation, which
                      it chose for n >> N (:197-198).  'gram': the fit only ever needs X~^T X~ / N, so that n x n matrix
                      is formed ONCE on the int8 tcgen05 engine (exact digit products) and every pass pair becomes one
                      n x n x m product -- independent of the number of samples, and with no exchange between ranks
                      after the one-off sum of the matrix.  Split precisions only.  'auto' (default): 'gram' when
                      N >= n, the problem is large enough to be bound by the passes over X (N n m >= 1e9) and the matrix
                      fits; `algorithm_used` tells which ran.
  exact_trials        False (default): backtracking trials are evaluated through the linearity of
                      `_sig` (rho(W + eta U) = rho(W) + eta _sig(U)) -- one pass pair over X per
                      iteration instead of one per trial (SURVEY.md 7.8).  True: every trial
                      re-reads X exactly like linearcorex.py:321.
  input_dtype         'float64' (default) keeps the input as given (the float64 reference path);
                      'float32' reproduces the reference's cast at :108 and :116.
  comm                None, or a torch.distributed process group / True for the default group:
                      `fit(x)` then takes this rank's row block of X (sample sharding).
  stream_rows         split modes: prepare X in row blocks of this many rows (three streaming passes over the raw
                      input, X~ never materialised in fp64).  Default: automatic when X~ would not fit -- this is
                      what lets the 1M x 20k x 100 target run on ONE B200 (120 GB of int8 digit planes).

Methods beyond the reference (sklearn's covariance-estimator interface; discourage_overlap=True models with theta):
  score_samples(x)    log N(x_l; theta[0], get_covariance()) per row, in the units of the input (g() of 'outliers' is not
                      applied: it is the density of the covariance estimate itself)
  score(x)            their mean (over all ranks' rows with `comm`); with sample_weight, the weighted mean
  mahalanobis(x)      squared Mahalanobis distances under the same Gaussian
  get_precision()     the inverse of get_covariance(), in row blocks, with get_covariance's output options
  impute(x)           conditional means E[x_M | x_O] of the missing entries; return_std=True adds their conditional
                      standard deviations
  sample_missing(x)   multiple imputation: draws of the missing entries from their conditional distribution
  sample(n_samples)   draws from N(theta[0], get_covariance()), reproducible per (seed, row) and splittable by `first_row`
  conditional(obs)    a ConditionalGaussian given a fixed set of observed columns: predict, std, get_covariance, sample and
                      the marginal score of the observed columns, one factor per pattern and a scoring pass per row
The estimate is low rank plus diagonal, S (Z^T Z + Delta) S, so none of these forms or factors an n x n matrix: a factor
B = G^-1 Z Delta^-1 (m x n) is built from the moments on each call and a row costs O(n m), in binary64 on the DMMA engine
(conditioning: one SPD system of order |M| or m per row).  Random draws come from counter-based Philox4x32-10 normals, so
they do not depend on how rows are blocked.
Inputs are handled as by transform (containers, row providers, imputation of missing entries with the new data's means).

Per-row sample weights: `fit(x, sample_weight=w)` (also fit_transform, hierarchy.fit_layers) estimates everything from the
w-weighted averages over rows -- theta, the moments and the fit itself -- so for integer weights the fit is the fit of the
data with row l repeated w_l times (only `n_samples` stays the row count).  DESIGN.md section 12.
"""
import ctypes as C
import os
import time

import numpy as np

from . import _lib
from .sharding import Reducer

ANNEAL_SCHEDULE = [0.6 ** k for k in range(1, 7)] + [0]  # linearcorex.py:119
_PEER_BUFFERS = {}  # (group, device, size) -> (symmetric tensor, handle): peer mappings are reused across fits


def _torch():
    import torch
    return torch


class LazyMoments(dict):
    """`moments` for large models: the m x n arrays stay on the device (a snapshot taken when the fit finished) and cross to
    the host the first time their key is read; everything else about it is a plain dict of numpy arrays like the reference's.
    Iterating, `len`, `items()`, `values()`, `==`, `copy()` and pickling materialise every key first."""

    def __init__(self, eager, lazy, order=None):
        dict.__init__(self, eager)
        self._lazy = dict(lazy)   # key -> callable returning the host array
        self._order = list(order) if order is not None else list(eager) + list(lazy)   # the reference's key order

    def _fetch(self, key):
        value = self._lazy.pop(key)()
        dict.__setitem__(self, key, value)
        return value

    def materialize(self):
        if self._lazy:
            for key in list(self._lazy):
                self._fetch(key)
            items = [(k, dict.__getitem__(self, k)) for k in self._order if dict.__contains__(self, k)]
            items += [(k, v) for k, v in dict.items(self) if k not in self._order]
            dict.clear(self)
            for k, v in items:
                dict.__setitem__(self, k, v)
        return self

    def pending(self):
        """Keys still resident on the device only."""
        return sorted(self._lazy)

    def __missing__(self, key):
        if key in self._lazy:
            return self._fetch(key)
        raise KeyError(key)

    def __contains__(self, key):
        return dict.__contains__(self, key) or key in self._lazy

    def get(self, key, default=None):
        return self[key] if key in self else default

    def __setitem__(self, key, value):
        self._lazy.pop(key, None)
        dict.__setitem__(self, key, value)

    def __delitem__(self, key):
        if self._lazy.pop(key, None) is None:
            dict.__delitem__(self, key)

    def __iter__(self):
        return dict.__iter__(self.materialize())

    def __len__(self):
        return dict.__len__(self) + len(self._lazy)

    def keys(self):
        return dict.keys(self.materialize())

    def items(self):
        return dict.items(self.materialize())

    def values(self):
        return dict.values(self.materialize())

    def copy(self):
        return dict(self.materialize())

    def __eq__(self, other):
        return dict.__eq__(self.materialize(), other)

    __hash__ = None

    def __reduce__(self):
        return (dict, (dict(self.materialize()),))


class _HostDraw(object):
    """np.random.randn(m, n) from the global legacy generator, on a background thread."""

    def __init__(self, m, n):
        import threading
        self.out, self.err = None, None
        self._th = threading.Thread(target=self._run, args=(m, n), daemon=True)
        self._th.start()

    def _run(self, m, n):
        try:
            self.out = np.random.randn(m, n)
        except BaseException as e:  # surfaced by result()
            self.err = e

    def result(self):
        self._th.join()
        if self.err is not None:
            raise self.err
        return self.out


class _DeviceSession(object):
    """Owns the lcx_session handle, the bound X~ block and the torch workspace."""

    def __init__(self, precision, device=None):
        torch = _torch()
        self.precision = precision
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.LcxError("no CUDA device: linearcorex_b200 has no CPU path")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        torch.cuda.set_device(self.device)
        h = C.c_void_p()
        _lib.check(self.lib.lcx_session_create(C.byref(h), self.device.index, precision), "lcx_session_create")
        self.h = h
        self.stream = torch.cuda.current_stream(self.device)
        _lib.check(self.lib.lcx_set_stream(self.h, C.c_void_p(self.stream.cuda_stream)), "lcx_set_stream")
        self.xt = None
        self.ws = None
        self._hook = None
        self.n = self.m = 0

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.lcx_session_destroy(self.h)
            self.h = None
        entry = getattr(self, "_peer_entry", None)
        if entry is not None:
            entry[2] = False  # the peer buffer may be reused by the next session
            self._peer_entry = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing ----------------------------------------------------------------------------
    def launches(self):
        v = C.c_longlong(0)
        _lib.check(self.lib.lcx_launch_count(self.h, C.byref(v)))
        return v.value + getattr(self, "launches_before", 0)

    def bind(self, xt, n_rows_total, n_vars, n_factors, reducer, n_local=None):
        """xt = preprocessed fp64 block, or None (split modes) when the digit planes are filled block by block
        through lcx_slice_block afterwards (`n_local` rows)."""
        torch = _torch()
        n_local = xt.shape[0] if xt is not None else int(n_local)
        need = self.lib.lcx_workspace_doubles(n_local, n_vars, n_factors, self.precision)
        if need <= 0:
            raise _lib.LcxError("bad problem shape")
        self.ws = torch.zeros(need, dtype=torch.float64, device=self.device)
        self.xt = xt
        self.n, self.m = n_vars, n_factors
        _lib.check(self.lib.lcx_bind(self.h, xt.data_ptr() if xt is not None else None, n_local, n_rows_total, n_vars,
                                     xt.stride(0) if xt is not None else self.lib.lcx_ld(n_vars), n_factors,
                                     self.ws.data_ptr(), need), "lcx_bind")
        if self.precision != _lib.PRECISION_FP64:
            self.xt = None  # the split modes keep int8 digit planes in the workspace; the fp64 block is released
        self._peer_buf = None
        if reducer is not None and reducer.world > 1 and reducer.backend == "nccl" and \
                os.environ.get("LCX_PEER_ALLREDUCE", "1") != "0" and self._bind_peers(reducer, n_vars, n_factors):
            self._hook = None  # sums over ranks run inside the fused peer-memory kernel
            _lib.check(self.lib.lcx_set_allreduce(self.h, C.cast(None, _lib.ALLREDUCE_FN), None), "lcx_set_allreduce")
        elif reducer is not None and reducer.world > 1:
            ws = self.ws

            def hook(_user, offset, count):
                try:
                    reducer.sum_(ws[offset:offset + count])
                    return 0
                except Exception:  # never let an exception unwind through the C frame
                    return 1
            self._hook = _lib.ALLREDUCE_FN(hook)
            _lib.check(self.lib.lcx_set_allreduce(self.h, self._hook, None), "lcx_set_allreduce")
        else:
            self._hook = None
            _lib.check(self.lib.lcx_set_allreduce(self.h, C.cast(None, _lib.ALLREDUCE_FN), None), "lcx_set_allreduce")

    def bind_gram(self, g, n_vars, n_factors):
        """Bind to the n x n matrix X~^T X~ / N (lcx_bind_gram): its digit planes live in the workspace, `g` is released."""
        torch = _torch()
        need = self.lib.lcx_gram_workspace_doubles(n_vars, n_factors, self.precision)
        if need <= 0:
            raise _lib.LcxError("bad problem shape")
        self.ws = torch.zeros(need, dtype=torch.float64, device=self.device)
        self.xt = None
        self.n, self.m = n_vars, n_factors
        _lib.check(self.lib.lcx_bind_gram(self.h, g.data_ptr(), g.stride(0), n_vars, n_factors, self.ws.data_ptr(), need),
                   "lcx_bind_gram")
        self._peer_buf = None
        self._hook = None
        _lib.check(self.lib.lcx_set_allreduce(self.h, C.cast(None, _lib.ALLREDUCE_FN), None), "lcx_set_allreduce")

    def _bind_peers(self, reducer, n_vars, n_factors):
        """Map one symmetric buffer on every rank (torch symmetric memory: CUDA VMM handles exchanged over the process
        group) and hand the peer pointers to the library.  Returns False when peer mapping is unavailable, in which
        case the NCCL hook is used instead."""
        torch = _torch()
        try:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm
            need = self.lib.lcx_peer_buffer_doubles(n_vars, n_factors)
            group = reducer.group if reducer.group is not None else dist.group.WORLD
            key = (id(group), self.device.index, need)
            prev = getattr(self, "_peer_entry", None)
            if prev is not None:  # a re-bind of this session (second fit on the same model) reuses its own buffer
                prev[2] = False
                self._peer_entry = None
            # mapping peers costs ~0.1 s (VMM handles over the process group): a released buffer is reused by the next
            # session of the same shape; a buffer still owned by a live session is never shared (its flags carry epochs)
            entry = _PEER_BUFFERS.get(key)
            if entry is None or entry[2]:
                buf = symm.empty(need, dtype=torch.float64, device=self.device)
                entry = [buf, symm.rendezvous(buf, group), True]
                if key not in _PEER_BUFFERS:
                    _PEER_BUFFERS[key] = entry
            entry[2] = True
            self._peer_entry = entry
            buf, hdl = entry[0], entry[1]
            buf.zero_()  # flags restart at zero for this session's epochs
            torch.cuda.synchronize(self.device)
            dist.barrier(group=reducer.group)  # nobody signals before every rank has zeroed its flags
            ptrs = (C.c_void_p * reducer.world)(*[int(p) for p in hdl.buffer_ptrs])
            _lib.check(self.lib.lcx_set_peer_allreduce(self.h, reducer.world, reducer.rank, ptrs, need),
                       "lcx_set_peer_allreduce")
            self._peer_buf, self._peer_hdl = buf, hdl
            return True
        except Exception as exc:  # noqa: BLE001 -- any failure here just selects the NCCL path
            if os.environ.get("LCX_PEER_ALLREDUCE") == "require":
                raise
            self._peer_error = repr(exc)
            return False

    def view(self, array_id, which=0):
        off, rows, cols, ld = (C.c_longlong() for _ in range(4))
        _lib.check(self.lib.lcx_array_info(self.h, array_id, which, C.byref(off), C.byref(rows), C.byref(cols),
                                           C.byref(ld)), "lcx_array_info")
        flat = self.ws[off.value: off.value + rows.value * ld.value]
        return flat.view(rows.value, ld.value)[:, :cols.value]

    def host(self, array_id, which=0, squeeze=False, transpose=False):
        """Host copy of an exported array (`transpose=True`: turned around on the device first, so the host receives the
        reference's n x m layout of `X_i Y_j` / `X_i Z_j` without a strided numpy copy)."""
        v = self.view(array_id, which)
        a = (v.t().contiguous() if transpose else v).cpu().numpy()  # .cpu() already owns fresh memory
        return a[0].copy() if squeeze else a


AUTO_SPLIT_MIN_WORK = 3e7  # N n m above which the split-integer tcgen05 contractions beat the DMMA ones (see 'auto')


def resolve_precision(precision, n_rows_total, n_vars, n_factors, gaussianize='standard'):
    """'auto' -> 'fp64_split' or, for launch-bound small problems, 'fp64'; anything else passes through.

    The split modes keep 48 bits below ONE exponent for all of X~ (max |X~|).  That is binary64-faithful for standardised data
    ('standard', 'outliers': every column has unit scale), but with gaussianize='none' the columns keep the user's scales and a
    small-magnitude column would silently hold far fewer than 48 significant bits -- so 'auto' stays on the all-binary64 DMMA
    path there; the split modes remain available by name."""
    if precision != 'auto':
        return precision
    if gaussianize == 'none':
        return 'fp64'
    return 'fp64_split' if float(n_rows_total) * float(n_vars) * float(n_factors) >= AUTO_SPLIT_MIN_WORK else 'fp64'


class Corex(object):
    """Linear Total Correlation Explanation on B200 (see module docstring)."""

    def __init__(self, n_hidden=10, max_iter=10000, tol=1e-5, anneal=True, missing_values=None,
                 discourage_overlap=True, gaussianize='standard', gpu=True, verbose=False, seed=None,
                 eliminate_synergy=None, precision='auto', exact_trials=False, input_dtype='float64',
                 comm=None, device=None, stream_rows=None, algorithm='auto'):
        self.m = n_hidden
        self.max_iter = max_iter
        self.tol = tol
        self.anneal = anneal
        self.eps = 0
        self.missing_values = missing_values
        if eliminate_synergy is not None:
            discourage_overlap = bool(eliminate_synergy)
        self.discourage_overlap = discourage_overlap
        self.gaussianize = gaussianize
        self.gpu = True  # kept for signature compatibility; the device path is the only path
        self.yscale = 1.
        if gaussianize not in ('standard', 'outliers', 'none'):
            raise ValueError("gaussianize must be 'standard', 'outliers' or 'none' "
                             "('empirical' is not supported: the reference itself cannot invert it, :425)")
        if precision != 'auto' and precision not in _lib.PRECISIONS:
            raise ValueError("precision must be 'auto' or one of %s" % sorted(_lib.PRECISIONS))
        if input_dtype not in ('float64', 'float32'):
            raise ValueError("input_dtype must be 'float64' or 'float32'")
        if algorithm not in ('auto', 'stream', 'gram'):
            raise ValueError("algorithm must be 'auto', 'stream' or 'gram'")
        self.algorithm = algorithm
        self.algorithm_used = None
        self.precision = precision
        self.precision_used = None if precision == 'auto' else precision  # 'auto' is resolved when fit sees the shape
        self.exact_trials = bool(exact_trials)
        self.input_dtype = input_dtype
        self.stream_rows = stream_rows  # row-block size of the streamed preparation (None = decide from free memory)
        np.random.seed(seed)  # :89 -- the reference seeds the *global* legacy RNG at construction
        self.verbose = verbose
        if verbose:
            np.set_printoptions(precision=3, suppress=True, linewidth=160)
            print('Linear CorEx with {:d} latent factors'.format(n_hidden))
        self.n_samples, self.nv = 0, 0
        self.ws = np.zeros((0, 0))
        self.moments = {}
        self.theta = None
        self.n_obs = 0
        self.history = {}
        self.trace = []          # per-iteration: eps, eta, trials, quick_fails, tangent, TC
        self.timings = {}        # wall-clock seconds of the one-off phases (upload, preprocess, bind, finish)
        self._comm = comm
        self._device = device
        self._sess = None
        self._theta_dev = None
        self._fitted_in_session = False  # the bound device workspace holds this model's final moments

    # ------------------------------------------------------------------------------------------
    # pickling (vis_corex.py:549): host state only
    # ------------------------------------------------------------------------------------------
    def __getstate__(self):
        d = dict(self.__dict__)
        for k in ("_sess", "_theta_dev", "_comm"):
            d[k] = None
        d["_fitted_in_session"] = False
        return d

    # ------------------------------------------------------------------------------------------
    # properties of the reference (:177-194)
    # ------------------------------------------------------------------------------------------
    @property
    def tc(self):
        return self.moments["TC"]

    @property
    def tcs(self):
        return self.moments["TCs"]

    @property
    def mis(self):
        return - 0.5 * np.log1p(-self.moments["rho"] ** 2)

    def clusters(self):
        return np.argmax(np.abs(self.ws), axis=0)

    # ------------------------------------------------------------------------------------------
    # device helpers
    # ------------------------------------------------------------------------------------------
    def _active_precision(self):
        return self.precision_used or 'fp64_split'

    def _session(self):
        want = _lib.PRECISIONS[self._active_precision()]
        if self._sess is not None and getattr(self._sess, "is_gram", False):
            return self._sess  # the Gram route's session (bound to X~^T X~ / N: _to_gram)
        if self._sess is not None and self._sess.precision != want:  # 'auto' resolved differently for a new shape
            self._sess.close()
            self._sess = None
        if self._sess is None:
            self._sess = _DeviceSession(want, self._device)
        return self._sess

    def _reducer(self):
        return Reducer(self._comm)

    def _upload(self, x):
        """Host array -> device tensor (float32 or float64), through pinned staging in row chunks."""
        torch = _torch()
        sess = self._session()
        x = np.ascontiguousarray(x)
        out = torch.empty(x.shape, dtype=torch.float32 if x.dtype == np.float32 else torch.float64, device=sess.device)
        row_bytes = max(1, x.shape[1] * x.itemsize)
        if x.nbytes <= (64 << 20):
            out.copy_(torch.from_numpy(x))
            return out
        # Large input: two pinned staging buffers.  Worker threads fill buffer b (pageable -> pinned memcpy, GIL
        # released) while the DMA engine drains buffer 1-b, so the upload runs at min(host memcpy, PCIe) speed.
        from concurrent.futures import ThreadPoolExecutor
        rows = max(1, int((128 << 20) // row_bytes))
        nthr = 8
        stages = [torch.empty((rows, x.shape[1]), dtype=out.dtype).pin_memory() for _ in range(2)]
        done = [None, None]
        stream = torch.cuda.current_stream()

        def fill(buf, base, lo, hi):
            if hi > lo:
                buf[lo:hi].copy_(torch.from_numpy(x[base + lo:base + hi]))

        with ThreadPoolExecutor(max_workers=nthr) as pool:
            for i, lo in enumerate(range(0, x.shape[0], rows)):
                hi = min(x.shape[0], lo + rows)
                b = i & 1
                if done[b] is not None:
                    done[b].synchronize()  # the DMA that last read this staging buffer has finished
                cnt = hi - lo
                step = (cnt + nthr - 1) // nthr
                list(pool.map(lambda k: fill(stages[b], lo, k * step, min(cnt, (k + 1) * step)), range(nthr)))
                out[lo:hi].copy_(stages[b][:cnt], non_blocking=True)
                done[b] = torch.cuda.Event()
                done[b].record(stream)
        stream.synchronize()
        return out

    def _as_input(self, x):
        """Device tensors pass through (row block already resident); host data is cast like :108."""
        torch = _torch()
        if isinstance(x, torch.Tensor) and x.is_cuda:
            if x.dtype not in (torch.float32, torch.float64):
                x = x.double()
            if self.input_dtype == 'float32' and x.dtype != torch.float32:
                x = x.float()
            return x.contiguous()
        want = np.float32 if self.input_dtype == 'float32' else np.float64
        if isinstance(x, torch.Tensor):  # host tensor: page-locked memory goes straight to the DMA engine
            if x.is_pinned() and x.is_contiguous() and x.dtype in (torch.float32, torch.float64) and \
                    not (self.input_dtype == 'float32' and x.dtype != torch.float32):
                out = torch.empty(x.shape, dtype=x.dtype, device=self._session().device)
                out.copy_(x, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                return out
            x = x.numpy()
        x = np.asarray(x)
        if x.dtype == np.float32 and want == np.float64:
            return self._upload(x)  # float32 values are exact in float64: keep the narrow upload
        return self._upload(np.asarray(x, dtype=want))

    def preprocess(self, x, fit=False, _weights=None):
        """Device preprocessing (:397-429).  Returns the fp64 X~ tensor (N x ld).

        `_weights` (fit only): (w, w_total) from `_sample_weights` -- weighted column statistics, and row l of X~ scaled by
        r_l = sqrt(N w_l / w_total) (DESIGN.md section 12)."""
        torch = _torch()
        sess = self._session()
        lib = sess.lib
        red = self._reducer()
        t_up = time.perf_counter()
        xd = self._as_input(x)
        self.timings["upload_s"] = time.perf_counter() - t_up
        N, n = xd.shape
        dt = _lib.F32 if xd.dtype == torch.float32 else _lib.F64
        ldo = lib.lcx_ld(n)
        out = torch.empty((N, ldo), dtype=torch.float64, device=sess.device)
        has_marker = self.missing_values is not None
        marker = float(self.missing_values) if has_marker else 0.0
        mode = _lib.GAUSS[self.gaussianize]
        vec = lambda: torch.zeros(n, dtype=torch.float64, device=sess.device)
        nscr = lib.lcx_colstats_scratch_doubles(N, n)
        scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
        impute = mean = sd = None
        n_total = red.sum_scalar(N)
        wd = rs = None
        if _weights is not None and fit:
            w_total = _weights[1]
            wd = torch.as_tensor(_weights[0], dtype=torch.float64).to(sess.device)
            rs = self._row_scale(wd, w_total, n_total)
        if has_marker or (fit and mode != _lib.GAUSS['none']):
            ssum, cnt = vec(), vec()
            if wd is None:
                _lib.check(lib.lcx_colstats_sum(sess.h, xd.data_ptr(), dt, N, n, xd.stride(0), int(has_marker), marker,
                                                ssum.data_ptr(), cnt.data_ptr(), scratch.data_ptr(), nscr), "lcx_colstats_sum")
            else:
                _lib.check(lib.lcx_colstats_sum_w(sess.h, xd.data_ptr(), dt, N, n, xd.stride(0), int(has_marker), marker,
                                                  ssum.data_ptr(), cnt.data_ptr(), scratch.data_ptr(), nscr, wd.data_ptr()),
                           "lcx_colstats_sum_w")
            red.sum_(ssum)
            red.sum_(cnt)
            impute = vec()
            _lib.check(lib.lcx_colstats_mean(sess.h, ssum.data_ptr(), cnt.data_ptr(), impute.data_ptr(), n))
            if wd is None:
                self.n_obs = cnt.cpu().numpy().astype(np.int64) if has_marker else int(n_total)
            else:
                self.n_obs = cnt.cpu().numpy() if has_marker else float(w_total)
        else:
            self.n_obs = int(n_total) if wd is None else float(w_total)
        if mode != _lib.GAUSS['none']:
            if fit:
                mean = impute
                sq, sd = vec(), vec()
                if wd is None:
                    _lib.check(lib.lcx_colstats_sqdev(sess.h, xd.data_ptr(), dt, N, n, xd.stride(0), int(has_marker), marker,
                                                      mean.data_ptr(), sq.data_ptr(), None, scratch.data_ptr(), nscr),
                               "lcx_colstats_sqdev")
                else:
                    _lib.check(lib.lcx_colstats_sqdev_w(sess.h, xd.data_ptr(), dt, N, n, xd.stride(0), int(has_marker), marker,
                                                        mean.data_ptr(), sq.data_ptr(), None, scratch.data_ptr(), nscr,
                                                        wd.data_ptr(), rs.data_ptr()), "lcx_colstats_sqdev_w")
                red.sum_(sq)
                _lib.check(lib.lcx_colstats_std(sess.h, sq.data_ptr(), cnt.data_ptr(), float(n_total if wd is None else w_total),
                                                int(self.gaussianize == 'standard'), sd.data_ptr(), n))
                self._theta_dev = (mean, sd)
                self.theta = (mean.cpu().numpy().copy(), sd.cpu().numpy().copy())
            else:
                if self._theta_dev is None:  # e.g. after unpickling
                    self._theta_dev = tuple(torch.as_tensor(np.asarray(t, dtype=np.float64), device=sess.device)
                                            for t in self.theta)
                mean, sd = self._theta_dev
        p = lambda t: t.data_ptr() if t is not None else None
        if rs is None:
            _lib.check(lib.lcx_standardize(sess.h, xd.data_ptr(), dt, N, n, xd.stride(0), int(has_marker), marker, mode,
                                           p(impute), p(mean), p(sd), out.data_ptr(), ldo), "lcx_standardize")
        else:
            _lib.check(lib.lcx_standardize_w(sess.h, xd.data_ptr(), dt, N, n, xd.stride(0), int(has_marker), marker, mode,
                                             p(impute), p(mean), p(sd), out.data_ptr(), ldo, rs.data_ptr()), "lcx_standardize_w")
        return out

    def _sample_weights(self, sample_weight, n_rows, red):
        """Validate per-row weights before any device work: (w as a host float64 array, their sum over all ranks).
        Raises ValueError (on every rank when one rank's weights are bad) unless w is 1-D with one finite, non-negative
        value per local row and the total over all ranks is positive."""
        torch = _torch()
        err = None
        try:
            if isinstance(sample_weight, torch.Tensor):
                w = sample_weight.detach().to(device="cpu", dtype=torch.float64).numpy()
            else:
                w = np.asarray(sample_weight, dtype=np.float64)
        except (TypeError, ValueError) as e:
            w, err = None, "sample_weight must be numeric: %s" % e
        if err is None:
            if w.ndim != 1:
                err = "sample_weight must be 1-D, got shape %s" % (w.shape,)
            elif w.shape[0] != n_rows:
                err = "sample_weight has %d entries for %d rows" % (w.shape[0], n_rows)
            elif not np.isfinite(w).all():
                err = "sample_weight must be finite"
            elif (w < 0).any():
                err = "sample_weight must be non-negative"
        bad = 1 if err else 0
        if red.world > 1:
            bad = red.max_scalar(bad)
        if err or bad:
            raise ValueError(err or "sample_weight is invalid on another rank")
        w_total = float(red.sum_scalar(float(np.sum(w))))
        if not (0.0 < w_total < np.inf):
            raise ValueError("sample_weight must have a positive, finite sum over all rows (got %r)" % w_total)
        return np.ascontiguousarray(w), w_total

    def _row_scale(self, wd, w_total, n_total):
        """The row scales r_l = sqrt(N_total w_l / W_total) of X~ (lcx_row_scale) from the device weights wd."""
        sess = self._session()
        rs = _torch().empty(wd.shape[0], dtype=_torch().float64, device=sess.device)
        _lib.check(sess.lib.lcx_row_scale(sess.h, wd.data_ptr(), wd.shape[0], float(n_total), float(w_total), rs.data_ptr()),
                   "lcx_row_scale")
        return rs

    # ------------------------------------------------------------------------------------------
    # fit (:107-164)
    # ------------------------------------------------------------------------------------------
    def fit(self, x, sample_weight=None):
        """Fit the model to the rows of x (:107-164).

        sample_weight: None, or one non-negative weight per row (ndarray, list, host or CUDA tensor; used as float64).  Every
        statistic of the fit becomes its weighted average -- the column means (also the imputation means of missing entries)
        and stds in theta, n_obs (the weighted observed count), the moments -- and for integer weights the fit equals the fit
        of the data with row l repeated w_l times; n_samples stays the row count.  With `comm`, each rank passes the weights
        of its own rows.  The weights are validated before any device work (ValueError) and not stored.  The split precisions
        keep one exponent for all of X~, whose row l is scaled by sqrt(N w_l / sum w): very uneven weights raise it by
        log2 of the largest such scale, and every other row loses those bits (DESIGN.md section 12)."""
        weights = None
        if sample_weight is not None:
            weights = self._sample_weights(sample_weight, int(np.shape(x)[0]), self._reducer())
        schedule = self._prepare(x, weights)
        for i_eps, eps in enumerate(schedule):
            self._begin_stage(eps, rescale=i_eps > 0)
            if self.discourage_overlap and not self.verbose:
                if not self._run_stage_native():
                    self.ws = self._get_w()
                    return self
                continue
            delta = 0.0
            for i_loop in range(self.max_iter):
                ok, delta = self._iterate()
                if not ok:  # the reference returns from inside the loop (:149) without the final sort
                    self.ws = self._get_w()
                    return self
                if delta < self.tol:
                    if self.verbose:
                        print('{:d} iterations to tol: {:f}, TC={:f}'.format(i_loop, self.tol, self.tc))
                    break
            else:
                if self.verbose:
                    print("Warning: Convergence not achieved in {:d} iterations. Final delta: {:f}".format(
                        self.max_iter, float(delta)))
        return self._finish()

    STAGE_CHUNK = 1024

    def _run_stage_native(self):
        """The iterations of one annealing stage inside the library (lcx_run_stage_ns: same control flow as `_iterate` +
        `_update_ns`, no interpreter between iterations).  Returns False where the reference returns early (:144-149)."""
        sess = self._sess
        lib = sess.lib
        left = int(self.max_iter)
        cap = max(1, min(self.STAGE_CHUNK, left))
        tc, tang, eta = ((C.c_double * cap)() for _ in range(3))
        trials, qf = ((C.c_int * cap)() for _ in range(2))
        n_done, reason = C.c_int(), C.c_int()
        hist = self.history.setdefault("TC", [])
        while left > 0:
            chunk = min(cap, left)
            _lib.check(lib.lcx_run_stage_ns(sess.h, float(self.eps), float(self.tol), int(self.exact_trials), chunk,
                                            float(self.tc), C.byref(n_done), C.byref(reason), tc, tang, eta, trials, qf),
                       "lcx_run_stage_ns")
            k = n_done.value
            invalid = reason.value == 2
            for i in range(k):
                if tang[i] >= 0:  # :306-311
                    print('Warning: covariance is nearly singular and this causes a loss of numerical precision.'
                          'For this reason, we can no longer find an update that increases the objective. '
                          'Hopefully this is a good solution. If not, this is caused by having many variables that are '
                          'near duplicates. You could try again with the duplicates removed to look for other structure.')
                if invalid and i == k - 1:
                    break
                if not np.isfinite(tc[i]):
                    print("Error: TC is no longer finite: {}".format(tc[i]))
                self.trace.append({"eps": self.eps, "tangent": tang[i], "eta": eta[i], "trials": trials[i],
                                   "quick_fails": qf[i], "TC": tc[i]})
                hist.append(tc[i])
            if k > 0 and not (invalid and k == 1):
                self.moments = {"TC": tc[k - 2] if invalid else tc[k - 1]}
            if invalid:
                print("Error... updates giving invalid solutions?")
                return False
            if reason.value == 1:
                return True
            left -= k
        return True

    def _prepare(self, x, weights=None):
        """Preprocess, bind the device problem and initialise W (:108-122).  Returns the anneal schedule.
        `weights`: None or (w, w_total) from `_sample_weights`."""
        if self.m is None:
            raise ValueError("n_hidden=None (pick_n_hidden) is not supported: the reference helper is broken (:458-480)")
        red = self._reducer()
        # W0 (:114-121) comes from numpy's legacy global generator exactly as in the reference -- a serial MT19937 + polar-method
        # stream (55 ms for 100 x 10 000 on one core).  Nothing else of fit draws from it, so it is drawn first, on a thread
        # (RandomState releases the GIL), while the device work of the preparation runs; joined where the reference draws it.
        w0_draw = _HostDraw(self.m, int(np.shape(x)[1])) if self.ws.size == 0 else None
        if self.precision == 'auto':  # every rank sees the same total, so every rank takes the same path
            self.precision_used = resolve_precision('auto', red.sum_scalar(int(np.shape(x)[0])), int(np.shape(x)[1]), self.m,
                                                    self.gaussianize)
        if self._sess is not None and getattr(self._sess, "is_gram", False):  # a refit starts from a fresh data session
            self._sess.close()
            self._sess = None
        sess = self._session()
        lib = sess.lib
        self._fitted_in_session = False
        rows = self._stream_rows_for(x, red)
        if rows:
            self._prepare_streamed(x, rows, red, weights)
        else:
            t0 = time.perf_counter()
            xt = self.preprocess(x, fit=True, _weights=weights)
            _torch().cuda.synchronize()
            self.timings["preprocess_s"] = time.perf_counter() - t0
            n_local, self.nv = xt.shape[0], int(np.shape(x)[1])
            self.n_samples = int(red.sum_scalar(n_local))
            t0 = time.perf_counter()
            sess.bind(xt, self.n_samples, self.nv, self.m, red)
            _torch().cuda.synchronize()
            self.timings["bind_s"] = time.perf_counter() - t0
        self.algorithm_used = 'gram' if self._want_gram(red) else 'stream'
        if self.algorithm_used == 'gram':
            self._to_gram(red)
            sess = self._sess
        schedule = [0.]
        if self.ws.size == 0:  # :114-121
            if self.discourage_overlap:
                w0 = w0_draw.result()
                if self.input_dtype == 'float32':
                    w0 = w0.astype(np.float32)
                self._set_w(w0)
                _lib.check(lib.lcx_init_scale(sess.h, float(self.eps)), "lcx_init_scale")
                if self.anneal:
                    schedule = list(ANNEAL_SCHEDULE)
            else:
                self._set_w(w0_draw.result() * self.yscale ** 2 / np.sqrt(self.nv))
        else:
            self._set_w(self.ws)
        self.moments = {"TC": self._moments_from_x()}  # :122
        return schedule

    GRAM_MIN_WORK = 1e9  # N n m from which an iteration is bound by the passes over X~ rather than by launches
    # Digits of the matrix X~^T X~ / N and of the operand it meets, per data precision.  The build is exact for the digit planes
    # of X~, so the route's own truncation is that of the matrix.  One digit more for the matrix (6 -> 7) was measured and
    # does NOT buy parity: the ill-conditioned adni fixture (2 414 iterations, rho -> 1) sits at 8.5e-9 on invrho / Qij / Si
    # either way and at 1.2e-11 only when the DATA planes carry 7 digits too (precision='fp64_split7') -- what it amplifies
    # is the 48-bit truncation of X~, as on the streaming route -- while the product costs 28 / 21 more (config 3: 2 020 ->
    # 1 845 it/s; profiles/r02_parity_report.txt, r02_gram_digits_ab.txt).  So: same digits as the data.
    GRAM_PRECISION = {"fast": "fast", "fp64_split5": "fp64_split5", "fp64_split": "fp64_split", "fp64_split7": "fp64_split7"}

    def _gram_precision(self):
        return _lib.PRECISIONS[self.GRAM_PRECISION[self._active_precision()]]

    def _want_gram(self, red):
        """Resolve `algorithm` for the bound problem; every rank sees the same totals and takes the same route."""
        if getattr(self, "algorithm", "stream") == 'stream':
            return False
        split = self._active_precision() != 'fp64'
        if self.algorithm == 'gram':
            if not split:
                raise ValueError("algorithm='gram' runs on the split-integer engine: choose a split precision, not 'fp64'")
            return True
        if not split or self.n_samples < self.nv or float(self.n_samples) * self.nv * self.m < self.GRAM_MIN_WORK:
            return False
        torch = _torch()
        sess = self._sess
        free, _total = torch.cuda.mem_get_info(sess.device)
        need = 8 * (self.nv * sess.lib.lcx_ld(self.nv) + sess.lib.lcx_gram_workspace_doubles(self.nv, self.m, self._gram_precision())
                    + sess.lib.lcx_gram_scratch_doubles(sess.h, 128))
        fits = 1 if need < 0.8 * free else 0
        return bool(red.min_scalar(fits)) if red.world > 1 else bool(fits)

    def _to_gram(self, red):
        """G = X~^T X~ / N from the bound digit planes (summed over ranks), then re-bind the fit loop to G: the digit planes
        of X~ are released, and from here on no step touches the samples."""
        torch = _torch()
        sess = self._sess
        lib = sess.lib
        t0 = time.perf_counter()
        n = self.nv
        ldg = lib.lcx_ld(n)
        g = torch.zeros((n, ldg), dtype=torch.float64, device=sess.device)
        free, _total = torch.cuda.mem_get_info(sess.device)
        block = 128
        for cand in (1024, 512, 256):
            if cand <= max(128, ((n + 127) // 128) * 128) and 8 * lib.lcx_gram_scratch_doubles(sess.h, cand) < 0.5 * free:
                block = cand
                break
        nscr = lib.lcx_gram_scratch_doubles(sess.h, block)
        scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
        _lib.check(lib.lcx_gram_build(sess.h, g.data_ptr(), ldg, block, scratch.data_ptr(), nscr), "lcx_gram_build")
        if red.world > 1:
            red.sum_(g)
        torch.cuda.synchronize(sess.device)
        self.timings["gram_build_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        marks = [("start", t0)]
        del scratch
        launches = sess.launches()
        precision, device = self._gram_precision(), sess.device.index
        sess.close()
        sess.ws = None
        self._sess = None
        need = 8 * lib.lcx_gram_workspace_doubles(n, self.m, precision)
        if need > 0.5 * torch.cuda.mem_get_info(g.device)[0]:  # hand the digit planes of X~ back before the next allocation
            torch.cuda.empty_cache()
        marks.append(("release_data_session", time.perf_counter()))
        gs = _DeviceSession(precision, device)
        marks.append(("create_session", time.perf_counter()))
        gs.bind_gram(g, n, self.m)
        torch.cuda.synchronize(gs.device)
        marks.append(("slice_matrix", time.perf_counter()))
        gs.is_gram = True
        # With NVLink peers the per-iteration product G A^T is sharded over the ranks' row tiles of G and its column slabs are
        # exchanged in place (far::gather_cols_kernel); without them every rank computes the whole product (no exchange).
        if red.world > 1 and red.backend == "nccl" and os.environ.get("LCX_PEER_ALLREDUCE", "1") != "0":
            gs._bind_peers(red, n, self.m)
            marks.append(("map_peers", time.perf_counter()))
        gs.launches_before = launches
        self._sess = gs
        torch.cuda.synchronize(gs.device)
        self.timings["gram_bind_s"] = time.perf_counter() - t0
        self.timings["gram_bind_parts_s"] = {b[0]: round(b[1] - a[1], 4) for a, b in zip(marks, marks[1:])}

    def _stream_rows_for(self, x, red=None):
        """Row-block size of the split modes' preparation, or 0 for the fp64 path (DMMA mode, gaussianize='none').

        The split modes never materialise X~ in binary64: column statistics, then ONE fused pass standardise + g() + impute +
        digit slicing from the raw input (lcx_standardize_slice).  When the raw block fits on the device beside its digit
        planes it is uploaded once and the block is the whole input; otherwise (or when `stream_rows` says so) the three passes
        re-read the source in row blocks -- what lets the 1M x 20k target run on one GPU.  The choice is collective: if any
        rank must stream, every rank does."""
        if self._active_precision() == 'fp64' or self.gaussianize == 'none':
            return 0
        n_rows, n_vars = int(np.shape(x)[0]), int(np.shape(x)[1])
        if self.stream_rows:
            return int(self.stream_rows)
        torch = _torch()
        free, _total = torch.cuda.mem_get_info(self._session().device)
        digits = _lib.SPLIT_DIGITS.get(self._active_precision(), 6)
        need = n_rows * self._session().lib.lcx_ld(n_vars) * (digits + 8)   # planes + the raw block (as float64 at worst)
        stream = 1 if need > 0.8 * free else 0
        if red is not None and red.world > 1:
            stream = int(red.max_scalar(stream))
        return 32768 if stream else max(n_rows, 1)

    def _prepare_streamed(self, x, rows, red, weights=None):
        """preprocess(fit=True) + bind without ever holding all of X~ in fp64 (SURVEY.md hard part 4): three passes over
        row blocks of the raw input -- column sums/counts; squared deviations and max |x - mean|; standardise + digit
        slicing.  `x` only needs `.shape` and row slicing (ndarray, memmap, tensor, or a generator-backed object).
        `weights` (w, w_total): the weighted passes, w and the row scales taken in the same row blocks as the rows."""
        torch = _torch()
        sess = self._session()
        lib = sess.lib
        t0 = time.perf_counter()
        N, n = int(np.shape(x)[0]), int(np.shape(x)[1])
        self.nv = n
        ld = lib.lcx_ld(n)
        has_marker = self.missing_values is not None
        marker = float(self.missing_values) if has_marker else 0.0
        mode = _lib.GAUSS[self.gaussianize]
        vec = lambda: torch.zeros(n, dtype=torch.float64, device=sess.device)
        nscr = lib.lcx_colstats_scratch_doubles(rows, n)
        scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
        blocks = [(lo, min(N, lo + rows)) for lo in range(0, N, rows)]
        resident = None
        if len(blocks) == 1:  # the raw block fits: one upload, three passes over the device copy
            t_up = time.perf_counter()
            resident = self._as_input(x[0:N])
            self.timings["upload_s"] = time.perf_counter() - t_up

        def block(lo, hi):
            xd = resident[lo:hi] if resident is not None else self._as_input(x[lo:hi])
            return xd, (_lib.F32 if xd.dtype == torch.float32 else _lib.F64)

        wd = rs = None
        if weights is not None:
            w_total = weights[1]
            wd = torch.as_tensor(weights[0], dtype=torch.float64).to(sess.device)
        ssum, cnt, t1, t2 = vec(), vec(), vec(), vec()
        for lo, hi in blocks:  # pass 1
            xd, dt = block(lo, hi)
            if wd is None:
                _lib.check(lib.lcx_colstats_sum(sess.h, xd.data_ptr(), dt, hi - lo, n, xd.stride(0), int(has_marker), marker,
                                                t1.data_ptr(), t2.data_ptr(), scratch.data_ptr(), nscr), "lcx_colstats_sum")
            else:
                _lib.check(lib.lcx_colstats_sum_w(sess.h, xd.data_ptr(), dt, hi - lo, n, xd.stride(0), int(has_marker), marker,
                                                  t1.data_ptr(), t2.data_ptr(), scratch.data_ptr(), nscr, wd[lo:hi].data_ptr()),
                           "lcx_colstats_sum_w")
            ssum += t1
            cnt += t2
        red.sum_(ssum)
        red.sum_(cnt)
        n_total = red.sum_scalar(N)
        if wd is not None:
            rs = self._row_scale(wd, w_total, n_total)
        mean, sq, maxdev, sd = vec(), vec(), vec(), vec()
        _lib.check(lib.lcx_colstats_mean(sess.h, ssum.data_ptr(), cnt.data_ptr(), mean.data_ptr(), n))
        for lo, hi in blocks:  # pass 2
            xd, dt = block(lo, hi)
            if wd is None:
                _lib.check(lib.lcx_colstats_sqdev(sess.h, xd.data_ptr(), dt, hi - lo, n, xd.stride(0), int(has_marker), marker,
                                                  mean.data_ptr(), t1.data_ptr(), t2.data_ptr(), scratch.data_ptr(), nscr),
                           "lcx_colstats_sqdev")
            else:
                _lib.check(lib.lcx_colstats_sqdev_w(sess.h, xd.data_ptr(), dt, hi - lo, n, xd.stride(0), int(has_marker), marker,
                                                    mean.data_ptr(), t1.data_ptr(), t2.data_ptr(), scratch.data_ptr(), nscr,
                                                    wd[lo:hi].data_ptr(), rs[lo:hi].data_ptr()), "lcx_colstats_sqdev_w")
            sq += t1
            maxdev = torch.maximum(maxdev, t2)
        red.sum_(sq)
        _lib.check(lib.lcx_colstats_std(sess.h, sq.data_ptr(), cnt.data_ptr(), float(n_total if wd is None else w_total),
                                        int(self.gaussianize == 'standard'), sd.data_ptr(), n))
        self._theta_dev = (mean, sd)
        self.theta = (mean.cpu().numpy().copy(), sd.cpu().numpy().copy())
        if wd is None:
            self.n_obs = cnt.cpu().numpy().astype(np.int64) if has_marker else int(n_total)
        else:
            self.n_obs = cnt.cpu().numpy() if has_marker else float(w_total)
        zmax = float((maxdev / sd).max().item())  # weighted: maxdev bounds r_l |x - mean| (r_l the row scale)
        if self.gaussianize == 'outliers' and np.isfinite(zmax):
            zmax = min(zmax, 4.0) + float(np.tanh(max(zmax - 4.0, 0.0)))  # g() is monotone (:483-487)
            if rs is not None:
                # |r_l g(z_l)| <= max(1, max r) g(zmax): g is concave with g(0) = 0, so r g(z) <= g(r z) for r <= 1, and
                # z <= r z <= zmax for r > 1.  All weights equal: max r = 1 and the bound is the unweighted one.
                zmax *= max(1.0, float(rs.max().item()))
        self.n_samples = int(n_total)
        self.timings["preprocess_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sess.bind(None, self.n_samples, n, self.m, red, n_local=N)
        _lib.check(lib.lcx_set_x_scale(sess.h, zmax), "lcx_set_x_scale")
        for lo, hi in blocks:  # pass 3: raw rows -> int8 digit planes, X~ never exists in binary64
            xd, dt = block(lo, hi)
            if rs is None:
                _lib.check(lib.lcx_standardize_slice(sess.h, xd.data_ptr(), dt, lo, hi - lo, xd.stride(0), int(has_marker), marker,
                                                     mode, mean.data_ptr(), mean.data_ptr(), sd.data_ptr()), "lcx_standardize_slice")
            else:
                _lib.check(lib.lcx_standardize_slice_w(sess.h, xd.data_ptr(), dt, lo, hi - lo, xd.stride(0), int(has_marker),
                                                       marker, mode, mean.data_ptr(), mean.data_ptr(), sd.data_ptr(),
                                                       rs[lo:hi].data_ptr()), "lcx_standardize_slice_w")
        del resident, wd, rs
        torch.cuda.synchronize()
        self.timings["bind_s"] = time.perf_counter() - t0

    def _moments_from_x(self):
        """quick moments of the current W from X~ (one pass pair); returns TC."""
        sess = self._sess
        tcv, muj, addv = C.c_double(), C.c_double(), C.c_double()
        if self.discourage_overlap:
            _lib.check(sess.lib.lcx_moments_ns(sess.h, float(self.eps), 0, C.byref(tcv), C.byref(muj)), "lcx_moments_ns")
        else:
            _lib.check(sess.lib.lcx_moments_syn(sess.h, C.byref(tcv), C.byref(addv)), "lcx_moments_syn")
        return tcv.value

    def _begin_stage(self, eps, rescale):
        """Switch the annealing parameter (:127-134): rescale W so uj < 1 still holds, recompute moments."""
        sess = self._sess
        eps0, self.eps = self.eps, eps
        if rescale:
            _lib.check(sess.lib.lcx_stage_rescale(sess.h, float(eps), float(eps0)), "lcx_stage_rescale")
        self.moments = {"TC": self._moments_from_x()}

    def _iterate(self):
        """One pass of the loop body (:137-151).  Returns (ok, |delta TC|)."""
        sess = self._sess
        last_tc = self.tc
        rec = {"eps": self.eps}
        if self.discourage_overlap:
            ok = self._update_ns(rec)
        else:
            tcv, addv = C.c_double(), C.c_double()
            _lib.check(sess.lib.lcx_update_syn(sess.h, 0.1, C.byref(tcv), C.byref(addv)), "lcx_update_syn")
            self.moments = {"TC": tcv.value, "additivity": addv.value}
            ok = True
        if not ok:  # :144-149: moments is False -> formatting raises -> early return
            print("Error... updates giving invalid solutions?")
            return False, 0.0
        if not np.isfinite(self.tc):
            print("Error: TC is no longer finite: {}".format(self.tc))
        delta = np.abs(self.tc - last_tc)
        rec["TC"] = self.tc
        self.trace.append(rec)
        self.history.setdefault("TC", []).append(self.tc)  # (the reference rebuilds the list every iteration, :170)
        if self.verbose:  # :172-174 -- quick moments carry neither key (0 / zeros); the synergy moments carry both
            self.history.setdefault("additivity", []).append(self.moments.get("additivity", 0))
            tcs = np.zeros(self.m) if self.discourage_overlap else sess.host(_lib.A_TCS, squeeze=True)
            self.history.setdefault("TCs", []).append(tcs)
        if self.verbose > 1:
            print("TC={:.3f}\tadd={:.3f}\tdelta={:.6f}".format(self.tc, self.moments.get("additivity", 0), delta))
        return True, delta

    def _finish(self):
        """:160-163 full moments, sort factors by TCs (descending), full moments again."""
        sess = self._sess
        t0 = time.perf_counter()
        self._full_moments(export=False)  # only TCs is needed to order the factors
        order = np.argsort(-self.moments["TCs"])
        _lib.check(sess.lib.lcx_permute_rows(sess.h, (C.c_int * self.m)(*[int(o) for o in order])), "lcx_permute_rows")
        self._full_moments()
        self.ws = self._get_w()
        self._fitted_in_session = True
        self.timings["finish_s"] = time.perf_counter() - t0
        return self

    def fit_transform(self, x, sample_weight=None):
        """fit(x, sample_weight), then transform(x) (unweighted: the representation of every row)."""
        self.fit(x, sample_weight=sample_weight)
        return self.transform(x)

    def _set_w(self, w):
        sess = self._session()
        w = np.ascontiguousarray(w, dtype=np.float64)
        _lib.check(sess.lib.lcx_set_w(sess.h, w.ctypes.data_as(C.c_void_p), w.shape[1]), "lcx_set_w")

    def _get_w(self):
        sess = self._session()
        w = np.empty((self.m, self.nv), dtype=np.float64)
        _lib.check(sess.lib.lcx_get_w(sess.h, w.ctypes.data_as(C.c_void_p), self.nv), "lcx_get_w")
        return w

    def _update_ns(self, rec):
        """Host control flow of _update_ns (:290-334).  Returns False when the reference would hand
        back `False` moments (step too small right after a uj >= 1 rejection)."""
        sess = self._sess
        lib = sess.lib
        tcv, muj, tang = C.c_double(), C.c_double(), C.c_double()
        first_rc = None
        if self.exact_trials:
            _lib.check(lib.lcx_direction_ns(sess.h, float(self.eps), C.byref(tang)), "lcx_direction_ns")
        else:  # direction and the eta = 1 trial share one host synchronisation (the trial is discarded if tangent >= 0)
            first_rc = _lib.check(lib.lcx_direction_trial_ns(sess.h, float(self.eps), 1.0, C.byref(tang), C.byref(tcv),
                                                             C.byref(muj)), "lcx_direction_trial_ns")
        tangent = tang.value
        rec.update(tangent=tangent, eta=0.0, trials=0, quick_fails=0)
        if tangent >= 0:  # :306-311
            print('Warning: covariance is nearly singular and this causes a loss of numerical precision.'
                  'For this reason, we can no longer find an update that increases the objective. '
                  'Hopefully this is a good solution. If not, this is caused by having many variables that are '
                  'near duplicates. You could try again with the duplicates removed to look for other structure.')
            return True
        tc_now = self.tc
        eta = 1.
        last_rc = None
        while True:
            if eta < min(self.tol, 1e-10):  # :316-319
                if self.verbose:
                    print('Warning: step size becoming too small')
                break
            if first_rc is not None:
                rc, first_rc = first_rc, None
            else:
                rc = _lib.check(lib.lcx_trial_ns(sess.h, float(self.eps), eta, int(self.exact_trials), C.byref(tcv),
                                                 C.byref(muj)), "lcx_trial_ns")
            last_rc = rc
            rec["trials"] += 1
            if rc == _lib.QUICK_FAIL:  # TEST 1 (:322-326)
                rec["quick_fails"] += 1
                eta *= 0.5
                if self.verbose > 1:
                    print('back:{:.7f}'.format(eta))
                continue
            if not (-tcv.value <= -tc_now + 0.1 * eta * tangent):  # TEST 2, first Wolfe condition (:327-332)
                eta *= 0.5
                if self.verbose > 1:
                    print('wolfe1:{:.7f}'.format(eta))
                continue
            break
        rec["eta"] = eta
        if last_rc is None or last_rc == _lib.QUICK_FAIL:
            return False
        _lib.check(lib.lcx_accept_trial(sess.h), "lcx_accept_trial")
        self.moments = {"TC": tcv.value}
        return True

    # ------------------------------------------------------------------------------------------
    # moments export
    # ------------------------------------------------------------------------------------------
    def _full_moments(self, export=True):
        """`_calculate_moments(x, ws, quick=False)` from X~, then pull every key (or only TCs) to the host."""
        sess = self._sess
        lib = sess.lib
        tcv, muj, a, b = (C.c_double() for _ in range(4))
        if self.discourage_overlap:
            _lib.check(lib.lcx_moments_ns(sess.h, float(self.eps), 0, C.byref(tcv), C.byref(muj)), "lcx_moments_ns")
            _lib.check(lib.lcx_details_ns(sess.h, C.byref(a), C.byref(b)), "lcx_details_ns")
        else:
            _lib.check(lib.lcx_moments_syn(sess.h, C.byref(tcv), C.byref(b)), "lcx_moments_syn")
        if export:
            self.moments = self._export_moments(sess, tcv.value)
        else:
            self.moments = {"TC": tcv.value, "TCs": sess.host(_lib.A_TCS, squeeze=True)}

    LAZY_MOMENTS_BYTES = 256 << 20  # m x n arrays of moments stay on the device until read when together they exceed this

    def _export_moments(self, sess, tc):
        """Every key of the reference's moments dict.  Large models (the seven m x n arrays together above LAZY_MOMENTS_BYTES)
        get a LazyMoments: each m x n array is snapshotted on the device (the workspace is reused by the next fit) and crosses
        to the host on first access -- at 1 000 x 50 000 x 500 the eager export is 1.6 GB over PCIe into pageable memory,
        most of the time `fit` spends after its last iteration."""
        L = _lib
        lazy = 7 * 8 * self.m * self.nv > self.LAZY_MOMENTS_BYTES

        def big(array_id, transpose=False):
            if not lazy:
                return sess.host(array_id, transpose=transpose)
            snap = sess.view(array_id).clone()
            return lambda: (snap.t().contiguous() if transpose else snap).cpu().numpy()

        m = {}
        sc = sess.host(L.A_SCALARS, squeeze=True)
        if self.discourage_overlap:  # key set of _calculate_moments_ns (:236-288)
            m["uj"] = sess.host(L.A_UJ, squeeze=True)
            m["rho"] = big(L.A_RHO)
            m["ry"] = sess.host(L.A_RY)
            m["Y_j^2"] = sess.host(L.A_YJ2, squeeze=True)
            m["invrho"] = big(L.A_INVRHO)
            m["rhoinvrho"] = big(L.A_RHOINVRHO)
            m["Qij"] = big(L.A_QIJ)
            m["Si"] = sess.host(L.A_SI, squeeze=True)
            m["Qi-Si^2"] = sess.host(L.A_QISI2, squeeze=True)
            m["TC"] = tc
            m["MI"] = big(L.A_MI)
            m["X_i Y_j"] = big(L.A_XY, transpose=True)
            m["X_i Z_j"] = big(L.A_XZ, transpose=True)
            m["X_i^2 | Y"] = sess.host(L.A_X2Y, squeeze=True)
            m["I(Y_j ; X)"] = sess.host(L.A_IYX, squeeze=True)
            m["I(X_i ; Y)"] = sess.host(L.A_IXY, squeeze=True)
            m["TCs"] = sess.host(L.A_TCS, squeeze=True)
            m["TC_no_overlap"] = float(sc[4])
            m["TC_direct"] = sess.host(L.A_TCDIRECT, squeeze=True)
            m["additivity"] = float(sc[6])
        else:  # key set of _calculate_moments_syn (:336-373)
            m["X_i Y_j"] = big(L.A_XY, transpose=True)
            m["cy"] = sess.host(L.A_CY)
            m["Y_j^2"] = sess.host(L.A_YJ2, squeeze=True)
            m["ry"] = sess.host(L.A_RY)
            m["rho"] = big(L.A_RHO)
            m["invrho"] = big(L.A_INVRHO)
            m["rhoinvrho"] = big(L.A_RHOINVRHO)
            m["Qij"] = big(L.A_QIJ)
            m["Qi"] = sess.host(L.A_QISI2, squeeze=True)
            m["Si"] = sess.host(L.A_SI, squeeze=True)
            m["MI"] = big(L.A_MI)
            m["X_i Z_j"] = big(L.A_XZ, transpose=True)
            m["X_i^2 | Y"] = sess.host(L.A_X2Y, squeeze=True)
            m["TCs"] = sess.host(L.A_TCS, squeeze=True)
            m["additivity"] = float(sc[6])
            m["TC"] = tc
        if not lazy:
            return m
        return LazyMoments({k: v for k, v in m.items() if not callable(v)}, {k: v for k, v in m.items() if callable(v)},
                           order=list(m))

    # ------------------------------------------------------------------------------------------
    # transform / invert / predict / get_covariance (:386-395, :431-455)
    # ------------------------------------------------------------------------------------------
    def _transform_rows_for(self, x):
        """Row-block size for a streamed transform (inputs that are row providers, or too large to preprocess at once)."""
        torch = _torch()
        if not isinstance(x, (np.ndarray, torch.Tensor, list, tuple)):
            return int(self.stream_rows or 32768)
        n_rows, n_vars = int(np.shape(x)[0]), int(np.shape(x)[1])
        free, _total = torch.cuda.mem_get_info(self._session().device)
        return int(self.stream_rows or 32768) if n_rows * self._session().lib.lcx_ld(n_vars) * 12 > 0.8 * free else 0

    def _row_blocks(self, x, rows, per_block, impute_pass=True):
        """The row-block loop over new data (transform, scoring): imputation means of the new data from a first pass when a
        missing marker is set (:389/:404; summed over ranks with `comm`; skipped with impute_pass=False), the stored theta,
        then per_block(lo, hi, xd, dtype, impute, mean, sd) for every block [lo, hi) of `rows` rows uploaded as device tensor
        xd.  `x` only needs `.shape` and row slicing."""
        torch = _torch()
        sess = self._session()
        lib = sess.lib
        red = self._reducer()
        N, n = int(np.shape(x)[0]), int(np.shape(x)[1])
        has_marker = self.missing_values is not None
        marker = float(self.missing_values) if has_marker else 0.0
        mode = _lib.GAUSS[self.gaussianize]
        blocks = [(lo, min(N, lo + rows)) for lo in range(0, N, rows)]
        vec = lambda: torch.zeros(n, dtype=torch.float64, device=sess.device)
        impute = None
        if has_marker and impute_pass:
            nscr = lib.lcx_colstats_scratch_doubles(rows, n)
            scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
            ssum, cnt, t1, t2, impute = vec(), vec(), vec(), vec(), vec()
            for lo, hi in blocks:
                xd = self._as_input(x[lo:hi])
                dt = _lib.F32 if xd.dtype == torch.float32 else _lib.F64
                _lib.check(lib.lcx_colstats_sum(sess.h, xd.data_ptr(), dt, hi - lo, n, xd.stride(0), 1, marker, t1.data_ptr(),
                                                t2.data_ptr(), scratch.data_ptr(), nscr), "lcx_colstats_sum")
                ssum += t1
                cnt += t2
            red.sum_(ssum)
            red.sum_(cnt)
            _lib.check(lib.lcx_colstats_mean(sess.h, ssum.data_ptr(), cnt.data_ptr(), impute.data_ptr(), n))
        mean = sd = None
        if mode != _lib.GAUSS['none']:
            if self._theta_dev is None:
                self._theta_dev = tuple(torch.as_tensor(np.asarray(t, dtype=np.float64), device=sess.device) for t in self.theta)
            mean, sd = self._theta_dev
        for lo, hi in blocks:
            xd = self._as_input(x[lo:hi])
            per_block(lo, hi, xd, _lib.F32 if xd.dtype == torch.float32 else _lib.F64, impute, mean, sd)

    def _transform_streamed(self, x, rows):
        """transform() in row blocks (_row_blocks): preprocess and project block by block into one (N, ldy) device tensor."""
        torch = _torch()
        sess = self._session()
        lib = sess.lib
        N, n = int(np.shape(x)[0]), int(np.shape(x)[1])
        ld, ldy = lib.lcx_ld(n), lib.lcx_ldy(self.m)
        has_marker = self.missing_values is not None
        marker = float(self.missing_values) if has_marker else 0.0
        mode = _lib.GAUSS[self.gaussianize]
        p = lambda t: t.data_ptr() if t is not None else None
        wd = torch.zeros((self.m, ld), dtype=torch.float64, device=sess.device)
        wd[:, :n].copy_(torch.from_numpy(np.ascontiguousarray(self.ws, dtype=np.float64)))
        xt = torch.empty((rows, ld), dtype=torch.float64, device=sess.device)
        y = torch.empty((N, ldy), dtype=torch.float64, device=sess.device)

        def block(lo, hi, xd, dt, impute, mean, sd):
            _lib.check(lib.lcx_standardize(sess.h, xd.data_ptr(), dt, hi - lo, n, xd.stride(0), int(has_marker), marker, mode,
                                           p(impute), p(mean), p(sd), xt.data_ptr(), ld), "lcx_standardize")
            _lib.check(lib.lcx_project(sess.h, xt.data_ptr(), hi - lo, n, ld, wd.data_ptr(), ld, self.m,
                                       y[lo:hi].data_ptr(), ldy, None, None, 0), "lcx_project")
        self._row_blocks(x, rows, block)
        return y

    def transform(self, x, details=False, return_device=False):
        """Y = preprocess(x) . ws^T (:386-395).  Returns an (N, m) float64 ndarray; with
        `details=True` also the full moments of `x` under the fitted weights.  `return_device=True`
        returns the (N, m) CUDA tensor instead (layer stacking keeps Y resident, hierarchy.py)."""
        torch = _torch()
        sess = self._session()
        lib = sess.lib
        nv = int(np.shape(x)[1])
        assert self.nv == nv, "Incorrect number of variables in input, %d instead of %d" % (nv, self.nv)
        rows = self._transform_rows_for(x)
        if rows and not details:
            y = self._transform_streamed(x, rows)
            return y[:, :self.m] if return_device else y[:, :self.m].cpu().numpy().copy()
        xt = self.preprocess(x)
        ns = xt.shape[0]
        w = np.ascontiguousarray(self.ws, dtype=np.float64)
        ld = lib.lcx_ld(nv)
        wd = torch.zeros((self.m, ld), dtype=torch.float64, device=sess.device)
        wd[:, :nv].copy_(torch.from_numpy(w))
        ldy = lib.lcx_ldy(self.m)
        y = torch.empty((ns, ldy), dtype=torch.float64, device=sess.device)
        _lib.check(lib.lcx_project(sess.h, xt.data_ptr(), ns, nv, xt.stride(0), wd.data_ptr(), ld, self.m, y.data_ptr(),
                                   ldy, None, None, 0), "lcx_project")
        if return_device and not details:
            return y[:, :self.m]
        y_host = y[:, :self.m].cpu().numpy().copy()
        if details:
            other = _DeviceSession(_lib.PRECISIONS[self._active_precision()], self._device)
            red = self._reducer()
            other.bind(xt, int(red.sum_scalar(ns)), nv, self.m, red)
            _lib.check(lib.lcx_set_w(other.h, w.ctypes.data_as(C.c_void_p), nv), "lcx_set_w")
            tcv, muj, a, b = (C.c_double() for _ in range(4))
            if self.discourage_overlap:
                _lib.check(lib.lcx_moments_ns(other.h, float(self.eps), 0, C.byref(tcv), C.byref(muj)))
                _lib.check(lib.lcx_details_ns(other.h, C.byref(a), C.byref(b)))
            else:
                _lib.check(lib.lcx_moments_syn(other.h, C.byref(tcv), C.byref(b)))
            moments = self._export_moments(other, tcv.value)
            other.close()
            return y_host, moments
        return y_host

    def invert(self, x):
        """Undo the preprocessing (:431-438); O(N n) host arithmetic on user-supplied arrays."""
        if self.gaussianize == 'standard':
            return self.theta[1] * x + self.theta[0]
        if self.gaussianize == 'outliers':
            core = np.clip(x, -4, 4)
            return self.theta[1] * (core + np.arctanh(np.clip(x - core, -1 + 1e-10, 1 - 1e-10))) + self.theta[0]
        return x

    def _live_moments(self):
        """True when the session's workspace holds this model's final moments."""
        sess = self._session()
        return sess.ws is not None and sess.n == self.nv and sess.m == self.m and getattr(self, "_fitted_in_session", False)

    def _factor_major_device(self, key, live_id):
        """(m x ld) device tensor of an n x m moments array: the live workspace view, or an upload of the host copy
        (a model restored from a pickle has only host state, which is all the reference reads at :440-455)."""
        torch = _torch()
        sess = self._session()
        if self._live_moments():
            v = sess.view(live_id)
            return v, v.stride(0)
        ld = sess.lib.lcx_ld(self.nv)
        t = torch.zeros((self.m, ld), dtype=torch.float64, device=sess.device)
        t[:, :self.nv].copy_(torch.from_numpy(np.ascontiguousarray(np.asarray(self.moments[key], dtype=np.float64).T)))
        return t, ld

    def predict(self, y):
        """E(X | Y = y) in the original space (:440-441): invert(y . X_i Z_j^T); the N x n product runs on the device."""
        torch = _torch()
        sess = self._session()
        y = np.ascontiguousarray(np.asarray(y, dtype=np.float64))
        ny = y.shape[0]
        xz, ld = self._factor_major_device("X_i Z_j", _lib.A_XZ)
        ldy = sess.lib.lcx_ldy(self.m)
        yd = torch.zeros((ny, ldy), dtype=torch.float64, device=sess.device)
        yd[:, :self.m].copy_(torch.from_numpy(y))
        out = torch.empty((ny, ld), dtype=torch.float64, device=sess.device)
        _lib.check(sess.lib.lcx_gemm_f64(sess.h, 2, ny, self.nv, self.m, yd.data_ptr(), ldy, xz.data_ptr(), ld, out.data_ptr(), ld,
                                         0, None, 1, None, 0), "lcx_gemm_f64")
        return self.invert(out[:, :self.nv].cpu().numpy())

    def get_covariance(self, block_rows=4096, out=None, block_callback=None):
        """n x n covariance estimate (:443-455), computed on the device in row blocks from `moments` and `theta` (host
        state is enough, so this also works on an unpickled model).

        out=None            returns a new (n, n) float64 ndarray like the reference.
        out=ndarray/memmap  (n, n) float64: filled block by block (n = 50 000 is 20 GB: pass an np.memmap).
        out=CUDA tensor     (n, n) float64, even row stride: blocks are written in place, nothing crosses to the host.
        block_callback      callable(row0, block) called with each (rows, n) CUDA row block instead of gathering anything."""
        torch = _torch()
        sess = self._session()
        lib = sess.lib
        n = self.nv
        if self.theta is None:
            raise ValueError("get_covariance needs theta (gaussianize='none' has none, like the reference)")
        sd = torch.as_tensor(np.asarray(self.theta[1], dtype=np.float64), device=sess.device)
        if self.discourage_overlap:  # :447-451
            m = self.moments
            z = np.asarray(m['rhoinvrho'], dtype=np.float64) / (1 + np.asarray(m['Si'], dtype=np.float64))
            ld = lib.lcx_ld(n)
            left = torch.zeros((self.m, ld), dtype=torch.float64, device=sess.device)
            left[:, :n].copy_(torch.from_numpy(np.ascontiguousarray(z)))
            right, scale = left, 1. - self.eps ** 2
        else:  # :453-454
            left, ld = self._factor_major_device("X_i Z_j", _lib.A_XZ)
            right, _ = self._factor_major_device("X_i Y_j", _lib.A_XY)
            scale = 1.

        def fill(r0, rows, dst, ldd):
            _lib.check(lib.lcx_covariance_rows(sess.h, left.data_ptr(), right.data_ptr(), ld, self.m, n, float(scale),
                                               sd.data_ptr(), r0, rows, dst.data_ptr(), ldd), "lcx_covariance_rows")
        return self._n_by_n_rows(fill, block_rows, out, block_callback)

    def _n_by_n_rows(self, fill, block_rows, out, block_callback, n=None):
        """Output side of get_covariance / get_precision: fill(row0, rows, dst, ld_dst) writes a row block of the n x n matrix
        (n = nv unless given) into device memory; the blocks go to a new ndarray, to `out` (ndarray / memmap, or a CUDA tensor
        written in place) or to `block_callback`."""
        torch = _torch()
        sess = self._session()
        n = self.nv if n is None else n
        on_device = isinstance(out, torch.Tensor) and out.is_cuda
        if on_device:
            assert tuple(out.shape) == (n, n) and out.dtype == torch.float64 and out.stride(1) == 1 and out.stride(0) % 2 == 0, \
                "out must be an (%d, %d) float64 CUDA tensor with unit column stride and an even row stride" % (n, n)
        elif out is None and block_callback is None:
            out = np.empty((n, n), dtype=np.float64)
        ldc = sess.lib.lcx_ld(n)
        block_rows = max(2, min(block_rows, n + (n % 2)))
        block_rows -= block_rows % 2
        buf = None if on_device else torch.empty((block_rows, ldc), dtype=torch.float64, device=sess.device)
        for r0 in range(0, n, block_rows):
            rows = min(block_rows, n - r0)
            dst, ldd = (out[r0:r0 + rows], out.stride(0)) if on_device else (buf, ldc)
            fill(r0, rows, dst, ldd)
            if block_callback is not None:
                block_callback(r0, dst[:rows, :n])
            elif not on_device:
                out[r0:r0 + rows] = buf[:rows, :n].cpu().numpy()
        return out

    # ------------------------------------------------------------------------------------------
    # scoring under the covariance estimate (lowrank_kernels.cuh)
    # ------------------------------------------------------------------------------------------
    def _lowrank_moments(self):
        """(rhoinvrho (m x ld), ld, Si, theta[1]) as CUDA tensors for the low-rank-plus-diagonal routines, after their
        preconditions: from the live workspace when the session holds this model's final moments, otherwise uploaded from the
        host moments (an unpickled model)."""
        torch = _torch()
        if self.theta is None:
            raise ValueError("scoring needs theta (gaussianize='none' has none, like get_covariance)")
        if not self.discourage_overlap:
            raise ValueError("scoring supports discourage_overlap=True only: the synergy covariance X_i Z_j X_i Y_j^T with its "
                             "diagonal reset has no symmetric low-rank factor to build on")
        sess = self._session()
        lib = sess.lib
        n, m = self.nv, self.m
        if self._live_moments():
            rinv, si = sess.view(_lib.A_RHOINVRHO), sess.view(_lib.A_SI)[0]
            ld = rinv.stride(0)
        else:  # rhoinvrho is factor-major (m x n) in the host moments already
            ld = lib.lcx_ld(n)
            rinv = torch.zeros((m, ld), dtype=torch.float64, device=sess.device)
            rinv[:, :n].copy_(torch.from_numpy(np.ascontiguousarray(self.moments["rhoinvrho"], dtype=np.float64)))
            si = torch.as_tensor(np.asarray(self.moments["Si"], dtype=np.float64), device=sess.device)
        sd = torch.as_tensor(np.asarray(self.theta[1], dtype=np.float64), device=sess.device)
        return rinv, ld, si, sd

    def _lowrank_factor(self, with_h=False):
        """Device factor of the ns estimate Sigma = S (Z^T Z + Delta) S (lcx_lowrank_factor): returns (B, ldb, 1/Delta,
        log det Sigma, theta[1]) as CUDA tensors, and with `with_h` also (H, ldh), H = G^-1 G^-T (lcx_lowrank_factor_h).  Built
        from the moments (_lowrank_moments) on every call, about one m x m x n product."""
        torch = _torch()
        rinv, ld, si, sd = self._lowrank_moments()
        sess = self._session()
        lib = sess.lib
        n, m = self.nv, self.m
        ldb = lib.lcx_ld(n)
        b = torch.zeros((m, ldb), dtype=torch.float64, device=sess.device)
        dinv = torch.empty(n, dtype=torch.float64, device=sess.device)
        logdet = torch.empty(1, dtype=torch.float64, device=sess.device)
        if with_h:
            ldh = lib.lcx_ld(m)
            h = torch.empty((m, ldh), dtype=torch.float64, device=sess.device)
            nscr = lib.lcx_lowrank_h_scratch_doubles(m, n)
            scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
            _lib.check(lib.lcx_lowrank_factor_h(sess.h, rinv.data_ptr(), si.data_ptr(), ld, m, n, float(self.eps), sd.data_ptr(),
                                                b.data_ptr(), ldb, dinv.data_ptr(), logdet.data_ptr(), h.data_ptr(), ldh,
                                                scratch.data_ptr(), nscr), "lcx_lowrank_factor_h")
            return b, ldb, dinv, logdet, sd, h, ldh
        nscr = lib.lcx_lowrank_scratch_doubles(m, n)
        scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
        _lib.check(lib.lcx_lowrank_factor(sess.h, rinv.data_ptr(), si.data_ptr(), ld, m, n, float(self.eps), sd.data_ptr(),
                                          b.data_ptr(), ldb, dinv.data_ptr(), logdet.data_ptr(), scratch.data_ptr(), nscr),
                   "lcx_lowrank_factor")
        return b, ldb, dinv, logdet, sd

    def _scores(self, x):
        """(q, log p) of the rows of x as (N,) float64 CUDA tensors: raw rows go through transform's row-block loop and
        lcx_score_rows (standardise + sum x~^2 / Delta, Y = X~ B^T on the DMMA engine, finish)."""
        torch = _torch()
        sess = self._session()
        lib = sess.lib
        N, nv = int(np.shape(x)[0]), int(np.shape(x)[1])
        assert self.nv == nv, "Incorrect number of variables in input, %d instead of %d" % (nv, self.nv)
        b, ldb, dinv, logdet, _sd = self._lowrank_factor()
        maha = torch.empty(N, dtype=torch.float64, device=sess.device)
        logp = torch.empty(N, dtype=torch.float64, device=sess.device)
        if N == 0:
            return maha, logp
        rows = min(self._transform_rows_for(x) or N, N)
        nscr = lib.lcx_score_scratch_doubles(rows, nv, self.m)
        scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
        has_marker = self.missing_values is not None
        marker = float(self.missing_values) if has_marker else 0.0

        def block(lo, hi, xd, dt, impute, mean, sd):
            _lib.check(lib.lcx_score_rows(sess.h, xd.data_ptr(), dt, hi - lo, nv, xd.stride(0), int(has_marker), marker,
                                          impute.data_ptr() if impute is not None else None, mean.data_ptr(), sd.data_ptr(),
                                          b.data_ptr(), ldb, self.m, dinv.data_ptr(), logdet.data_ptr(), maha[lo:hi].data_ptr(),
                                          logp[lo:hi].data_ptr(), scratch.data_ptr(), nscr), "lcx_score_rows")
        self._row_blocks(x, rows, block)
        return maha, logp

    def _conditioned(self, x, imputed=False, scores=True, std=False, n_draws=0, seed=0, first_row=0):
        """lcx_condition_rows over the rows of x in transform's row blocks, without the column-mean pass: returns
        (imputed (N, ld) or None, q (N,) or None, log p (N,) or None, std (N, ld) or None, draws (n_draws, N, ld) or None) as
        CUDA tensors.  With `std` or `n_draws` the rows go through lcx_condition_sample_rows instead (imputed values, no
        scores), its draws from the stream of `seed` with x's first row at global index `first_row`.  Entries that are NaN, or
        equal missing_values, are missing.  The per-class row counts of the call are kept in self._condition_counts."""
        torch = _torch()
        sess = self._session()
        lib = sess.lib
        N, nv = int(np.shape(x)[0]), int(np.shape(x)[1])
        assert self.nv == nv, "Incorrect number of variables in input, %d instead of %d" % (nv, self.nv)
        b, ldb, dinv, logdet, _sd, h, ldh = self._lowrank_factor(with_h=True)
        sample = bool(std or n_draws)
        ld = lib.lcx_ld(nv)
        new = lambda *shape: torch.empty(shape, dtype=torch.float64, device=sess.device)
        out = new(N, ld) if imputed or sample else None
        maha = new(N) if scores and not sample else None
        logp = new(N) if scores and not sample else None
        sdo = new(N, ld) if std else None
        draws = new(n_draws, N, ld) if n_draws else None
        self._condition_counts = np.zeros(8, dtype=np.int64)
        if N == 0:
            return out, maha, logp, sdo, draws
        rows = min(self._transform_rows_for(x) or N, N)
        nscr = (lib.lcx_condition_sample_scratch_doubles if sample else lib.lcx_condition_scratch_doubles)(rows, nv, self.m)
        scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
        has_marker = self.missing_values is not None
        marker = float(self.missing_values) if has_marker else 0.0
        counts = np.zeros(8, dtype=np.int64)
        p = lambda t, lo: t[lo].data_ptr() if t is not None else None

        def block(lo, hi, xd, dt, _impute, mean, sd):
            if sample:
                _lib.check(lib.lcx_condition_sample_rows(
                    sess.h, xd.data_ptr(), dt, hi - lo, nv, xd.stride(0), int(has_marker), marker, mean.data_ptr(), sd.data_ptr(),
                    b.data_ptr(), ldb, self.m, h.data_ptr(), ldh, dinv.data_ptr(), p(out, lo), ld, p(sdo, lo),
                    draws[0, lo].data_ptr() if draws is not None else None, ld, N * ld, seed, first_row + lo, n_draws,
                    counts.ctypes.data_as(C.POINTER(C.c_longlong)), scratch.data_ptr(), nscr), "lcx_condition_sample_rows")
            else:
                _lib.check(lib.lcx_condition_rows(sess.h, xd.data_ptr(), dt, hi - lo, nv, xd.stride(0), int(has_marker), marker,
                                                  mean.data_ptr(), sd.data_ptr(), b.data_ptr(), ldb, self.m, h.data_ptr(), ldh,
                                                  dinv.data_ptr(), logdet.data_ptr(), p(out, lo), ld, p(maha, lo), p(logp, lo),
                                                  counts.ctypes.data_as(C.POINTER(C.c_longlong)), scratch.data_ptr(), nscr),
                           "lcx_condition_rows")
            self._condition_counts += counts
        self._row_blocks(x, rows, block, impute_pass=False)
        return out, maha, logp, sdo, draws

    def _scores_for(self, x, missing):
        if missing == 'impute':
            return self._scores(x)
        if missing == 'marginalize':
            return self._conditioned(x)[1:3]
        raise ValueError("missing must be 'impute' or 'marginalize', not %r" % (missing,))

    def impute(self, x, return_std=False, return_device=False):
        """x with every missing entry (NaN, or equal to missing_values) replaced by its conditional mean given the row's
        observed entries, E[x_M | x_O] under N(theta[0], get_covariance()): an (N, n) float64 ndarray (an (N, n) CUDA tensor
        view with `return_device=True`).  Observed entries come back as the binary64 value of the input, bit for bit; a row
        with nothing observed gets theta[0].  Computed like score_samples(missing='marginalize'): one SPD system per row, of
        order |M| or m whichever is cheaper, from the low-rank-plus-diagonal structure, never an n x n matrix.  The same preconditions and
        errors as score_samples.

        return_std=True returns (imputed, std): std is the conditional standard deviation sqrt(var(x_i | x_O)) of each missing
        entry, in the units of the input, and exactly 0.0 at observed entries (theta[1] for a row with nothing observed).  It
        comes from more triangular sweeps on the factor of the same per-row system; `imputed` is the same bit for bit."""
        res = self._conditioned(x, imputed=True, scores=False, std=return_std)
        out = res[0][:, :self.nv]
        if not return_std:
            return out if return_device else out.cpu().numpy()
        sd = res[3][:, :self.nv]
        return (out, sd) if return_device else (out.cpu().numpy(), sd.cpu().numpy())

    def sample_missing(self, x, n_draws=1, seed=None, first_row=0, return_device=False):
        """Multiple imputation: n_draws completed copies of x, an (n_draws, N, n) float64 ndarray (a CUDA tensor view with
        `return_device=True`).  Each missing entry set x_M of each row is drawn from its conditional distribution
        N(E[x_M | x_O], Cov[x_M | x_O]) under N(theta[0], get_covariance()); observed entries are the binary64 of the input, bit
        for bit.  A row with nothing observed gets unconditional draws, a complete row n_draws copies of itself.  Draw d of
        row l depends only on (seed, first_row + l, d): `first_row` is the global index of x's first row, so a caller that
        splits the rows between calls or ranks gets the same draws as one call.  seed=None takes a seed from numpy's global
        legacy RNG (seeded by Corex(seed=...)).  The same preconditions and errors as impute."""
        n_draws = int(n_draws)
        if n_draws < 1:
            raise ValueError("n_draws must be >= 1")
        seed = self._sample_seed(seed)
        first_row = int(first_row)
        if first_row < 0:
            raise ValueError("first_row must be >= 0")
        draws = self._conditioned(x, scores=False, n_draws=n_draws, seed=seed, first_row=first_row)[4][:, :, :self.nv]
        return draws if return_device else draws.cpu().numpy()

    @staticmethod
    def _sample_seed(seed):
        if seed is None:  # numpy's global legacy RNG, like the reference's seeding at :89
            return int(np.random.randint(np.iinfo(np.int64).max, dtype=np.int64))
        seed = int(seed)
        if not 0 <= seed < 2 ** 64:
            raise ValueError("seed must lie in [0, 2**64)")
        return seed

    def sample(self, n_samples, seed=None, first_row=0, return_device=False):
        """Draws from the fitted Gaussian N(theta[0], get_covariance()): rows first_row .. first_row + n_samples - 1 of one
        stream per (model, seed), an (n_samples, n) float64 ndarray (a CUDA tensor view with `return_device=True`).  Row l
        depends only on (seed, l), so sample(10, s)[3:] equals sample(7, s, first_row=3) bit for bit: a sample larger than
        memory, or one piece per rank, comes in pieces.  seed=None takes a seed from numpy's global legacy RNG (seeded by
        Corex(seed=...)).

        x = theta[0] + theta[1] (Z^T u + Delta^1/2 eps), u ~ N(0, I_m), eps ~ N(0, I_n), from the low-rank-plus-diagonal
        structure of the estimate: O(n m) per row, no n x n matrix (a dense Cholesky would need n^3 / 3 flops and n^2 doubles).
        For 'outliers' the draws are of the estimate's Gaussian itself (no g^-1), as score_samples defines its density.  The
        same preconditions and errors as score_samples; host moments are enough (an unpickled model)."""
        torch = _torch()
        n_samples, first_row = int(n_samples), int(first_row)
        if n_samples < 0 or first_row < 0:
            raise ValueError("n_samples and first_row must be >= 0")
        seed = self._sample_seed(seed)
        rinv, ld, si, sd = self._lowrank_moments()
        sess = self._session()
        lib = sess.lib
        n, m = self.nv, self.m
        if self._theta_dev is None:
            self._theta_dev = tuple(torch.as_tensor(np.asarray(t, dtype=np.float64), device=sess.device) for t in self.theta)
        mean = self._theta_dev[0]
        ldo = lib.lcx_ld(n)
        free, _total = torch.cuda.mem_get_info(sess.device)
        rows = int(self.stream_rows or 32768) if n_samples * ldo * 12 > 0.8 * free else n_samples
        rows = max(1, min(rows, n_samples))
        out = torch.empty((n_samples, ldo), dtype=torch.float64, device=sess.device) if return_device else \
            np.empty((n_samples, n), dtype=np.float64)
        buf = None if return_device else torch.empty((rows, ldo), dtype=torch.float64, device=sess.device)
        nscr = lib.lcx_sample_scratch_doubles(rows, n, m)
        scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
        for lo in range(0, n_samples, rows):
            hi = min(n_samples, lo + rows)
            dst = out[lo:hi] if return_device else buf
            _lib.check(lib.lcx_sample_rows(sess.h, rinv.data_ptr(), si.data_ptr(), ld, m, n, float(self.eps), mean.data_ptr(),
                                           sd.data_ptr(), seed, first_row + lo, hi - lo, dst.data_ptr(), ldo, scratch.data_ptr(),
                                           nscr), "lcx_sample_rows")
            if not return_device:
                out[lo:hi] = buf[:hi - lo, :n].cpu().numpy()
        return out[:, :n] if return_device else out

    def score_samples(self, x, missing='impute'):
        """log p(x_l) under N(theta[0], get_covariance()) for every row, in the units of the input: an (N,) float64 ndarray.

        For gaussianize='standard' this is multivariate_normal(theta[0], get_covariance()).logpdf(x).  For 'outliers' it is
        the same Gaussian density of the raw x -- theta and get_covariance() as the model reports them; g() is deliberately
        not applied, so the density is that of the covariance estimate itself.  Computed in binary64 from the low-rank-plus-
        diagonal structure of the estimate (O(n m) per row, no n x n matrix); results do not depend on how the rows are
        blocked.  Raises LinAlgError when the estimate is not positive definite (some Delta_i <= 0).

        missing='impute' (default): missing entries (missing_values) are imputed with the new data's column means, as
        transform does, and the row is scored as if complete.  missing='marginalize': the marginal density of the observed
        entries, log N(x_O; theta[0]_O, Sigma_OO), with NaN entries missing too; a complete row scores exactly as with
        'impute', a row with nothing observed scores 0."""
        return self._scores_for(x, missing)[1].cpu().numpy()

    def mahalanobis(self, x, missing='impute'):
        """Squared Mahalanobis distances (x_l - theta[0])^T Sigma^-1 (x_l - theta[0]) of the rows: an (N,) float64 ndarray.
        missing='marginalize' gives the distance of the observed part under Sigma_OO (see score_samples)."""
        return self._scores_for(x, missing)[0].cpu().numpy()

    def score(self, x, missing='impute', sample_weight=None):
        """Mean log-likelihood of the rows of x (the mean of score_samples(x, missing)).  With `comm` set, x is this rank's row
        block and the mean is over all ranks' rows; every rank returns the same value.  sample_weight (one non-negative weight
        per row, as for fit): the weighted mean sum w log p / sum w over all ranks."""
        red = self._reducer()
        weights = None
        if sample_weight is not None:
            weights = self._sample_weights(sample_weight, int(np.shape(x)[0]), red)
        logp = self._scores_for(x, missing)[1].cpu().numpy()
        if weights is None:
            return float(red.sum_scalar(float(np.sum(logp)))) / float(red.sum_scalar(len(logp)))
        w, w_total = weights
        return float(red.sum_scalar(float(np.sum(w * logp)))) / w_total

    def get_precision(self, block_rows=4096, out=None, block_callback=None):
        """n x n precision matrix Sigma^-1 = S^-1 (Delta^-1 - B^T B) S^-1 of the covariance estimate, in row blocks on the
        device; `block_rows`, `out` and `block_callback` as for get_covariance."""
        lib = self._session().lib
        n = self.nv
        b, ldb, dinv, _logdet, sd = self._lowrank_factor()

        def fill(r0, rows, dst, ldd):
            _lib.check(lib.lcx_precision_rows(self._sess.h, b.data_ptr(), ldb, self.m, n, dinv.data_ptr(), sd.data_ptr(), r0,
                                              rows, dst.data_ptr(), ldd), "lcx_precision_rows")
        return self._n_by_n_rows(fill, block_rows, out, block_callback)

    def conditional(self, observed, targets=None):
        """The fitted Gaussian N(theta[0], get_covariance()) conditioned on a fixed set of observed columns: a
        ConditionalGaussian that predicts, scores and draws the `targets` (default: every column not in `observed`) for many
        rows that all observe the columns `observed`, in that order.  Building it factors the order-m system of the pattern
        once (about m^2 (|O| + |T|) + m^3 / 3 flops); a row then costs O(m (|O| + |T|)), as scoring does.  Indices out of
        range, duplicated or in both lists raise ValueError; the preconditions and errors are those of score_samples."""
        return ConditionalGaussian(self, observed, targets)


class ConditionalGaussian(object):
    """N(theta[0], get_covariance()) of a Corex model conditioned on the columns `observed` (Corex.conditional).

    In standardised space x~ = (x - theta[0]) / theta[1], with Sigma~ = Z^T Z + Delta (DESIGN.md section 8) and
    E_O = I + Z_O Delta_O^-1 Z_O^T = L L^T,  A = L^-1 Z_O Delta_O^-1,  P = L^-1 Z_T,  v = A x~_O:
        E[x~_T | x~_O] = P^T v,   Cov[x~_T | x~_O] = Delta_T + P^T P   (the same for every row),
        log p(x_O) = -(|O| log 2 pi + log det Sigma_OO + sum_O x~_i^2 / Delta_i - |v|^2) / 2.
    The object holds its own device factor (A, P, the gathered theta and Delta, log det Sigma_OO), built once: refitting the
    parent does not change it, and it pickles with host copies that give the same bits.

    x_obs arguments hold the observed columns only, in the order of `observed`: a float32 / float64 ndarray, a CUDA tensor,
    or a row provider with `.shape` and row slicing, blocked as transform blocks its input.  A missing entry (NaN, or the
    parent's missing_values) raises ValueError: rows with their own missing patterns go to Corex.impute."""

    _as_input = Corex._as_input
    _upload = Corex._upload
    _n_by_n_rows = Corex._n_by_n_rows
    _DEVICE = ("_a", "_p", "_ocols", "_tcols", "_logdet")

    def __init__(self, model, observed, targets=None):
        torch = _torch()
        n = int(model.nv)
        observed = self._indices(observed, n, "observed")
        if targets is None:
            keep = np.ones(n, dtype=bool)
            keep[observed] = False
            targets = np.flatnonzero(keep)
        else:
            targets = self._indices(targets, n, "targets")
            if np.intersect1d(observed, targets).size:
                raise ValueError("observed and targets must be disjoint")
        rinv, ld, si, sd = model._lowrank_moments()
        self.observed, self.targets = observed, targets
        self.m, self.nv = int(model.m), n
        self.missing_values = model.missing_values
        self.input_dtype = model.input_dtype
        self.stream_rows = model.stream_rows
        self._comm = model._comm
        self._device = model._device
        self._sess = None
        sess = self._session()
        lib = sess.lib
        m, no, nt = self.m, len(observed), len(targets)
        new = lambda *shape: torch.zeros(shape, dtype=torch.float64, device=sess.device)
        self._a, self._p = new(m, lib.lcx_ld(no)), new(m, lib.lcx_ld(nt))
        self._ocols, self._tcols, self._logdet = new(3 * no), new(5 * nt), new(1)
        mean = torch.as_tensor(np.asarray(model.theta[0], dtype=np.float64), device=sess.device)
        idx = lambda a: torch.as_tensor(a.astype(np.int32), device=sess.device) if len(a) else None
        oi, ti = idx(observed), idx(targets)
        nscr = lib.lcx_conditional_factor_scratch_doubles(m, no, nt)
        scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
        ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None
        _lib.check(lib.lcx_conditional_factor(sess.h, rinv.data_ptr(), si.data_ptr(), ld, m, n, float(model.eps), mean.data_ptr(),
                                              sd.data_ptr(), ptr(oi), no, ptr(ti), nt, ptr(self._a), self._a.shape[1],
                                              ptr(self._p), self._p.shape[1], ptr(self._ocols), ptr(self._tcols),
                                              self._logdet.data_ptr(), scratch.data_ptr(), nscr), "lcx_conditional_factor")

    @staticmethod
    def _indices(v, n, what):
        a = np.asarray(v)
        if a.size == 0:
            return np.zeros(0, dtype=np.int64)
        if a.ndim != 1 or a.dtype.kind not in "iu":
            raise ValueError("%s must be a 1-d sequence of column indices" % what)
        a = a.astype(np.int64)
        if np.any((a < 0) | (a >= n)):
            raise ValueError("%s has a column index outside [0, %d)" % (what, n))
        if np.unique(a).size != a.size:
            raise ValueError("%s has a duplicate column index" % what)
        return a

    def __getstate__(self):
        d = dict(self.__dict__)
        d["_sess"] = d["_comm"] = None
        for k in self._DEVICE:
            d[k] = d[k].cpu().numpy() if not isinstance(d[k], np.ndarray) else d[k]
        return d

    def _session(self):
        if self._sess is None:
            self._sess = _DeviceSession(_lib.PRECISION_FP64, self._device)
        return self._sess

    def _factor(self):
        """The device factor (A, P, ocols, tcols, log det), uploaded once after unpickling."""
        torch = _torch()
        dev = self._session().device
        for k in self._DEVICE:
            v = getattr(self, k)
            if isinstance(v, np.ndarray):
                setattr(self, k, torch.as_tensor(v, device=dev))
        return tuple(getattr(self, k) for k in self._DEVICE)

    def _check(self, rc, what):
        if rc == _lib.ERR_MISSING:
            raise ValueError("x_obs has a missing entry (NaN or missing_values) in an observed column; a ConditionalGaussian "
                             "conditions every row on all of its observed columns -- use Corex.impute for rows with missing "
                             "entries of their own")
        return _lib.check(rc, what)

    def _blocks(self, x, n_draws=1):
        """(N, row-block size) of x_obs after its checks; blocks as transform's (whole arrays when they fit)."""
        torch = _torch()
        shape = tuple(np.shape(x))
        if len(shape) != 2 or shape[1] != len(self.observed):
            raise ValueError("x_obs must have shape (N, %d): the observed columns, in the order of `observed`"
                             % len(self.observed))
        N = int(shape[0])
        if not isinstance(x, (np.ndarray, torch.Tensor, list, tuple)):
            return N, int(self.stream_rows or 32768)
        lib = self._session().lib
        width = lib.lcx_ld(len(self.observed)) + n_draws * lib.lcx_ld(len(self.targets))
        free, _total = torch.cuda.mem_get_info(self._session().device)
        return N, (int(self.stream_rows or 32768) if N * width * 12 > 0.8 * free else max(N, 1))

    def _rows(self, x, per_block, n_draws=1):
        """per_block(lo, hi, x pointer, dtype, ldx) over the row blocks of x_obs, with the scratch of the block size."""
        torch = _torch()
        N, rows = self._blocks(x, n_draws)
        if N == 0:
            return N
        sess = self._session()
        nscr = sess.lib.lcx_conditional_scratch_doubles(min(rows, N), len(self.observed), self.m)
        scratch = torch.empty(nscr, dtype=torch.float64, device=sess.device)
        for lo in range(0, N, rows):
            hi = min(N, lo + rows)
            if len(self.observed):
                xd = self._as_input(x[lo:hi])
                per_block(lo, hi, xd.data_ptr(), _lib.F32 if xd.dtype == torch.float32 else _lib.F64, xd.stride(0), scratch)
            else:
                per_block(lo, hi, None, _lib.F64, 0, scratch)
        return N

    def _conditioned(self, x, pred, scores):
        torch = _torch()
        sess = self._session()
        lib = sess.lib
        a, p, oc, tc, logdet = self._factor()
        no, nt = len(self.observed), len(self.targets)
        N = int(np.shape(x)[0]) if len(np.shape(x)) == 2 else 0
        new = lambda *shape: torch.empty(shape, dtype=torch.float64, device=sess.device)
        out = new(N, p.shape[1]) if pred else None
        maha, logp = (new(N), new(N)) if scores else (None, None)
        has_marker = self.missing_values is not None
        marker = float(self.missing_values) if has_marker else 0.0
        at = lambda t, lo: t[lo].data_ptr() if t is not None else None

        def block(lo, hi, xp, dt, ldx, scratch):
            self._check(lib.lcx_conditional_rows(sess.h, xp, dt, hi - lo, no, ldx, int(has_marker), marker, a.data_ptr(), a.shape[1],
                                                 oc.data_ptr(), p.data_ptr(), p.shape[1], nt, tc.data_ptr(), self.m,
                                                 logdet.data_ptr(), at(out, lo) if nt else None, p.shape[1], at(maha, lo),
                                                 at(logp, lo), scratch.data_ptr(), scratch.numel()), "lcx_conditional_rows")
        self._rows(x, block)
        return out, maha, logp

    def predict(self, x_obs, return_device=False):
        """E[x_T | x_O] in the units of the input: an (N, |T|) float64 ndarray (a CUDA tensor view with return_device=True)."""
        out = self._conditioned(x_obs, True, False)[0][:, :len(self.targets)]
        return out if return_device else out.cpu().numpy()

    @property
    def std(self):
        """(|T|,) conditional standard deviations theta1_T sqrt(Delta_T + |p_t|^2), the same for every row."""
        nt = len(self.targets)
        return self._factor()[3][4 * nt:5 * nt].cpu().numpy()

    def get_covariance(self, block_rows=4096, out=None, block_callback=None):
        """The |T| x |T| conditional covariance theta1_T (Delta_T + P^T P) theta1_T, in row blocks on the device, with
        Corex.get_covariance's output options (`out` ndarray / memmap / CUDA tensor, `block_callback`)."""
        lib = self._session().lib
        _a, p, _oc, tc, _ld = self._factor()
        nt = len(self.targets)

        def fill(r0, rows, dst, ldd):
            _lib.check(lib.lcx_conditional_covariance_rows(self._sess.h, p.data_ptr(), p.shape[1], self.m, nt, tc.data_ptr(), r0,
                                                           rows, dst.data_ptr(), ldd), "lcx_conditional_covariance_rows")
        return self._n_by_n_rows(fill, min(block_rows, 65534), out, block_callback, n=nt)

    def sample(self, x_obs, n_draws=1, seed=None, first_row=0, return_device=False):
        """n_draws draws of x_T from N(E[x_T | x_O], Cov[x_T | x_O]) for every row: an (n_draws, N, |T|) float64 ndarray (a
        CUDA tensor view with return_device=True).  Draw d of row l depends only on (seed, first_row + l, d), so rows split
        between calls or ranks get the same draws as one call.  seed=None takes a seed from numpy's global legacy RNG, as
        Corex.sample does."""
        torch = _torch()
        n_draws = int(n_draws)
        if n_draws < 1:
            raise ValueError("n_draws must be >= 1")
        seed = Corex._sample_seed(seed)
        first_row = int(first_row)
        if first_row < 0:
            raise ValueError("first_row must be >= 0")
        sess = self._session()
        lib = sess.lib
        a, p, oc, tc, _logdet = self._factor()
        no, nt = len(self.observed), len(self.targets)
        N = int(np.shape(x_obs)[0]) if len(np.shape(x_obs)) == 2 else 0
        ldo = p.shape[1]
        draws = torch.empty((n_draws, N, ldo), dtype=torch.float64, device=sess.device)
        has_marker = self.missing_values is not None
        marker = float(self.missing_values) if has_marker else 0.0

        def block(lo, hi, xp, dt, ldx, scratch):
            self._check(lib.lcx_conditional_sample_rows(sess.h, xp, dt, hi - lo, no, ldx, int(has_marker), marker, a.data_ptr(),
                                                        a.shape[1], oc.data_ptr(), p.data_ptr(), ldo, nt, tc.data_ptr(), self.m,
                                                        draws[0, lo].data_ptr() if nt else None, ldo, N * ldo, seed,
                                                        first_row + lo, n_draws, scratch.data_ptr(), scratch.numel()),
                        "lcx_conditional_sample_rows")
        self._rows(x_obs, block, n_draws)
        out = draws[:, :, :nt]
        return out if return_device else out.cpu().numpy()

    def score_samples(self, x_obs):
        """log p(x_O) of every row under the marginal N(theta[0]_O, Sigma_OO): an (N,) float64 ndarray (0 when O is empty)."""
        return self._conditioned(x_obs, False, True)[2].cpu().numpy()

    def mahalanobis(self, x_obs):
        """Squared Mahalanobis distances of the rows under Sigma_OO: an (N,) float64 ndarray."""
        return self._conditioned(x_obs, False, True)[1].cpu().numpy()

    def score(self, x_obs):
        """Mean of score_samples(x_obs); with the parent's `comm`, x_obs is this rank's row block and the mean is over all
        ranks' rows (every rank returns the same value)."""
        logp = self.score_samples(x_obs)
        red = Reducer(self._comm)
        return float(red.sum_scalar(float(np.sum(logp)))) / float(red.sum_scalar(len(logp)))
