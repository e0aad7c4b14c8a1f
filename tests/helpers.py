"""Shared helpers for the parity tests (test infrastructure; may use oracle/)."""
import hashlib
import io
import json
import os
import types
import zipfile

import numpy as np

from oracle import oracle as O

RTOL = 1e-4  # BASELINE.json north_star: fp distances within 1e-4 relative
ATOL = 2e-6
TAPES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_tapes")


def _digest_into(h, x):
    if isinstance(x, (np.ndarray, np.generic)):
        a = np.ascontiguousarray(x)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(b"[")
        for v in x:
            _digest_into(h, v)
        h.update(b"]")
    elif isinstance(x, dict):
        for k in sorted(x):
            h.update(str(k).encode())
            _digest_into(h, x[k])
    elif x is None or isinstance(x, (bool, int, float, str)):
        h.update(repr(x).encode())
    else:  # an oracle object (FtProblem): its public state
        _digest_into(h, {k: v for k, v in vars(x).items() if not k.startswith("_")})


def digest(*inputs):
    h = hashlib.blake2b(digest_size=8)
    _digest_into(h, inputs)
    return np.frombuffer(h.digest(), np.uint64)[0]


def _flatten(x, arrays):
    """an output of the reference (arrays, scalars, strings, None, nested in tuples / lists / dicts) -> JSON-able spec + arrays"""
    if isinstance(x, dict):
        return {"d": {k: _flatten(v, arrays) for k, v in x.items()}}
    if isinstance(x, (tuple, list)):
        return {"t": [_flatten(v, arrays) for v in x]}
    if x is None:
        return None
    arrays.append(np.asarray(x))
    return len(arrays) - 1


def _unflatten(spec, arrays):
    if spec is None:
        return None
    if isinstance(spec, int):
        a = arrays[spec]
        return a.item() if a.ndim == 0 else a
    if "d" in spec:
        return {k: _unflatten(v, arrays) for k, v in spec["d"].items()}
    return tuple(_unflatten(v, arrays) for v in spec["t"])


def _narrowest(a):
    """integer arrays are stored in the narrowest integer type that holds their values, labels (row << 32) as row ids: (array, shift)"""
    if a.dtype.kind not in "iu" or a.size == 0:
        return a, 0
    shift = 32 if a.dtype == np.uint64 and not (a & np.uint64(0xFFFFFFFF)).any() else 0
    if shift:
        a = a >> np.uint64(32)
    lo, hi = int(a.min()), int(a.max())
    for t in (np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32):
        if np.iinfo(t).min <= lo and hi <= np.iinfo(t).max:
            return a.astype(t), shift
    return a, shift


class RefTape:
    """Outputs of the reference's own code (oracle/_ref) for one test, stored under tests/golden/ref_tapes/ so that the test compares
    with the reference where the reference is not available.  tape(run, *inputs) returns run()'s result: recorded from the reference
    when RX_RECORD_REF_TAPES names an output directory (needs oracle/_ref), otherwise replayed in call order, each call checked
    against a digest of its inputs so that a tape can only answer the question it was recorded for, and every recorded call must be
    asked for again.  A test without a stored tape (its reference state is too large to store) calls the reference directly.
    tape.proxy(make) stands for a reference object whose method calls go through the tape."""

    def __init__(self, name):
        self.name = name
        self.record_dir = os.environ.get("RX_RECORD_REF_TAPES")
        self.calls = []
        # no stored tape: the test asks the reference itself (and skips where it is not built)
        self.live = not self.record_dir and not os.path.exists(os.path.join(TAPES, f"{name}.npz"))
        if not self.record_dir and not self.live:
            self.z = np.load(os.path.join(TAPES, f"{name}.npz"))
            self.keys, self.specs, self.meta, self.dtypes = self.z["keys"], self.z["specs"], self.z["meta"], self.z["dtypes"]
            self.first = np.searchsorted(self.meta[:, 0], np.arange(len(self.keys) + 1))

    def __call__(self, run, *inputs):
        if self.live:
            return run()
        key = digest(*inputs)
        if self.record_dir:
            out = run()
            self.calls.append((key, out))
            return out
        i = len(self.calls)
        assert i < len(self.keys), f"{self.name}: more reference calls than recorded"
        assert self.keys[i] == key, f"{self.name}: call {i} has other inputs than the recorded one (re-record the tape)"
        self.calls.append(key)
        arrays = []
        for _, pool, off, size, ndim, s0, s1, s2, dt, shift in self.meta[self.first[i]:self.first[i + 1]]:
            a = self.z[f"pool{pool}"][off:off + size].reshape((s0, s1, s2)[:ndim])
            a = a if dt < 0 else a.astype(self.dtypes[dt])
            arrays.append(a << np.uint64(shift) if shift else a)
        return _unflatten(json.loads(str(self.specs[i])), arrays)

    def proxy(self, make, *inputs):
        return _RefProxy(self, make, inputs)

    def save(self):
        if self.live:
            return
        if not self.record_dir:
            assert len(self.calls) == len(self.keys), f"{self.name}: {len(self.keys) - len(self.calls)} recorded reference calls never asked for"
            return
        pools, meta, keys, specs, dtypes = [], [], [], [], []
        for i, (key, out) in enumerate(self.calls):
            keys.append(key)
            arrays = []
            specs.append(json.dumps(_flatten(out, arrays)))
            for a in arrays:
                assert a.ndim <= 3, a.shape
                n, shift = _narrowest(a)
                dt = -1
                if n.dtype != a.dtype:
                    if a.dtype.str not in dtypes:
                        dtypes.append(a.dtype.str)
                    dt = dtypes.index(a.dtype.str)
                p = next((k for k, pl in enumerate(pools) if pl[0].dtype == n.dtype), None)
                if p is None:
                    pools.append([])
                    p = len(pools) - 1
                off = sum(x.size for x in pools[p])
                pools[p].append(n.ravel())
                meta.append([i, p, off, a.size, a.ndim] + list(a.shape) + [0] * (3 - a.ndim) + [dt, shift])
        arrays = dict(keys=np.array(keys, np.uint64), specs=np.array(specs), dtypes=np.array(dtypes, dtype="U8"),
                      meta=np.array(meta, np.int64).reshape(-1, 10), **{f"pool{p}": np.concatenate(pl) for p, pl in enumerate(pools)})
        os.makedirs(self.record_dir, exist_ok=True)
        save_npz_lzma(os.path.join(self.record_dir, f"{self.name}.npz"), arrays)


def save_npz_lzma(path, arrays):
    """an .npz that np.load reads, its members LZMA-compressed (about 10 % smaller than np.savez_compressed on these tapes)"""
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as f:
        for name, a in arrays.items():
            buf = io.BytesIO()
            np.save(buf, a)
            f.writestr(f"{name}.npy", buf.getvalue())


class _RefProxy:
    """A reference object (RefHnsw, RefIvf, ...) behind a tape: created by make() only when recording; method results (generators
    drained into tuples) are recorded / replayed under a digest of the method name, the arguments and the object's own inputs."""

    def __init__(self, tape, make, inputs):
        self._tape, self._make, self._inputs, self._obj = tape, make, digest(*inputs), None

    def real(self):
        if self._obj is None:
            self._obj = self._make()
        return self._obj

    def __getattr__(self, method):
        def call(*args, **kwargs):
            def run():
                out = getattr(self.real(), method)(*args, **kwargs)
                return tuple(out) if isinstance(out, types.GeneratorType) else out
            return self._tape(run, self._inputs, method, args, kwargs)
        return call


def prep_query(metric, q, use_ref=None):
    return O.normalize_copy(q, use_ref)[0] if metric == O.COS else np.ascontiguousarray(q, np.float32)


def assert_same_knn(d_gpu, l_gpu, d_ref, l_ref, ctx=""):
    """Distances within RTOL; ids exact wherever neighbouring reference distances are separated by more than the fp noise
    (the reference itself is not bit-reproducible across its SSE/AVX/AVX-512 kernels, SURVEY.md §8a rule 6).  Inside a group
    of near-equal distances the order may differ; the last group may also trade members with rows just outside the top-k."""
    d_gpu, d_ref = np.asarray(d_gpu), np.asarray(d_ref)
    l_gpu, l_ref = np.asarray(l_gpu), np.asarray(l_ref)
    assert len(d_gpu) == len(d_ref), (ctx, len(d_gpu), len(d_ref))
    assert np.allclose(d_gpu, d_ref, rtol=RTOL, atol=ATOL), (ctx, d_gpu, d_ref)
    if (l_gpu == l_ref).all():
        return
    noise = RTOL * np.maximum(np.abs(d_ref), 1e-2)
    n = len(d_ref)
    i = 0
    while i < n:
        j = i
        while j + 1 < n and d_ref[j + 1] - d_ref[j] <= noise[j]:
            j += 1
        if j + 1 < n:
            assert set(l_ref[i:j + 1].tolist()) == set(l_gpu[i:j + 1].tolist()), (ctx, i, j, l_gpu, l_ref, d_ref)
        i = j + 1


def numpy_dists(metric, q, vecs, norm_coefs=None):
    """fp64 distances in map space (for property checks, not for bit parity)."""
    q64, v64 = q.astype(np.float64), vecs.astype(np.float64)
    if metric == O.L2:
        return ((v64 - q64) ** 2).sum(1)
    d = -(v64 @ q64)
    if metric == O.COS:
        d = d / np.sqrt((v64 ** 2).sum(1))
    return d
