"""Helpers shared by the -m gpu tests (test infrastructure)."""
import importlib.machinery
import importlib.util
import os
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref", "omniserve_backend")


def t(x, dev="cuda"):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


_ref_cache = {}


def ref_module(name):
    """Load one of the reference's own extension modules rebuilt for sm_100 by oracle/build_ref.py
    (oracle/_ref/omniserve_backend/<name>.so).  Returns None when it was not shipped."""
    if name in _ref_cache:
        return _ref_cache[name]
    path = os.path.join(REF_DIR, f"{name}.so")
    mod = None
    if os.path.exists(path):
        loader = importlib.machinery.ExtensionFileLoader(name, path)
        spec = importlib.util.spec_from_loader(name, loader)
        mod = importlib.util.module_from_spec(spec)
        loader.exec_module(mod)
    _ref_cache[name] = mod
    return mod


GOLDEN_REF = os.path.join(ROOT, "tests", "golden", "ref_kernels.npz")
RECORD_REF = os.environ.get("OB_RECORD_REF_GOLDEN")   # path of an .npz that live reference runs are recorded into
SAMPLE = 1024


class RefOutputs:
    """What the reference's own kernel computed for one test case.  Live (oracle/_ref present): the full arrays.  Otherwise
    the record in tests/golden/ref_kernels.npz: per array a fixed seeded sample of SAMPLE elements (all of them when the
    array is smaller), its shape and its largest magnitude, plus any statistic the test derived from the full arrays."""

    def __init__(self, case, arrays, bases=None):
        self.case, self.arrays, self.bases = case, arrays, bases or {}
        self.golden = None
        if arrays is None:
            assert os.path.exists(GOLDEN_REF), f"{GOLDEN_REF} missing"
            self.golden = np.load(GOLDEN_REF)
            assert any(k.startswith(case + "|") for k in self.golden.files), f"no recorded reference outputs for {case}"

    def _key(self, name, what):
        return f"{self.case}|{name}|{what}"

    def _g(self, name, what):
        k = self._key(name, what)
        assert k in self.golden.files, f"{k} not recorded in {GOLDEN_REF}"
        return self.golden[k]

    def pair(self, name, ours):
        """(ours, reference) as flat arrays over the same elements: all of them live, the recorded sample otherwise."""
        ours = ours.cpu().numpy() if torch.is_tensor(ours) else np.asarray(ours)
        if self.golden is None:
            ref = self.arrays[name]
            assert ours.shape == ref.shape
            return ours.reshape(-1), ref.reshape(-1)
        assert tuple(ours.shape) == tuple(self._g(name, "shape")), f"{name}: shape {ours.shape}"
        if self._key(name, "didx") in self.golden.files:   # the whole array: its input state plus the recorded changes
            ref = np.array(self.bases[name]).reshape(-1)
            ref[self._g(name, "didx")] = self._g(name, "dval")
            return ours.reshape(-1), ref
        v = self._g(name, "v")
        if v.size == ours.size:                             # recorded whole
            return ours.reshape(-1), v
        return ours.reshape(-1)[_sample_index(self.case, name, ours.size)], v

    def absmax(self, name):
        if self.golden is None:
            return float(np.abs(self.arrays[name].astype(np.float64)).max())
        return float(self._g(name, "absmax"))

    def stat(self, name, fn):
        """fn(full reference arrays) -> float, computed live (and recorded) or read from the record."""
        if self.golden is None:
            v = float(fn(self.arrays))
            if RECORD_REF:
                _record({self._key(name, "stat"): np.float64(v)})
            return v
        return float(self._g(name, "stat"))


def _sample_index(case, name, size):
    if size <= SAMPLE:
        return np.arange(size)
    rng = np.random.default_rng(zlib.crc32(f"{case}|{name}".encode()))
    return np.sort(rng.choice(size, SAMPLE, replace=False))


def _record(entries):
    old = dict(np.load(RECORD_REF)) if os.path.exists(RECORD_REF) else {}
    old.update(entries)
    np.savez_compressed(RECORD_REF, **old)


def reference_outputs(case, live, run, bases=None, whole=()):
    """Outputs of the reference's own kernels for test case `case`: run() -> {name: np.ndarray} when `live` (the
    oracle/_ref modules the case needs are present; recorded when OB_RECORD_REF_GOLDEN is set), the committed record
    otherwise.  A case without a record fails: the comparison with the reference is never skipped.
    bases: {name: the array's state before the kernel ran} for arrays the kernel changes in a few places (KV page pools
    it appends one token to): those are recorded as their changed elements and replayed whole.  whole: names of small
    arrays recorded in full rather than sampled."""
    bases = {k: (v.cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in (bases or {}).items()}
    if not live:
        return RefOutputs(case, None, bases)
    arrays = {k: (v.cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in run().items()}
    if RECORD_REF:
        rec = {}
        for name, a in arrays.items():
            k = f"{case}|{name}|"
            if name in bases:
                d = np.flatnonzero(a.reshape(-1) != bases[name].reshape(-1))
                rec[k + "didx"], rec[k + "dval"] = d, a.reshape(-1)[d]
            elif name in whole:
                rec[k + "v"] = a.reshape(-1)
            else:
                rec[k + "v"] = a.reshape(-1)[_sample_index(case, name, a.size)]
            rec[k + "shape"] = np.asarray(a.shape, np.int64)
            rec[k + "absmax"] = np.float64(np.abs(a.astype(np.float64)).max()) if a.size else np.float64(0)
        _record(rec)
    return RefOutputs(case, arrays)


def make_gemm_inputs(M, N, K, seed, per_group=False):
    from oracle import w4a8 as ow
    rng = np.random.default_rng(seed)
    d = {}
    q = rng.integers(0, 16, (N, K), dtype=np.uint8)
    d["a"] = rng.integers(-127, 128, (M, K), dtype=np.int8)
    d["s1"] = rng.uniform(0.005, 0.02, N).astype(np.float16)
    d["sa"] = rng.uniform(0.01, 0.05, M).astype(np.float16)
    d["qw"] = ow.pack_w4(q)
    if per_group:
        ng = K // 128
        s2 = rng.integers(1, 9, (N, ng)).astype(np.int64)
        z = rng.integers(0, 16, (N, ng)).astype(np.int64)
        d["s2"] = ow.pack_s2(s2).astype(np.int8)
        d["z2"] = (ow.pack_s2(-z) * ow.pack_s2(s2)).astype(np.int8)
    else:
        z = rng.integers(0, 16, N).astype(np.float32)
        d["szs"] = (z * d["s1"].astype(np.float32)).astype(np.float16)
        d["ssum"] = (d["a"].astype(np.float32) * d["sa"].astype(np.float32)[:, None]).sum(1).astype(np.float16)
    return d


def make_kv_case(B, Hq, Hkv, lens, seed, extra_pages=2, k_stats_subchunks=0):
    from oracle import kv4 as okv
    rng = np.random.default_rng(seed)
    Dh = 128
    n_pages = sum((l + 63) // 64 for l in lens) + extra_pages
    cache = okv.PagedKV4(n_pages, Hkv, Dh, k_stats_subchunks)
    perm = rng.permutation(n_pages)
    max_pages = max((l + 63) // 64 for l in lens)
    bt = np.zeros((B, max_pages), np.int64)
    c = 0
    for b, l in enumerate(lens):
        for j in range((l + 63) // 64):
            bt[b, j] = perm[c]
            c += 1
    okv.fill_random(cache, bt, [l - 1 for l in lens], rng)
    q = rng.standard_normal((B, Hq, Dh)).astype(np.float16)
    k = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    v = rng.standard_normal((B, Hkv, Dh)).astype(np.float16)
    return cache, bt, q, k, v


def device_tables(cache, bt):
    kpool, vpool = t(cache.k_pool), t(cache.v_pool)
    B, P = bt.shape
    ptrs = np.zeros((B, 2, P), np.int64)
    ptrs[:, 0] = kpool.data_ptr() + bt * cache.k_page_bytes
    ptrs[:, 1] = vpool.data_ptr() + bt * cache.v_page_bytes
    return kpool, vpool, t(ptrs)


def qkv_views(q, k, v):
    """q,k,v as strided views into one [B,(Hq+2Hkv)*Dh] buffer like the model passes them (llama_w4a8_unpad.py:343-349)."""
    B, Hq, Dh = q.shape
    Hkv = k.shape[1]
    qkv = torch.cat([t(q).reshape(B, -1), t(k).reshape(B, -1), t(v).reshape(B, -1)], dim=1).contiguous()
    return (qkv, qkv[:, :Hq * Dh].view(B, Hq, Dh), qkv[:, Hq * Dh:(Hq + Hkv) * Dh].view(B, Hkv, Dh),
            qkv[:, (Hq + Hkv) * Dh:].view(B, Hkv, Dh))


def assert_k_pool_equal(got_pool, cache, max_stat_ulp=2, max_stat_frac=1e-3, max_pos=0):
    """K pages: nibbles, scales and zeros bit-exact; the kmax / kmin statistics (raw post-RoPE fp16 keys) may differ
    from the numpy oracle in the last bits of a few elements (fp32 sincosf on the device vs numpy's libm).  The rotation
    angle pos / base^(2i/d) is formed in fp32 on both sides, so a one-ulp difference between CUDA's powf and numpy's is
    multiplied by the position: `max_pos` widens the ulp budget accordingly (1 ulp(fp32) * pos radians)."""
    max_stat_ulp = max_stat_ulp + max_pos // 200
    got = got_pool.cpu().numpy() if hasattr(got_pool, "cpu") else got_pool
    cut = cache.data_bytes + cache.sz_bytes
    np.testing.assert_array_equal(got[:, :cut], cache.k_pool[:, :cut])
    if cache.stats_bytes:
        a = np.ascontiguousarray(got[:, cut:]).view(np.int16).astype(np.int32)
        b = np.ascontiguousarray(cache.k_pool[:, cut:]).view(np.int16).astype(np.int32)
        diff = np.abs(a - b)
        assert diff.max() <= max_stat_ulp, f"statistics differ by {diff.max()} fp16 ulps"
        assert (diff != 0).mean() <= max_stat_frac
