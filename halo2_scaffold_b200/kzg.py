"""
Host-side mirror of halo2_proofs::poly::kzg::commitment::ParamsKZG for the callers of
best_multiexp ([UP] halo2_proofs/src/poly/kzg/commitment.rs, SURVEY.md row a7): the two SRS vectors
`g` and `g_lagrange` are registered once (device resident on every GPU), and `commit` /
`commit_lagrange` are MSMs over their prefixes.  The `Blind` argument of the reference is ignored
by KZG and therefore absent here.
"""
from __future__ import annotations

import numpy as np

from . import _lib


class SerdeFormat:
    """[UP] halo2_proofs::SerdeFormat"""
    Processed, RawBytes, RawBytesUnchecked = 0, 1, 2


class ParamsKZG:
    def __init__(self, k: int, g: np.ndarray, g_lagrange: np.ndarray, lib=None, g2_bytes: bytes = b"", _handles=None):
        self.lib = lib or _lib.load()
        if self.lib.device_count() == 0:
            self.lib.init(0)
        self.k = k
        self.n = 1 << k
        self.g = np.ascontiguousarray(g, dtype=np.uint64).reshape(-1, 8)
        self.g_lagrange = np.ascontiguousarray(g_lagrange, dtype=np.uint64).reshape(-1, 8)
        self.g2_bytes = g2_bytes                       # g2 | s_g2 as stored; G2 arithmetic is the verifier's (host) business
        assert self.g.shape[0] == self.n and self.g_lagrange.shape[0] == self.n
        if _handles:
            self._g, self._g_lagrange = _handles
        else:
            self._g = self.lib.register_bases(self.g)
            self._g_lagrange = self.lib.register_bases(self.g_lagrange)

    @classmethod
    def read_custom(cls, path: str, fmt: int, lib=None) -> "ParamsKZG":
        """ParamsKZG::read_custom: the file is decoded on the device and both vectors stay resident there as registered
        base sets (no second upload); the host copies are what `get_g()` and the verifier read"""
        lib = lib or _lib.load()
        if lib.device_count() == 0:
            lib.init(0)
        r = lib.srs_read(path, fmt)
        return cls(r["k"], r["g"], r["g_lagrange"], lib, r["g2_bytes"], (r["handle_g"], r["handle_g_lagrange"]))

    @classmethod
    def setup(cls, k: int, s, lib=None, g2_bytes: bytes = b"") -> "ParamsKZG":
        """ParamsKZG::setup with the caller's toxic waste s (4 words, Montgomery): both vectors are computed on the device and
        stay resident there as registered base sets.  g2_bytes (g2 | s_g2 as write_custom stores them) come from the caller:
        G2 arithmetic is the host's business."""
        lib = lib or _lib.load()
        if lib.device_count() == 0:
            lib.init(0)
        r = lib.srs_setup(k, s)
        return cls(k, r["g"], r["g_lagrange"], lib, g2_bytes, (r["handle_g"], r["handle_g_lagrange"]))

    @classmethod
    def read(cls, path: str, lib=None) -> "ParamsKZG":
        """ParamsKZG::read = read_custom(reader, SerdeFormat::RawBytes)"""
        return cls.read_custom(path, SerdeFormat.RawBytes, lib)

    def downsize(self, k: int):
        """ParamsKZG::downsize: keep the first 2^k points of g and recompute g_lagrange from them on the device
        (g_to_lagrange); both become new resident sets and the old ones are given back.  g2_bytes are kept."""
        assert k <= self.k, "downsize: k = %d above the params' k = %d" % (k, self.k)
        r = self.lib.srs_downsize(self._g, k)
        old = (self._g, self._g_lagrange)
        self.k, self.n = k, 1 << k
        self.g = self.g[:self.n].copy()
        self.g_lagrange = r["g_lagrange"]
        self._g, self._g_lagrange = r["handle_g"], r["handle_g_lagrange"]
        for h in old:
            if h:
                self.lib.unregister_bases(h)

    def write_custom(self, path: str, fmt: int):
        self.lib.srs_write(path, fmt, self.k, self.g, self.g_lagrange, self.g2_bytes)

    def write(self, path: str):
        self.write_custom(path, SerdeFormat.RawBytes)

    def commit(self, poly: np.ndarray) -> np.ndarray:
        """best_multiexp(poly, g[..poly.len()]) -> G1 Jacobian"""
        poly = np.ascontiguousarray(poly, dtype=np.uint64).reshape(-1, 4)
        assert poly.shape[0] <= self.n
        return self.lib.msm_registered(poly, self._g, 0)

    def commit_lagrange(self, poly: np.ndarray) -> np.ndarray:
        """best_multiexp(poly, g_lagrange[..poly.len()]) -> G1 Jacobian"""
        poly = np.ascontiguousarray(poly, dtype=np.uint64).reshape(-1, 4)
        assert poly.shape[0] <= self.n
        return self.lib.msm_registered(poly, self._g_lagrange, 0)

    def commit_many(self, polys) -> np.ndarray:
        """the independent commitments of one prover phase over `g`: one batched kernel sequence per device -> (len(polys), 12)"""
        return self.lib.msm_batch_registered(polys, self._g)

    def commit_lagrange_many(self, polys) -> np.ndarray:
        return self.lib.msm_batch_registered(polys, self._g_lagrange)

    def commit_lagrange_and_convert(self, domain, lagrange: np.ndarray, want_extended: bool = True, keep_on_device: bool = False):
        """commit_lagrange + EvaluationDomain::lagrange_to_coeff + coeff_to_extended of one column with a single upload
        (h2b_column_pipeline) -> dict(commitment, coeff, extended, d_extended)"""
        from .domain import fr_to_words
        zs = np.stack([fr_to_words(1), fr_to_words(domain.g_coset), fr_to_words(domain.g_coset_inv)])
        return self.lib.column_pipeline(lagrange, self._g_lagrange, self.k, domain.extended_k, fr_to_words(domain.omega_inv), fr_to_words(domain.ifft_divisor),
                                        fr_to_words(domain.extended_omega), zs, want_extended=want_extended, keep_on_device=keep_on_device)

    def close(self):
        for h in (self._g, self._g_lagrange):
            if h:
                self.lib.unregister_bases(h)
        self._g = self._g_lagrange = 0
