"""
The multi-point openings of KZG on the device: SHPLONK ([UP] halo2_proofs/src/poly/kzg/multiopen/shplonk/prover.rs,
ProverSHPLONK::create_proof) through h2b_shplonk_*, GWC (.../multiopen/gwc/prover.rs, ProverGWC::create_proof) through
h2b_gwc_create_proof, and the query evaluation of plonk/prover.rs through h2b_fr_eval_queries_dev.

A query is (poly, point): poly is a host array of n Fr (n x 4 uint64, Montgomery) or a device pointer (int) on the session's device,
point 4 Montgomery words.  Polynomials are identified the way upstream identifies them, by object (pointer) identity: two distinct
arrays with equal contents are two polynomials, the same array queried twice is one.
"""
from __future__ import annotations

import numpy as np


def _index_queries(queries):
    """[(poly, point)] -> (distinct polys in first-appearance order, [(index, point words)])"""
    polys, index, out = [], {}, []
    for poly, point in queries:
        key = poly if isinstance(poly, int) else id(poly)
        if key not in index:
            index[key] = len(polys)
            polys.append(poly)
        out.append((index[key], np.ascontiguousarray(point, dtype=np.uint64).reshape(4)))
    return polys, out


def eval_queries(lib, device: int, d_polys, n: int, queries, d_out: int, stream: int = 0):
    """eval_polynomial(d_polys[poly], point) of every (poly index, point) query -> d_out (one Fr per query, in query order)"""
    lib.eval_queries_dev(device, d_polys, n, queries, d_out, stream)


def _polys_and_n(polys, params):
    on_host = not isinstance(polys[0], int)
    if any(isinstance(p, int) == on_host for p in polys):
        raise ValueError("create_proof: polynomials are either all host arrays or all device pointers")
    if not on_host:
        return polys, on_host, params.n
    polys = [np.ascontiguousarray(p, dtype=np.uint64).reshape(-1, 4) for p in polys]
    n = polys[0].shape[0]
    if any(p.shape[0] != n for p in polys):
        raise ValueError("create_proof: polynomials of different lengths")
    return polys, on_host, n


class ProverSHPLONK:
    """ProverSHPLONK::new(params): create_proof over the params' registered g on one device"""

    def __init__(self, params, device: int = 0):
        self.params = params
        self.lib = params.lib
        self.device = device

    def create_proof(self, queries, y, v, squeeze_u):
        """queries [(poly, point)] in the prover's order; y and v the challenges the caller squeezed (upstream squeezes y, then v);
        squeeze_u(h1) is called after h1 (Jacobian) is written and returns u.  Returns (h1, h2), Jacobian."""
        polys, indexed = _index_queries(queries)
        polys, on_host, n = _polys_and_n(polys, self.params)
        h1, session = self.lib.shplonk_begin(self.device, polys, on_host, n, indexed, self.params._g, y, v)
        try:
            u = squeeze_u(h1)
            h2 = self.lib.shplonk_finish(session, u)
        finally:
            self.lib.shplonk_release(session)
        return h1, h2


class ProverGWC:
    """ProverGWC::new(params): create_proof over the params' registered g on one device"""

    def __init__(self, params, device: int = 0):
        self.params = params
        self.lib = params.lib
        self.device = device

    def create_proof(self, queries, v):
        """queries [(poly, point)] in the prover's order; v the challenge the caller squeezed.  Returns [W, ...] (Jacobian), one per
        distinct point in first-appearance order, which upstream writes to the transcript in that order."""
        polys, indexed = _index_queries(queries)
        polys, on_host, n = _polys_and_n(polys, self.params)
        return list(self.lib.gwc_create_proof(self.device, polys, on_host, n, indexed, self.params._g, v))


__all__ = ["ProverGWC", "ProverSHPLONK", "eval_queries"]
