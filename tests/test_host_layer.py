"""The C ABI's host layer: a device allocation the runtime refuses leaves no error pending on the calling thread, so the next
call on that thread that launches a kernel succeeds.  The runtime keeps a failed cudaMalloc as the thread's last error; the
library checks its launches with cudaGetLastError, so an allocation site that did not clear it would fail the next launch.

CPU: the kernel sources through the emulator, which keeps that per-thread last error too.  GPU: a B200."""
import pytest

import parity_cases as pc
import test_srs_setup as srs
from halo2_scaffold_b200._lib import H2BError

H2B_ERR_OOM = -4
TOO_LARGE = 1 << 50      # more than any device holds: refused by the runtime before any memory is touched


def refuse_allocation(L):
    with pytest.raises(H2BError) as e:
        L.dev_alloc(0, TOO_LARGE)
    assert e.value.code == H2B_ERR_OOM


def check_launches_after_a_refused_allocation(L, oc, k):
    n = 1 << k
    refuse_allocation(L)
    assert (L.gen_scalars(11, n) == oc.random_fr(11, n)).all()
    refuse_allocation(L)
    a = oc.random_fr(12, n)
    w = pc.omega_words(oc, k)
    assert (L.ntt(a.copy(), w, k) == oc.best_fft(a, w, k)).all()
    refuse_allocation(L)
    import halo2_scaffold_b200 as h2
    s = oc.random_fr(13, 1)[0]
    params = h2.ParamsKZG.setup(k, s, lib=L)
    try:
        g, gl = srs.orc_srs_setup(k, s)
        assert (params.g == g).all() and (params.g_lagrange == gl).all()
    finally:
        params.close()


def test_launches_after_a_refused_allocation_emu(emu, oc):
    check_launches_after_a_refused_allocation(emu, oc, 5)


@pytest.mark.gpu
def test_launches_after_a_refused_allocation(gpu, oc):
    check_launches_after_a_refused_allocation(gpu, oc, 12)
