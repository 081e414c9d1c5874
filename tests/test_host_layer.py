"""The C ABI's host layer: a device allocation the runtime refuses leaves no error pending on the calling thread, so the next
call on that thread that launches a kernel succeeds.  The runtime keeps a failed cudaMalloc as the thread's last error; the
library checks its launches with cudaGetLastError, so an allocation site that did not clear it would fail the next launch.

CPU: the kernel sources through the emulator, which keeps that per-thread last error too.  GPU: a B200."""
import pytest

import parity_cases as pc
from harness import orc_srs_setup
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
        g, gl = orc_srs_setup(k, s)
        assert (params.g == g).all() and (params.g_lagrange == gl).all()
    finally:
        params.close()


def test_launches_after_a_refused_allocation_emu(emu, oc):
    check_launches_after_a_refused_allocation(emu, oc, 5)


@pytest.mark.gpu
def test_launches_after_a_refused_allocation(gpu, oc):
    check_launches_after_a_refused_allocation(gpu, oc, 12)


def test_concurrent_scale_on_one_device_emu(emu, oc):
    """h2b_fr_scale_dev with more than 8 factors stages them in a table its device context holds for every call.  Host threads that
    scale on one device at once each get their own factors: the device lock keeps one call's table from being overwritten by another's
    while its kernel reads it.  Emulator only: without the lock a GPU kernel could read a table another call has freed."""
    import threading

    import numpy as np

    L, n, count, n_threads, calls = emu, 1 << 12, 16, 4, 50
    warm = L.dev_alloc(0, 32 * count)
    try:
        L.fr_scale_dev(0, warm, count, oc.random_fr(30, count))      # the table reaches its size here and does not grow below
    finally:
        L.dev_free(0, warm)
    failures = []

    def scale_repeatedly(t):
        a, f = oc.random_fr(31 + t, n), oc.random_fr(41 + t, count)
        want = a.copy()
        for r in range(count):
            want[r::count] = oc.fr_scale(np.ascontiguousarray(a[r::count]), f[r])
        d = L.dev_alloc(0, 32 * n)
        try:
            got = np.empty_like(a)
            for call in range(calls):
                L.h2d(0, d, a)
                L.fr_scale_dev(0, d, n, f)
                L.d2h(0, got, d)
                if not (got == want).all():
                    failures.append((t, call))
        except Exception as e:      # reported by the main thread
            failures.append((t, repr(e)))
        finally:
            L.dev_free(0, d)

    threads = [threading.Thread(target=scale_repeatedly, args=(t,)) for t in range(n_threads)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert failures == []
