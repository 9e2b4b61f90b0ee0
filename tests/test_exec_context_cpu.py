"""CPU tests (no GPU) of the library's per-thread state: b200pci_last_error() is thread-local
(include/b200pci.h), so concurrent callers each read the message of their own last failing call.
The calls here fail on their arguments before any CUDA call, so no device is needed."""
import threading

import pytest


@pytest.fixture(scope="module")
def lib():
    from mocopci_b200 import build
    build.build()
    from mocopci_b200 import _lib
    return _lib


ROUNDS = 200


def _bad_knn(L, k):
    """b200pci_knn with k outside [1, 64]: EINVAL from the argument check, no CUDA call."""
    return L.b200pci_knn(1, 4, 8, k, 0, None, 0, 0, 0, None, 0, 0, 0, None, 1, None, None, 0, None)


def test_last_error_is_per_thread(lib):
    """Two threads fail in lockstep (a barrier before every call and before every read): thread A
    with k = 0, thread B with k = 65. With a process-global message, whichever thread wrote last
    would overwrite the other's; each thread must always read its own k back."""
    L = lib.lib
    barrier = threading.Barrier(2)
    seen = {0: [], 65: []}
    errors = []

    def worker(k):
        try:
            for _ in range(ROUNDS):
                barrier.wait()
                rc = _bad_knn(L, k)
                barrier.wait()  # both threads have written their message before either reads
                seen[k].append((rc, L.b200pci_last_error().decode()))
        except Exception as e:  # noqa: BLE001  (reported below; a dead thread would hang the barrier)
            barrier.abort()
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(k,)) for k in (0, 65)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for k in (0, 65):
        assert len(seen[k]) == ROUNDS
        want = f"knn: k={k} outside [1,64]"
        bad = [(rc, msg) for rc, msg in seen[k] if rc != -1 or msg != want]
        assert not bad, f"thread with k={k}: {len(bad)} of {ROUNDS} rounds read {bad[:3]}"


def test_last_error_of_a_new_thread_is_empty(lib):
    """A thread that has made no failing call reads "" even after another thread failed."""
    L = lib.lib
    assert _bad_knn(L, 0) == -1
    assert L.b200pci_last_error() == b"knn: k=0 outside [1,64]"
    got = []
    t = threading.Thread(target=lambda: got.append(L.b200pci_last_error()))
    t.start()
    t.join()
    assert got == [b""]
    assert L.b200pci_last_error() == b"knn: k=0 outside [1,64]"  # the caller's own is untouched

