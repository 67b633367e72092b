"""Host-side checks of the cluster head at any feature_dim (1 <= C <= 4096): argument validation of the relaxed entry
points happens before any CUDA call, C above 4096 is refused, and the workspace queries grow with C."""
import videoad_b200 as V  # noqa: F401  (loads the library)
from videoad_b200 import _lib

ERR_BAD_SHAPE, ERR_NULL, ERR_UNSUPPORTED = -1, -2, -6
RAGGED = [1, 3, 6, 30, 190, 770, 1026, 1535, 1539, 2047, 2049, 3001, 4095]


def _fwd(l, C, K):
    return l.vadc_cluster_fwd(None, None, None, None, 8, C, K, 16.0, 1e-5, None, None, None, None,
                              None, None, None, None, None, None, 0, 0, None)


def _bwd(l, C, K):
    return l.vadc_cluster_bwd(None, None, None, None, None, None, None, None, None, None, None, None, None, None, None,
                              8, C, K, 16.0, None, None, None, None, None, 0, None)


def _padded(l, C, K, Kv):
    return l.vadc_cluster_fwd_padded(None, None, None, None, 8, C, K, Kv, 16.0, 1e-5, None, None, None, None,
                                     None, None, None, None, None, None, 0, None)


def test_any_c_up_to_4096_passes_the_shape_checks():
    l = _lib.lib()
    for C in RAGGED + [4096]:
        assert _fwd(l, C, 32) == ERR_NULL, C               # past the shape checks: the NULL pointers are what is refused
        assert _bwd(l, C, 32) == ERR_NULL, C
        assert _padded(l, C, 8, 5) == ERR_NULL, C


def test_c_above_4096_and_k_not_multiple_of_4_are_refused_on_the_host():
    l = _lib.lib()
    for C in (4097, 8192):
        assert _fwd(l, C, 32) == ERR_UNSUPPORTED
        assert _bwd(l, C, 32) == ERR_UNSUPPORTED
        assert _padded(l, C, 8, 5) == ERR_UNSUPPORTED
    assert _fwd(l, 190, 30) == ERR_BAD_SHAPE
    assert _bwd(l, 190, 30) == ERR_BAD_SHAPE
    assert _fwd(l, 0, 32) == ERR_BAD_SHAPE


def test_workspace_queries_are_positive_and_monotone_in_c():
    l = _lib.lib()
    for N, K in ((1, 32), (1000, 32), (300, 8), (65536, 1024), (65536 - 37, 64)):
        for impl in (0, 1):
            f = [l.vadc_cluster_fwd_workspace_bytes(N, C, K, impl) for C in RAGGED]
            assert all(v > 0 for v in f) and all(a <= b for a, b in zip(f, f[1:])), (N, K, impl, f)
        b = [l.vadc_cluster_bwd_workspace_bytes(N, C, K) for C in RAGGED]
        assert all(v > 0 for v in b) and all(a <= c for a, c in zip(b, b[1:])), (N, K, b)
        # every ragged width up to 1100 in steps of one
        b = [l.vadc_cluster_bwd_workspace_bytes(N, C, K) for C in range(1, 1100, 2)]
        assert all(a <= c for a, c in zip(b, b[1:])), (N, K)
