"""CPU: K-EPISODE's argument checks (b200_episode_scan) return their error codes before any CUDA call, and
b200_episode_scratch_bytes sizes the per-block partials of its statistics."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    import os
    import __graft_entry__ as g
    from reinforcementlearningplatform_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        g.build()
    return _lib.load()


ESIZE, EDTYPE, ENULL, EPARAMS = -6, -2, -4, -3
P = C.c_void_p(0x1000)        # never dereferenced: every call below fails its checks first


def scan(lib, r_dtype=1, T=4, N=300, r=P, done=P, flag=P, acc_r=P, acc_l=P, ep_r=None, ep_l=None, ep_f=None,
         first_only=0, stats=None, scratch=None, scratch_bytes=0):
    return lib.b200_episode_scan(r_dtype, T, N, r, done, flag, acc_r, acc_l, ep_r, ep_l, ep_f, first_only, stats,
                                 scratch, scratch_bytes, None)


def test_stats_layout_constant_matches_header():
    import os
    import re
    from conftest import ROOT
    from reinforcementlearningplatform_b200 import episodes
    src = open(os.path.join(ROOT, "include", "b200env.h")).read()
    assert int(re.search(r"#define B200_EPISODE_STATS (\d+)", src).group(1)) == episodes.STATS == 6 + episodes.FLAG_BINS


def test_scratch_bytes(lib):
    assert lib.b200_episode_scratch_bytes(0) == 0
    assert lib.b200_episode_scratch_bytes(-5) == 0
    for n, blocks in ((1, 1), (127, 1), (128, 1), (129, 2), (100003, 782), (1 << 20, 8192)):
        assert lib.b200_episode_scratch_bytes(n) == blocks * 22 * 8, n


def test_error_codes_without_device(lib):
    big = C.c_void_p(0x10000)
    # sizes
    for T, N in ((0, 5), (-1, 5), (5, 0), (5, -3), (5, 1 << 31), (5, 1 << 40)):
        assert scan(lib, T=T, N=N) == ESIZE, (T, N)
    # dtype
    for dt in (-1, 2, 7):
        assert scan(lib, r_dtype=dt) == EDTYPE
    # required pointers
    for k in ("r", "done", "flag", "acc_r", "acc_l"):
        assert scan(lib, **{k: None}) == ENULL, k
    assert scan(lib, first_only=1) == ENULL                      # first_only needs ep_flag
    assert scan(lib, stats=P) == ENULL                           # stats needs scratch
    # scratch too small or misaligned
    assert scan(lib, stats=P, scratch=big, scratch_bytes=lib.b200_episode_scratch_bytes(300) - 8) == EPARAMS
    assert scan(lib, stats=P, scratch=C.c_void_p(0x10004), scratch_bytes=1 << 20) == EPARAMS
    # precedence: size before dtype before null before params
    assert scan(lib, T=0, r_dtype=9, r=None) == ESIZE
    assert scan(lib, r_dtype=9, r=None, stats=P, scratch=big, scratch_bytes=0) == EDTYPE
    assert scan(lib, r=None, stats=P, scratch=big, scratch_bytes=0) == ENULL


def test_tracker_refuses_cpu_device():
    from reinforcementlearningplatform_b200 import EpisodeTracker, _lib
    with pytest.raises(_lib.B200EnvError):
        EpisodeTracker(4, "cpu")
