"""ssd_advantages / ssd_vtrace / ssd_advantages_workspace_bytes check every argument before they touch a device: these tests need
no GPU."""
import ctypes as C

import pytest

INF, NAN = float("inf"), float("nan")
P = C.c_void_p(256)             # a 16-byte aligned stand-in for a device pointer; nothing is launched


def _lib():
    from sequential_social_dilemma_games_b200 import _lib
    return _lib


def _gae(**kw):
    """Valid arguments of ssd_advantages (T = 8, M = 10, N = 5, GAE, int32 rewards), overridden by kw."""
    a = dict(mode=0, T=8, M=10, N=5, rewards=P, dtype=0, intrinsic=None, w=0.5, values=P, dones=P, bootstrap=P, gamma=0.99,
             lam=0.95, adv=P, vt=P, ws=None, ws_bytes=0, stream=None)
    a.update(kw)
    return list(a.values())


def _vtrace(**kw):
    a = dict(T=8, M=10, N=5, rewards=P, dtype=1, intrinsic=None, w=0.0, values=P, dones=P, bootstrap=P, tl=P, bl=P, gamma=0.99,
             rho=1.0, pg=1.0, vs=P, pga=P, ws=None, ws_bytes=0, stream=None)
    a.update(kw)
    return list(a.values())


def _id(kw):
    return ",".join("%s=%r" % (k, getattr(v, "value", v)) for k, v in kw.items())


GAE_ERRORS = [
    ({"mode": 2}, b"mode"), ({"mode": -1}, b"mode"),
    ({"rewards": None}, b"null"), ({"values": None}, b"null"), ({"dones": None}, b"null"), ({"bootstrap": None}, b"null"),
    ({"adv": None}, b"null"), ({"vt": None}, b"null"),
    ({"T": 0}, b"positive"), ({"T": -3}, b"positive"), ({"M": 0}, b"positive"), ({"M": -10}, b"positive"),
    ({"N": 0}, b"multiple"), ({"N": 3}, b"multiple"), ({"N": -5}, b"multiple"),
    ({"dtype": 2}, b"dtype"), ({"dtype": -1}, b"dtype"),
    ({"gamma": -0.1}, b"gamma"), ({"gamma": 1.01}, b"gamma"), ({"gamma": NAN}, b"gamma"), ({"gamma": INF}, b"gamma"),
    ({"lam": -0.5}, b"lambda"), ({"lam": 1.5}, b"lambda"), ({"lam": NAN}, b"lambda"),
    ({"values": C.c_void_p(258)}, b"aligned"), ({"intrinsic": C.c_void_p(257)}, b"aligned"), ({"adv": C.c_void_p(2)}, b"aligned"),
    ({"mode": 1}, b"NULL"),                                  # returns mode with a value_targets pointer
    ({"T": 1000, "M": 320}, b"workspace"),                    # the chunked path needs a workspace
]


@pytest.mark.parametrize("kw,msg", GAE_ERRORS, ids=[_id(kw) for kw, _ in GAE_ERRORS])
def test_advantages_argument_errors(kw, msg):
    L = _lib()
    assert L.lib.ssd_advantages(*_gae(**kw)) == -1
    assert msg in L.lib.ssd_last_error(), L.lib.ssd_last_error()


VTRACE_ERRORS = [
    ({"tl": None}, b"null"), ({"bl": None}, b"null"), ({"vs": None}, b"null"), ({"pga": None}, b"null"),
    ({"rewards": None}, b"null"), ({"bootstrap": None}, b"null"),
    ({"T": 0}, b"positive"), ({"M": -1}, b"positive"), ({"N": 4}, b"multiple"), ({"dtype": 7}, b"dtype"),
    ({"gamma": 2.0}, b"gamma"), ({"rho": -1.0}, b"clip"), ({"pg": -1e-3}, b"clip"), ({"rho": NAN}, b"clip"), ({"pg": NAN}, b"clip"),
    ({"tl": C.c_void_p(6)}, b"aligned"), ({"pga": C.c_void_p(6)}, b"aligned"),
    ({"T": 1000, "M": 320}, b"workspace"),
]


@pytest.mark.parametrize("kw,msg", VTRACE_ERRORS, ids=[_id(kw) for kw, _ in VTRACE_ERRORS])
def test_vtrace_argument_errors(kw, msg):
    L = _lib()
    assert L.lib.ssd_vtrace(*_vtrace(**kw)) == -1
    assert msg in L.lib.ssd_last_error(), L.lib.ssd_last_error()


def test_workspace_size_and_checks():
    L = _lib().lib
    assert L.ssd_advantages_workspace_bytes(0, 10) == 0 and L.ssd_advantages_workspace_bytes(10, -1) == 0
    assert L.ssd_advantages_workspace_bytes(1000, 327680) == 0          # one pass over time: no workspace
    assert L.ssd_advantages_workspace_bytes(15, 320) == 0               # too short to split
    need = L.ssd_advantages_workspace_bytes(1000, 320)
    assert need > 0 and need % 16 == 0
    for ws, nbytes in ((None, need), (P, need - 1), (C.c_void_p(264), need)):   # missing, too small, misaligned
        assert L.ssd_advantages(*_gae(T=1000, M=320, ws=ws, ws_bytes=nbytes)) == -1
        assert b"workspace" in L.ssd_last_error()
        assert L.ssd_vtrace(*_vtrace(T=1000, M=320, ws=ws, ws_bytes=nbytes)) == -1
        assert b"workspace" in L.ssd_last_error()
