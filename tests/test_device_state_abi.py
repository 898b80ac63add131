"""CPU-side checks of the device-resident per-step state of crypto (io.window_head_dev) and snake (the self-managed
done-counter block, done_count_next == done_count): argument checks happen before anything launches, and the ctypes
binding of beng_crypto_io follows include/beng.h."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAD_ARG = -1
ADDR = 1 << 20  # a 16-byte aligned stand-in address: the checks below never dereference it


def header_fields(struct):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "beng.h")).read(), flags=re.S)
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
    return re.findall(r"(\w+);", body)


def test_crypto_io_binding_matches_header():
    from custom_gymnasium_environments_b200 import _lib

    assert [f[0] for f in _lib.CryptoIO._fields_] == header_fields("beng_crypto_io")
    assert C.sizeof(_lib.CryptoIO) == 12 * 8
    assert _lib.CryptoIO._fields_[-1][0] == "window_head_dev"


def crypto_call_args(L, window_head, window_head_dev):
    p = L.CryptoParams(10000.0, 0.001, 0.0005, 100.0, 100000.0, 0.02, 0.1, 1000, 2, 0, window_head, 0, 0, 0, 0)
    st = L.CryptoState(ADDR, ADDR, ADDR, ADDR, ADDR)
    io = L.CryptoIO(ADDR, ADDR, ADDR, ADDR)
    io.window_head_dev = window_head_dev
    return p, st, io


def test_misaligned_window_head_dev_is_rejected_before_launch():
    from custom_gymnasium_environments_b200 import _lib as L

    lib = L.load()
    before = lib.beng_launch_count()
    p, st, io = crypto_call_args(L, 0, ADDR + 4)  # 4-byte but not 8-byte aligned
    assert lib.beng_crypto_step(C.byref(p), C.byref(st), ADDR, C.byref(io), 64, None) == BAD_ARG
    assert lib.beng_crypto_reset(C.byref(p), C.byref(st), C.byref(io), None, 64, 1, None) == BAD_ARG
    assert lib.beng_crypto_step_host(C.byref(p), C.byref(st), ADDR, C.byref(io), 64, ADDR, None, None, None, None,
                                     None) == BAD_ARG
    assert lib.beng_launch_count() == before


def test_window_head_is_not_validated_when_the_head_lives_on_the_device():
    from custom_gymnasium_environments_b200 import _lib as L

    lib = L.load()
    before = lib.beng_launch_count()
    for head in (-1, 50, 77):
        p, st, io = crypto_call_args(L, head, ADDR)
        # n_envs = 0: every argument check runs, nothing launches
        assert lib.beng_crypto_step(C.byref(p), C.byref(st), ADDR, C.byref(io), 0, None) == 0
        assert lib.beng_crypto_reset(C.byref(p), C.byref(st), C.byref(io), None, 0, 1, None) == 0
        p, st, io = crypto_call_args(L, head, None)  # the host head keeps its range check
        assert lib.beng_crypto_step(C.byref(p), C.byref(st), ADDR, C.byref(io), 0, None) == BAD_ARG
    assert lib.beng_launch_count() == before


def snake_call_args(L, done_count, done_count_next):
    p = L.SnakeParams(20, 1000, 2, 0, 0, 0)
    st = L.SnakeState(ADDR, ADDR)
    io = L.SnakeIO(ADDR, ADDR, ADDR)
    io.done_env, io.done_count, io.done_count_next = ADDR, done_count, done_count_next
    return p, st, io


def test_misaligned_self_managed_done_counters_are_rejected_before_launch():
    from custom_gymnasium_environments_b200 import _lib as L

    lib = L.load()
    before = lib.beng_launch_count()
    p, st, io = snake_call_args(L, ADDR + 8, ADDR + 8)  # the 16-byte block, only 8-byte aligned
    for fn in (lib.beng_snake_step, lib.beng_snake_step_inplace):
        assert fn(C.byref(p), C.byref(st), ADDR, C.byref(io), 64, None) == BAD_ARG
    assert lib.beng_snake_reset(C.byref(p), C.byref(st), C.byref(io), None, 64, 1, None) == BAD_ARG
    assert lib.beng_launch_count() == before

    # aligned, and the caller-managed pair at 4-byte alignment, pass the checks (n_envs = 0 launches nothing)
    for count, nxt in ((ADDR + 16, ADDR + 16), (ADDR + 4, ADDR + 8), (ADDR + 4, None)):
        p, st, io = snake_call_args(L, count, nxt)
        assert lib.beng_snake_step(C.byref(p), C.byref(st), ADDR, C.byref(io), 0, None) == 0
    assert lib.beng_launch_count() == before
