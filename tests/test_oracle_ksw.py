"""Mate-rescue local alignment (SURVEY 8f item 1, groundwork for the next widening step): the oracle's scalar restatement of the
reference's striped SSE2 kernels (ksw_align2 = ksw_u8 / ksw_i16 forward + reversed-prefix pass, src/ksw.cpp:111-381) against
golden vectors made by the UNMODIFIED reference (tests/golden/make_ksw_golden.py) and against the reference's results on seeded request
sets of other query lengths (recorded by tests/golden/make_live_golden.py)."""
import numpy as np
import pytest
import ksw_util as ku
import refgolden


def _golden(golden_dir):
    g = np.load(golden_dir + "/ksw_c0.npz")
    reqs = [(g["query"][g["qoff"][i]:g["qoff"][i + 1]], g["target"][g["toff"][i]:g["toff"][i + 1]], int(g["xtra"][i])) for i in range(len(g["xtra"]))]
    return reqs, g["out"]


def test_oracle_matches_reference_golden(pkg, golden_dir):
    reqs, want = _golden(golden_dir)
    got = ku.oracle_ksw(reqs, pkg.capi.default_opt())
    assert np.array_equal(got, want)
    assert (want[:, 5] >= 0).sum() > 800 and (want[:, 3] > 0).sum() > 200      # start positions and second-best scores are covered
    assert sum(1 for r in reqs if r[2] & ku.KSW_XBYTE) > 500 and sum(1 for r in reqs if not r[2] & ku.KSW_XBYTE) > 200      # both kernels


KSW_CASES = [(11, (151,)), (12, (36, 50, 76, 100)), (13, (249, 250, 251, 400)), (14, (15, 16, 17, 8, 9))]


@pytest.mark.parametrize("seed,qlens", KSW_CASES)
def test_oracle_matches_the_live_reference(pkg, seed, qlens):
    reqs = ku.make_requests(np.random.default_rng(seed), 1200, qlens=qlens)
    want = refgolden.get(f"ksw/{seed}")
    got = ku.oracle_ksw(reqs, pkg.capi.default_opt())
    bad = np.nonzero((got != want).any(1))[0]
    assert len(bad) == 0, (bad[:5], got[bad[:5]], want[bad[:5]])


# ---- the device logic (ksw_device.cuh: one sweep per row with a segment-local and a complete F) against the oracle -------------------
import ctypes as C, os, subprocess
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_EMUL = None


def _emul():
    global _EMUL
    if _EMUL is None:
        d = os.path.join(ROOT, "tests", "host_emul")
        so = os.path.join(d, "libkswemul.so")
        srcs = [os.path.join(d, f) for f in ("ksw_emul.cpp", "ksw_warp_emul.cpp")] + [os.path.join(ROOT, "bwa-mem2_b200", "csrc", f) for f in ("ksw_device.cuh", "ksw_warp.cuh", "hd.h")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(s) for s in srcs):
            subprocess.check_call(["g++", "-O2", "-g", "-std=c++17", "-fPIC", "-shared", "-w", "-I" + os.path.join(ROOT, "bwa-mem2_b200", "csrc"),
                                   "-I" + os.path.join(ROOT, "include"), srcs[0], srcs[1], "-o", so])
        _EMUL = C.CDLL(so)
    return _EMUL


def emul_ksw(reqs, opt, warp=False):
    """ksw_device.cuh's one-thread sweep, or (warp=True) ksw_warp.cuh's 32-lane formulation; queries beyond the latter's 497 bases fall back to the sweep."""
    L = _emul()
    out = np.zeros((len(reqs), 7), np.int32)
    mat = (C.c_int8 * 25)(*[opt.mat[i] for i in range(25)])
    for i, (q, t, x) in enumerate(reqs):
        q = np.ascontiguousarray(q); t = np.ascontiguousarray(t)
        f = L.emul_ksw_warp_align2 if warp and len(q) <= 497 else L.emul_ksw_align2
        ov = f(C.c_int32(len(q)), q.ctypes.data_as(C.c_void_p), C.c_int32(len(t)), t.ctypes.data_as(C.c_void_p), mat,
                               C.c_int32(opt.o_del), C.c_int32(opt.e_del), C.c_int32(opt.o_ins), C.c_int32(opt.e_ins), C.c_int32(x),
                               out[i].ctypes.data_as(C.c_void_p))
        assert ov == 0
    return out


@pytest.mark.parametrize("warp", [False, True], ids=["thread_sweep", "warp_scan"])
def test_device_logic_matches_reference_golden(pkg, golden_dir, warp):
    reqs, want = _golden(golden_dir)
    assert np.array_equal(emul_ksw(reqs, pkg.capi.default_opt(), warp=warp), want)


@pytest.mark.parametrize("seed,qlens,sc", [(21, (151, 100, 36), {}), (22, (249, 250, 300, 17), {}),
                                           (23, (151, 76), dict(o_del=1, e_del=1, o_ins=1, e_ins=1, b=1)),     # gap open == 0 after update: F ties
                                           (24, (120, 260), dict(o_del=4, e_del=2, o_ins=5, e_ins=1, a=2, b=3)),
                                           (25, (497, 481, 33, 32, 31), {})])                                  # the warp formulation's longest query, lanes without columns
@pytest.mark.parametrize("warp", [False, True], ids=["thread_sweep", "warp_scan"])
def test_device_logic_matches_oracle(pkg, seed, qlens, sc, warp):
    o = pkg.capi.default_opt()
    for k, v in sc.items():
        setattr(o, k, v)
    k = 0
    for i in range(4):
        for j in range(4):
            o.mat[k] = o.a if i == j else -o.b; k += 1
        o.mat[k] = -1; k += 1
    reqs = ku.make_requests(np.random.default_rng(seed), 1000, qlens=qlens)
    reqs = [(q, t, ku.mate_xtra(len(q), a=o.a, min_seed_len=o.min_seed_len)) for q, t, _ in reqs]
    want = ku.oracle_ksw(reqs, o)
    got = emul_ksw(reqs, o, warp=warp)
    bad = np.nonzero((got != want).any(1))[0]
    assert len(bad) == 0, (bad[:5], got[bad[:5]], want[bad[:5]])
