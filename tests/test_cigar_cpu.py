"""Seam 3 (CIGAR / NM / MD == bwa_gen_cigar2, SURVEY 8f item 2) on the CPU: the oracle's restatement against the golden vectors
made by the UNMODIFIED reference (tests/golden/make_cigar_golden.py) and against the reference's results on a second, seeded random
request set (recorded by tests/golden/make_live_golden.py); the device logic (cigar_device.cuh compiled for the host) against the oracle."""
import ctypes as C, hashlib, os, subprocess
import numpy as np
import pytest
import oracle_lib as ol
import cigar_util as cu
import refgolden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_EMUL = None


def _emul():
    global _EMUL
    if _EMUL is None:
        d = os.path.join(ROOT, "tests", "host_emul")
        so = os.path.join(d, "libcigaremul.so")
        srcs = [os.path.join(d, "cigar_emul.cpp")] + [os.path.join(ROOT, "bwa-mem2_b200", "csrc", f) for f in ("cigar_device.cuh", "chain_device.cuh", "hd.h")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(s) for s in srcs):
            subprocess.check_call(["g++", "-O2", "-g", "-std=c++17", "-fPIC", "-shared", "-w", "-ffp-contract=off", "-I" + os.path.join(ROOT, "bwa-mem2_b200", "csrc"),
                                   "-I" + os.path.join(ROOT, "include"), srcs[0], "-o", so])
        _EMUL = C.CDLL(so)
    return _EMUL


def emul_gen_cigar(capi, index, opt, codes, offsets, reqs):
    codes = np.ascontiguousarray(codes, np.uint8); offsets = np.ascontiguousarray(offsets, np.int64)
    reqs = np.ascontiguousarray(reqs, capi.CIGAR_REQ_DT)
    rb = capi.ReadBatch(len(offsets) - 1, codes.ctypes.data, offsets.ctypes.data)
    recs = C.c_void_p(); cig = C.c_void_p(); md = C.c_void_p(); n_ops = C.c_int64(); n_md = C.c_int64()
    rc = _emul().emul_gen_cigar(C.byref(index.desc), C.byref(opt), C.byref(rb), reqs.ctypes.data_as(C.c_void_p), C.c_int64(len(reqs)),
                                C.byref(recs), C.byref(cig), C.byref(n_ops), C.byref(md), C.byref(n_md))
    assert rc == 0, rc
    def arr(p, n, dt):
        dt = np.dtype(dt)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(n, 1) * dt.itemsize,))[:n * dt.itemsize].view(dt).copy()
    out = arr(recs, len(reqs), capi.CIGAR_REC_DT), arr(cig, n_ops.value, "<u4"), arr(md, n_md.value, "u1")
    for p in (recs, cig, md):
        ol.lib().bm2o_free(p)
    return out


@pytest.fixture(scope="module")
def c0(pkg, golden_dir):
    idx = pkg.capi.Index(golden_dir + "/c0_index/ref.fa")
    reads = np.load(golden_dir + "/c0_reads.npz")["reads"]
    codes = reads.reshape(-1); offs = (np.arange(len(reads) + 1) * reads.shape[1]).astype(np.int64)
    g = np.load(golden_dir + "/cigar_c0.npz")
    yield idx, codes, offs, g, reads.shape[1]
    idx.close()


def test_oracle_matches_reference_golden(pkg, c0):
    idx, codes, offs, g, _ = c0
    got = ol.gen_cigar(idx, pkg.capi.default_opt(), codes, offs, g["reqs"])
    assert got[3] == 0
    assert cu.same(got[:3], (g["recs"], g["cigar"], g["md"])) == []
    assert (g["recs"]["nm"] < 0).sum() == 4 and (g["recs"]["n_cigar"] > 1).sum() > 500      # the fixture covers rejects and indels


def test_device_logic_matches_reference_golden(pkg, c0):
    idx, codes, offs, g, _ = c0
    got = emul_gen_cigar(pkg.capi, idx, pkg.capi.default_opt(), codes, offs, g["reqs"])
    assert cu.same(got, (g["recs"], g["cigar"], g["md"])) == []


def live_requests(capi, idx, codes, offs, read_len):
    """6000 requests drawn (seeded) from the oracle's regions of the C0 reads, with extra end-point variants."""
    regs, ro, _, rc = ol.seed_chain_extend(idx, capi.default_opt(), codes, offs)
    assert rc == 0
    reqs = cu.make_requests(capi, np.random.default_rng(99), regs, ro, read_len, idx.desc.l_pac, n_extra=1500)
    return reqs[np.random.default_rng(3).choice(len(reqs), 6000, replace=False)]


def test_oracle_and_device_logic_match_the_live_reference(pkg, c0):
    idx, codes, offs, g, read_len = c0
    capi = pkg.capi
    reqs = live_requests(capi, idx, codes, offs, read_len)
    assert hashlib.sha256(reqs.tobytes()).hexdigest() == refgolden.get("cigar/reqs_sha256").tobytes().decode(), \
        "the request set differs from the one the reference was run on"
    want = tuple(refgolden.get("cigar/" + k) for k in ("recs", "cigar", "md"))
    got = ol.gen_cigar(idx, capi.default_opt(), codes, offs, reqs)
    assert got[3] == 0 and cu.same(got[:3], want) == []
    assert cu.same(emul_gen_cigar(capi, idx, capi.default_opt(), codes, offs, reqs), want) == []


def test_non_default_scoring_device_logic_matches_oracle(pkg, c0):
    idx, codes, offs, g, _ = c0
    o = pkg.capi.default_opt()
    o.o_del, o.e_del, o.o_ins, o.e_ins = 4, 2, 5, 1
    reqs = g["reqs"][:1500]
    want = ol.gen_cigar(idx, o, codes, offs, reqs)
    assert want[3] == 0
    assert cu.same(emul_gen_cigar(pkg.capi, idx, o, codes, offs, reqs), want[:3]) == []
