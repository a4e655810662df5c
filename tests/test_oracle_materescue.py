"""Mate rescue around the local alignment (SURVEY 8f item 1, groundwork): the oracle's mem_pestat and mem_matesw against the UNMODIFIED
reference - mem_pestat through the link-time hook of ref_driver (dump of a normal `mem` run), mem_matesw through `ref_driver matesw`,
which runs the rescue block of mem_sam_pe with the reference's own mem_matesw on the pairs of a file (mate_input).  Both outputs are
recorded by tests/golden/make_live_golden.py."""
import ctypes as C, hashlib, os, struct, subprocess
import numpy as np
import pytest
import oracle_lib as ol
import refgolden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("rb", "re", "qb", "qe", "rid", "score", "truesc", "sub", "alt_sc", "csub", "sub_n", "w", "seedcov", "secondary", "secondary_all", "seedlen0",
          "n_comp_is_alt", "frac_rep", "hash")


@pytest.fixture(scope="module")
def c0(pkg, golden_dir):
    capi = pkg.capi
    idx = capi.Index(golden_dir + "/c0_index/ref.fa")
    reads = np.load(golden_dir + "/c0_reads.npz")["reads"]
    codes = reads.reshape(-1); offs = (np.arange(len(reads) + 1) * reads.shape[1]).astype(np.int64)
    opt = capi.default_opt()
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    assert rc == 0
    buf = refgolden.get("mate/pestat").tobytes()
    assert len(buf) == 4 + 4 * 28
    pes = [struct.unpack_from("<iiidd", buf, 4 + 28 * d) for d in range(4)]
    yield capi, idx, opt, reads, regs, ro, pes
    idx.close()


def mate_input(reads, regs, ro, pes):
    """The input file of `ref_driver matesw`: the pestat bounds, then per read its codes and its regs."""
    lh = np.array([v for d in range(4) for v in pes[d][:3]], np.int32)
    out = [lh.tobytes(), struct.pack("<q", len(reads) // 2)]
    for r in range(len(reads)):
        out += [struct.pack("<i", reads.shape[1]), reads[r].tobytes()]
        a = regs[ro[r]:ro[r + 1]]
        out += [struct.pack("<i", len(a)), a.tobytes()]
    return b"".join(out)


def test_pestat_matches_reference(c0):
    capi, idx, opt, reads, regs, ro, pes = c0
    lh = np.zeros(12, np.int32); as_ = np.zeros(8, np.float64)
    regs_c = np.ascontiguousarray(regs); ro_c = np.ascontiguousarray(ro, np.int64)
    ol.lib().bm2o_pestat(C.byref(opt), C.c_int64(idx.desc.l_pac), C.c_int32(len(reads)), regs_c.ctypes.data_as(C.c_void_p), ro_c.ctypes.data_as(C.c_void_p),
                         lh.ctypes.data_as(C.c_void_p), as_.ctypes.data_as(C.c_void_p))
    for d in range(4):
        assert tuple(lh[3 * d:3 * d + 3]) == pes[d][:3], (d, lh, pes)
        if not pes[d][2]:
            assert as_[2 * d] == pes[d][3] and as_[2 * d + 1] == pes[d][4]       # same double arithmetic
    assert pes[1][2] == 0 and pes[1][0] > 0                                      # FR is the orientation of the data set


def test_product_pestat_matches_reference(c0):
    """bm2_pestat of the C ABI (host code of the product, bwa-mem2_b200/csrc/pestat.cpp) against the reference's mem_pestat dump."""
    capi, idx, opt, reads, regs, ro, pes = c0
    got = capi.pestat(opt, idx.desc.l_pac, regs, ro)
    for d in range(4):
        assert (int(got[d]["low"]), int(got[d]["high"]), int(got[d]["failed"])) == pes[d][:3], (d, got, pes)
        assert got[d]["avg"] == pes[d][3] and got[d]["std"] == pes[d][4]          # bit-identical doubles (0 for a failed orientation)
    # degenerate chunks: no reads, reads without regions
    empty = capi.pestat(opt, idx.desc.l_pac, regs[:0], np.zeros(1, np.int64))
    assert all(int(e["failed"]) == 1 for e in empty)
    none = capi.pestat(opt, idx.desc.l_pac, regs[:0], np.zeros(9, np.int64))
    assert all(int(e["failed"]) == 1 for e in none)


def test_matesw_matches_reference(c0):
    capi, idx, opt, reads, regs, ro, pes = c0
    lh = np.array([v for d in range(4) for v in pes[d][:3]], np.int32)
    assert hashlib.sha256(mate_input(reads, regs, ro, pes)).hexdigest() == refgolden.get("mate/matesw_in_sha256").tobytes().decode(), \
        "the regs differ from those the reference was given"
    buf = refgolden.get("mate/matesw_out").tobytes()
    L = ol.lib()
    pos = 0; n_calls = 0; n_sw = 0; n_added = 0
    cur_pair = -1; a = None
    while pos < len(buf):
        pr, i, j, n_ref, n_after = struct.unpack_from("<iiiii", buf, pos); pos += 20
        want = np.frombuffer(buf, capi.REG_DT, n_after, pos); pos += n_after * capi.REG_DT.itemsize
        if pr != cur_pair:                    # a new pair: the state mem_sam_pe starts from
            cur_pair = pr
            a = [regs[ro[2 * pr]:ro[2 * pr + 1]].copy(), regs[ro[2 * pr + 1]:ro[2 * pr + 2]].copy()]
            b = [x[x["score"] >= x["score"][0] - opt.pen_unpaired].copy() if len(x) else x.copy() for x in a]
        anchor = np.ascontiguousarray(b[i][j:j + 1])
        ma = np.zeros(len(a[1 - i]) + 4, capi.REG_DT); ma[:len(a[1 - i])] = a[1 - i]
        n_ma = C.c_int32(len(a[1 - i]))
        ms = np.ascontiguousarray(reads[2 * pr + (1 - i)])
        n = L.bm2o_matesw(C.byref(idx.desc), C.byref(opt), lh.ctypes.data_as(C.c_void_p), anchor.ctypes.data_as(C.c_void_p), C.c_int32(len(ms)),
                          ms.ctypes.data_as(C.c_void_p), ma.ctypes.data_as(C.c_void_p), C.byref(n_ma))
        got = ma[:n_ma.value]
        assert n == n_ref and len(got) == n_after, (pr, i, j, n, n_ref, len(got), n_after)
        for fld in FIELDS:
            assert np.array_equal(got[fld], want[fld]), (pr, i, j, fld, got[fld], want[fld])
        n_added += len(got) - len(a[1 - i]) if len(got) > len(a[1 - i]) else 0
        a[1 - i] = got.copy()
        n_calls += 1; n_sw += n
    print("mem_matesw calls", n_calls, "orientations aligned", n_sw, "regs added", n_added)
    assert n_calls > 500 and n_sw > 20 and n_added > 5, (n_calls, n_sw, n_added)


def test_device_logic_of_the_rescue_block_matches_the_oracle(c0):
    """bwa-mem2_b200/csrc/mate_device.cuh (matesw_d, mate_rescue_pair_d over ksw_device.cuh and the tail's sort_dedup_patch_d), compiled for
    the host, against the oracle's chained mem_matesw calls (pinned to the reference by the test above)."""
    capi, idx, opt, reads, regs, ro, pes = c0
    d = os.path.join(ROOT, "tests", "host_emul")
    so = os.path.join(d, "libmateemul.so")
    srcs = [os.path.join(d, "mate_emul.cpp")] + [os.path.join(ROOT, "bwa-mem2_b200", "csrc", f) for f in ("mate_device.cuh", "ksw_device.cuh", "ext_device.cuh", "chain_device.cuh", "hd.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-g", "-std=c++17", "-fPIC", "-shared", "-w", "-ffp-contract=off", "-I" + os.path.join(ROOT, "bwa-mem2_b200", "csrc"),
                               "-I" + os.path.join(ROOT, "include"), srcs[0], "-o", so])
    E = C.CDLL(so); E.emul_mate_rescue.restype = C.c_longlong
    lh = np.array([v for dd in range(4) for v in pes[dd][:3]], np.int32)
    codes = np.ascontiguousarray(reads.reshape(-1)); offs = (np.arange(len(reads) + 1) * reads.shape[1]).astype(np.int64)
    rb = capi.ReadBatch(len(reads), codes.ctypes.data, offs.ctypes.data)
    regs_c = np.ascontiguousarray(regs); ro_c = np.ascontiguousarray(ro, np.int64)
    cap = len(regs) + 8 * len(reads) + 1024
    out = np.zeros(cap, capi.REG_DT); out_off = np.zeros(len(reads) + 1, np.int64)
    tot = E.emul_mate_rescue(C.byref(idx.desc), C.byref(opt), C.byref(rb), regs_c.ctypes.data_as(C.c_void_p), ro_c.ctypes.data_as(C.c_void_p),
                             lh.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), C.c_int64(cap), out_off.ctypes.data_as(C.c_void_p))
    assert tot > 1000, tot
    # the oracle's chain for every pair
    L = ol.lib(); n_sw = 0
    for p in range(len(reads) // 2):
        a = [regs[ro[2 * p]:ro[2 * p + 1]].copy(), regs[ro[2 * p + 1]:ro[2 * p + 2]].copy()]
        b = [x[x["score"] >= x["score"][0] - opt.pen_unpaired].copy() if len(x) else x.copy() for x in a]
        for i in (0, 1):
            for j in range(min(len(b[i]), opt.max_matesw)):
                anchor = np.ascontiguousarray(b[i][j:j + 1])
                ma = np.zeros(len(a[1 - i]) + 4, capi.REG_DT); ma[:len(a[1 - i])] = a[1 - i]
                n_ma = C.c_int32(len(a[1 - i])); ms = np.ascontiguousarray(reads[2 * p + (1 - i)])
                n_sw += L.bm2o_matesw(C.byref(idx.desc), C.byref(opt), lh.ctypes.data_as(C.c_void_p), anchor.ctypes.data_as(C.c_void_p), C.c_int32(len(ms)),
                                      ms.ctypes.data_as(C.c_void_p), ma.ctypes.data_as(C.c_void_p), C.byref(n_ma))
                a[1 - i] = ma[:n_ma.value].copy()
        for i in (0, 1):
            got = out[out_off[2 * p + i]:out_off[2 * p + i + 1]]
            assert len(got) == len(a[i]), (p, i, len(got), len(a[i]))
            for fld in FIELDS:
                assert np.array_equal(got[fld], a[i][fld]), (p, i, fld)
    assert n_sw == tot
