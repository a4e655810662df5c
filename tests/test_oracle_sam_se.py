"""Single-end SAM stage of the oracle (groundwork for SURVEY 8f items 2-3): mem_mark_primary_se, mem_approx_mapq_se, mem_reg2aln and the
record selection of mem_reg2sam against the SAM the UNMODIFIED reference writes for the same reads in single-end mode (recorded by
tests/golden/make_live_golden.py): FLAG, RNAME, POS, MAPQ, CIGAR with soft / hard clips, NM, MD, AS, XS of every line, supplementary
lines included."""
import ctypes as C
import numpy as np
import pytest
import oracle_lib as ol
import refgolden

ALN_DT = np.dtype([("read", "<i4"), ("flag", "<i4"), ("rid", "<i4"), ("mapq", "<i4"), ("nm", "<i4"), ("score", "<i4"), ("sub", "<i4"), ("is_rev", "<i4"),
                   ("is_alt", "<i4"), ("alt_sc", "<i4"), ("n_cigar", "<i4"), ("n_md", "<i4"), ("pos", "<i8"), ("cigar_off", "<i8"), ("md_off", "<i8")])


def oracle_sam_se(capi, idx, opt, codes, offs, regs, ro, id_base=0):
    codes = np.ascontiguousarray(codes, np.uint8); offs = np.ascontiguousarray(offs, np.int64)
    regs = np.ascontiguousarray(regs).copy(); ro = np.ascontiguousarray(ro, np.int64)
    rb = capi.ReadBatch(len(offs) - 1, codes.ctypes.data, offs.ctypes.data)
    al = C.c_void_p(); cg = C.c_void_p(); md = C.c_void_p(); na = C.c_int64(); no = C.c_int64(); nm = C.c_int64()
    L = ol.lib()
    rc = L.bm2o_sam_se(C.byref(idx.desc), C.byref(opt), C.byref(rb), regs.ctypes.data_as(C.c_void_p), ro.ctypes.data_as(C.c_void_p), C.c_int64(id_base),
                       C.byref(al), C.byref(na), C.byref(cg), C.byref(no), C.byref(md), C.byref(nm))
    assert rc == 0
    def arr(p, n, dt):
        dt = np.dtype(dt)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(n, 1) * dt.itemsize,))[:n * dt.itemsize].view(dt).copy()
    out = arr(al, na.value, ALN_DT), arr(cg, no.value, "<u4"), arr(md, nm.value, "u1")
    for p in (al, cg, md):
        L.bm2o_free(p)
    return out


def sam_fields(alns, cigar, md, names, soft_clip_all=False):
    """What mem_aln2sam prints for an alignment list (src/bwamem.cpp:1592-1730): one tuple per line."""
    lines = []
    which = 0; prev = -1
    for a in alns:
        which = which + 1 if a["read"] == prev else 0
        prev = a["read"]
        flag = a["flag"] | (0x4 if a["rid"] < 0 else 0) | (0x10 if a["is_rev"] else 0)
        flag = (flag & 0xffff) | (0x100 if flag & 0x10000 else 0)
        if a["rid"] < 0:
            lines.append((int(a["read"]), flag, "*", 0, 0, "*", None, None, None, None)); continue
        ops = cigar[a["cigar_off"]:a["cigar_off"] + a["n_cigar"]]
        cs = ""
        for o in ops:
            c = int(o & 0xf)
            if not soft_clip_all and not a["is_alt"] and c in (3, 4):
                c = 4 if which else 3
            cs += f"{int(o >> 4)}{'MIDSH'[c]}"
        mds = bytes(md[a["md_off"]:a["md_off"] + a["n_md"] - 1]).decode()
        lines.append((int(a["read"]), flag, names[a["rid"]], int(a["pos"]) + 1, int(a["mapq"]), cs, int(a["nm"]), mds, int(a["score"]),
                      int(a["sub"]) if a["sub"] >= 0 else None))
    return lines


def parse_sam(lines):
    out = []
    for ln in lines:
        if ln.startswith("@"):
            continue
        f = ln.rstrip("\n").split("\t")
        tags = {t[:2]: t[5:] for t in f[11:]}
        rid = int(f[0][1:])
        if f[2] == "*":
            out.append((rid, int(f[1]), "*", 0, 0, "*", None, None, None, None)); continue
        out.append((rid, int(f[1]), f[2], int(f[3]), int(f[4]), f[5], int(tags["NM"]), tags["MD"], int(tags["AS"]), int(tags["XS"]) if "XS" in tags else None))
    return out


# option sets of the single-end runs (the reads of the r1 file of C0): (id, `bwa-mem2 mem` arguments)
SE_CASES = [("default", []), ("all", ["-a"]), ("no_multi", ["-M"]), ("T50", ["-T", "50"]), ("softclip", ["-Y"]), ("primary5", ["-5"]), ("keep_supp_mapq", ["-q"])]


def se_reads(golden_dir):
    return np.load(golden_dir + "/c0_reads.npz")["reads"][0::2]              # the r1 file


@pytest.mark.parametrize("name,args", SE_CASES, ids=[c[0] for c in SE_CASES])
def test_single_end_sam_matches_reference(pkg, golden_dir, name, args):
    capi = pkg.capi
    idx = capi.Index(golden_dir + "/c0_index/ref.fa")
    reads = se_reads(golden_dir)
    codes = reads.reshape(-1); offs = (np.arange(len(reads) + 1) * reads.shape[1]).astype(np.int64)
    want = parse_sam(refgolden.sam_lines("se/" + name))
    opt = capi.default_opt()
    if "-a" in args: opt.flag |= 0x8
    if "-M" in args: opt.flag |= 0x10
    if "-Y" in args: opt.flag |= 0x200
    if "-5" in args: opt.flag |= 0x1800                                      # MEM_F_PRIMARY5 | MEM_F_KEEP_SUPP_MAPQ (src/fastmap.cpp:673)
    if "-q" in args: opt.flag |= 0x1000
    if "-T" in args: opt.T = int(args[args.index("-T") + 1])
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    assert rc == 0
    alns, cig, md = oracle_sam_se(capi, idx, opt, codes, offs, regs, ro)
    names = [l.split()[1] for i, l in enumerate(open(golden_dir + "/c0_index/ref.fa.ann")) if i % 2 == 1]
    got = sam_fields(alns, cig, md, names, soft_clip_all="-Y" in args)
    assert len(got) == len(want), (len(got), len(want))
    bad = [i for i in range(len(got)) if got[i] != want[i]]
    assert not bad, (len(bad), [(got[i], want[i]) for i in bad[:3]])
    assert sum(1 for w in want if w[1] & 0x800) >= 3 or "-M" in args or "-a" in args or "-T" in args
    idx.close()


# ---- the single-end device logic (sam_se_read_d of sam_device.cuh, compiled for the host inside the bounded arenas) --------------------------
def emul_sam_se(capi, idx, opt, codes, offs, regs, ro, id_base=0):
    import test_oracle_sam_pe as tp
    codes = np.ascontiguousarray(codes, np.uint8); offs = np.ascontiguousarray(offs, np.int64)
    regs = np.ascontiguousarray(regs); ro = np.ascontiguousarray(ro, np.int64)
    rb = capi.ReadBatch(len(offs) - 1, codes.ctypes.data, offs.ctypes.data)
    rc_ = C.c_void_p(); cg = C.c_void_p(); md = C.c_void_p(); nr = C.c_int64(); no = C.c_int64(); nm = C.c_int64()
    rr = C.c_void_p(); xa = C.c_void_p(); nxa = C.c_int64(); xc = C.c_void_p(); nxc = C.c_int64()
    rc = tp._emul().emul_sam_se(C.byref(idx.desc), C.byref(opt), C.byref(rb), regs.ctypes.data_as(C.c_void_p), ro.ctypes.data_as(C.c_void_p), C.c_int64(id_base),
                                C.byref(rc_), C.byref(nr), C.byref(cg), C.byref(no), C.byref(md), C.byref(nm), C.byref(rr), C.byref(xa), C.byref(nxa), C.byref(xc), C.byref(nxc))
    assert rc == 0, rc
    def arr(p, n, dt):
        dt = np.dtype(dt)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(n, 1) * dt.itemsize,))[:n * dt.itemsize].view(dt).copy()
    out = arr(rc_, nr.value, tp.REC_DT), arr(cg, no.value, "<u4"), arr(md, nm.value, "u1")
    for p in (rc_, cg, md, rr, xa, xc):
        ol.lib().bm2o_free(p)
    return out


def rec_fields(recs, cigar, md, names):
    """The tuples of parse_sam from printed records (flags and clip letters already as printed)."""
    out = []
    for r in recs:
        if r["rid"] < 0:
            out.append((int(r["read"]), int(r["flag"]), "*", 0, 0, "*", None, None, None, None)); continue
        cs = "".join(f"{int(o >> 4)}{'MIDSH'[int(o & 0xf)]}" for o in cigar[r["cigar_off"]:r["cigar_off"] + r["n_cigar"]])
        out.append((int(r["read"]), int(r["flag"]), names[r["rid"]], int(r["pos"]), int(r["mapq"]), cs, int(r["nm"]),
                    bytes(md[r["md_off"]:r["md_off"] + r["n_md"] - 1]).decode(), int(r["score"]), int(r["sub"]) if r["sub"] >= 0 else None))
    return out


@pytest.mark.parametrize("name,args", SE_CASES[:6], ids=[c[0] for c in SE_CASES[:6]])
def test_single_end_device_logic_matches_reference(pkg, golden_dir, name, args):
    capi = pkg.capi
    idx = capi.Index(golden_dir + "/c0_index/ref.fa")
    reads = se_reads(golden_dir)
    codes = reads.reshape(-1); offs = (np.arange(len(reads) + 1) * reads.shape[1]).astype(np.int64)
    want = parse_sam(refgolden.sam_lines("se/" + name))
    opt = capi.default_opt()
    if "-a" in args: opt.flag |= 0x8
    if "-M" in args: opt.flag |= 0x10
    if "-Y" in args: opt.flag |= 0x200
    if "-5" in args: opt.flag |= 0x1800
    if "-T" in args: opt.T = int(args[args.index("-T") + 1])
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    names = [l.split()[1] for i, l in enumerate(open(golden_dir + "/c0_index/ref.fa.ann")) if i % 2 == 1]
    got = rec_fields(*emul_sam_se(capi, idx, opt, codes, offs, regs, ro), names)
    assert len(got) == len(want), (len(got), len(want))
    bad = [i for i in range(len(got)) if got[i] != want[i]]
    assert not bad, (len(bad), [(got[i], want[i]) for i in bad[:3]])
    idx.close()

