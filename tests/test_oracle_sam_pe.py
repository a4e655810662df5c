"""Paired-end SAM stage of the oracle (groundwork for SURVEY 8f): mate rescue + mem_mark_primary_se + mem_pair + the paired / unpaired MAPQ
logic of mem_sam_pe + the columns of mem_aln2sam, against the committed SAM of the UNMODIFIED reference (tests/golden/c0.sam) and
against its SAM of runs with options (recorded by tests/golden/make_live_golden.py): FLAG, RNAME, POS, MAPQ, CIGAR, RNEXT, PNEXT, TLEN,
NM, MD, AS, XS of every line."""
import ctypes as C, os, struct, subprocess, tempfile
import numpy as np
import pytest
import oracle_lib as ol
import refgolden

REC_DT = np.dtype([("read", "<i4"), ("flag", "<i4"), ("rid", "<i4"), ("mapq", "<i4"), ("rnext", "<i4"), ("tlen_valid", "<i4"), ("nm", "<i4"), ("score", "<i4"),
                   ("sub", "<i4"), ("n_cigar", "<i4"), ("n_md", "<i4"), ("_pad", "<i4"), ("pos", "<i8"), ("pnext", "<i8"), ("tlen", "<i8"),
                   ("cigar_off", "<i8"), ("md_off", "<i8")])


def oracle_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_):
    codes = np.ascontiguousarray(codes, np.uint8); offs = np.ascontiguousarray(offs, np.int64)
    regs = np.ascontiguousarray(regs); ro = np.ascontiguousarray(ro, np.int64)
    lh = np.ascontiguousarray(lh, np.int32); as_ = np.ascontiguousarray(as_, np.float64)
    rb = capi.ReadBatch(len(offs) - 1, codes.ctypes.data, offs.ctypes.data)
    rc_ = C.c_void_p(); cg = C.c_void_p(); md = C.c_void_p(); nr = C.c_int64(); no = C.c_int64(); nm = C.c_int64()
    L = ol.lib()
    rc = L.bm2o_sam_pe(C.byref(idx.desc), C.byref(opt), C.byref(rb), regs.ctypes.data_as(C.c_void_p), ro.ctypes.data_as(C.c_void_p),
                       lh.ctypes.data_as(C.c_void_p), as_.ctypes.data_as(C.c_void_p), C.c_int64(0), C.byref(rc_), C.byref(nr), C.byref(cg), C.byref(no),
                       C.byref(md), C.byref(nm))
    assert rc == 0
    def arr(p, n, dt):
        dt = np.dtype(dt)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(n, 1) * dt.itemsize,))[:n * dt.itemsize].view(dt).copy()
    out = arr(rc_, nr.value, REC_DT), arr(cg, no.value, "<u4"), arr(md, nm.value, "u1")
    for p in (rc_, cg, md):
        L.bm2o_free(p)
    return out


def fields(recs, cigar, md, names):
    out = []
    for r in recs:
        rname = names[r["rid"]] if r["rid"] >= 0 else "*"
        cs = "".join(f"{int(o >> 4)}{'MIDSH'[int(o & 0xf)]}" for o in cigar[r["cigar_off"]:r["cigar_off"] + r["n_cigar"]]) or "*"
        rnext = "*" if r["rnext"] < 0 else ("=" if r["rnext"] == r["rid"] else names[r["rnext"]])
        tags = {}
        if r["n_cigar"]:
            tags["NM"] = str(int(r["nm"])); tags["MD"] = bytes(md[r["md_off"]:r["md_off"] + r["n_md"] - 1]).decode()
        if r["score"] >= 0: tags["AS"] = str(int(r["score"]))
        if r["sub"] >= 0: tags["XS"] = str(int(r["sub"]))
        out.append((int(r["read"]), int(r["flag"]), rname, int(r["pos"]), int(r["mapq"]), cs, rnext, int(r["pnext"]), int(r["tlen"]), tags))
    return out


def parse_sam(lines):
    out = []; idx = {}
    for ln in lines:
        if ln.startswith("@"):
            continue
        f = ln.rstrip("\n").split("\t")
        flag = int(f[1])
        read = 2 * int(f[0][1:]) + (1 if flag & 0x80 else 0)
        tags = {t[:2]: t[5:] for t in f[11:] if t[:2] in ("NM", "MD", "AS", "XS")}
        out.append((read, flag, f[2], int(f[3]), int(f[4]), f[5], f[6], int(f[7]), int(f[8]), tags))
    return out


def _compare(got, want):
    assert len(got) == len(want), (len(got), len(want))
    bad = [i for i in range(len(got)) if got[i] != want[i]]
    assert not bad, (len(bad), [(got[i], want[i]) for i in bad[:3]])


@pytest.fixture(scope="module")
def c0(pkg, golden_dir):
    capi = pkg.capi
    idx = capi.Index(golden_dir + "/c0_index/ref.fa")
    reads = np.load(golden_dir + "/c0_reads.npz")["reads"]
    codes = reads.reshape(-1); offs = (np.arange(len(reads) + 1) * reads.shape[1]).astype(np.int64)
    names = [l.split()[1] for i, l in enumerate(open(golden_dir + "/c0_index/ref.fa.ann")) if i % 2 == 1]
    yield capi, idx, reads, codes, offs, names
    idx.close()


def _pestat(capi, idx, opt, reads, regs, ro):
    lh = np.zeros(12, np.int32); as_ = np.zeros(8, np.float64)
    regs_c = np.ascontiguousarray(regs); ro_c = np.ascontiguousarray(ro, np.int64)
    ol.lib().bm2o_pestat(C.byref(opt), C.c_int64(idx.desc.l_pac), C.c_int32(len(reads)), regs_c.ctypes.data_as(C.c_void_p), ro_c.ctypes.data_as(C.c_void_p),
                         lh.ctypes.data_as(C.c_void_p), as_.ctypes.data_as(C.c_void_p))
    return lh, as_


def test_paired_end_sam_matches_reference_golden(c0, golden_dir):
    capi, idx, reads, codes, offs, names = c0
    opt = capi.default_opt()
    opt.flag |= 0x2                                   # MEM_F_PE (two input files)
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    lh, as_ = _pestat(capi, idx, opt, reads, regs, ro)
    recs, cig, md = oracle_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_)
    want = parse_sam(open(golden_dir + "/c0.sam"))
    _compare(fields(recs, cig, md, names), want)
    flags = np.array([w[1] for w in want])
    assert (flags & 0x2).sum() > 800 and (flags & 0x800).sum() >= 3 and (flags & 0x4).sum() >= 5      # proper pairs, supplementary, unmapped


# option sets of the paired-end runs: (id, `bwa-mem2 mem` arguments)
PE_CASES = [("all", ["-a"]), ("no_multi", ["-M"]), ("no_pairing", ["-P"]), ("no_rescue", ["-S"]), ("softclip_T40", ["-Y", "-T", "40"]), ("U9", ["-U", "9"]),
            ("primary5", ["-5"]), ("keep_supp_mapq", ["-q"]), ("primary5_P_a", ["-5", "-P", "-a"]), ("all_no_multi", ["-a", "-M"])]


@pytest.mark.parametrize("name,args", PE_CASES, ids=[c[0] for c in PE_CASES])
def test_paired_end_sam_matches_the_live_reference(c0, name, args):
    capi, idx, reads, codes, offs, names = c0
    ref_sam = refgolden.sam_lines("pe/" + name)
    opt = capi.default_opt(); opt.flag |= 0x2
    for fl, bit in (("-a", 0x8), ("-M", 0x10), ("-P", 0x4), ("-S", 0x20), ("-Y", 0x200), ("-5", 0x1800), ("-q", 0x1000)):
        if fl in args: opt.flag |= bit
    if "-T" in args: opt.T = int(args[args.index("-T") + 1])
    if "-U" in args: opt.pen_unpaired = int(args[args.index("-U") + 1])
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    lh, as_ = _pestat(capi, idx, opt, reads, regs, ro)
    recs, cig, md = oracle_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_)
    _compare(fields(recs, cig, md, names), parse_sam(ref_sam))
    # the device logic's records, formatted by tests/sam_text.py, against the reference's text (from FLAG on)
    import sam_text
    e_recs, e_cig, e_md, e_xa, e_aux = emul_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_, xa_names=names)
    refgolden.assert_sam_text("pe/" + name, sam_text.format_lines(e_recs, e_cig, e_md, e_xa, names, codes, offs, is_alt=e_aux[:, 1], n_mc=e_aux[:, 2]))


def oracle_sam_text(capi, idx, opt, codes, offs, regs, ro, lh, as_, names, qual_char="I"):
    codes = np.ascontiguousarray(codes, np.uint8); offs = np.ascontiguousarray(offs, np.int64)
    regs = np.ascontiguousarray(regs); ro = np.ascontiguousarray(ro, np.int64)
    lh = np.ascontiguousarray(lh, np.int32); as_ = np.ascontiguousarray(as_, np.float64)
    rb = capi.ReadBatch(len(offs) - 1, codes.ctypes.data, offs.ctypes.data)
    quals = (qual_char * len(codes)).encode()
    arr = (C.c_char_p * len(names))(*[n.encode() for n in names])
    text = C.c_void_p(); ln = C.c_int64()
    L = ol.lib()
    rc = L.bm2o_sam_pe_text(C.byref(idx.desc), C.byref(opt), C.byref(rb), C.c_char_p(quals), arr, regs.ctypes.data_as(C.c_void_p), ro.ctypes.data_as(C.c_void_p),
                            lh.ctypes.data_as(C.c_void_p), as_.ctypes.data_as(C.c_void_p), C.c_int64(0), C.byref(text), C.byref(ln))
    assert rc == 0
    out = C.string_at(text, ln.value).decode()
    L.bm2o_free(text)
    return out.split("\n")[:-1]


def test_paired_end_sam_text_is_byte_identical_to_the_reference_golden(c0, golden_dir):
    """Every character of every SAM line after QNAME (all columns, SEQ / QUAL with hard clips, NM MD MC AS XS SA pa XA tags)."""
    capi, idx, reads, codes, offs, names = c0
    opt = capi.default_opt(); opt.flag |= 0x2
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    lh, as_ = _pestat(capi, idx, opt, reads, regs, ro)
    got = oracle_sam_text(capi, idx, opt, codes, offs, regs, ro, lh, as_, names)
    want = [ln.rstrip("\n").split("\t", 1)[1] for ln in open(golden_dir + "/c0.sam") if not ln.startswith("@")]
    assert len(got) == len(want)
    bad = [i for i in range(len(got)) if got[i] != want[i]]
    assert not bad, (len(bad), [(got[i], want[i]) for i in bad[:2]])
    assert sum("SA:Z:" in w for w in want) >= 6 and sum("MC:Z:" in w for w in want) > 900


XA_ALT = "c1_alt\t0\tc1\t20001\t60\t40000M\t*\t0\t0\t*\t*\n"


def xa_dataset(work):
    """A genome with 2-4 copy segmental duplications and an ALT contig, written to work/ref.fa (+ .alt), and 1500 read pairs written to
    work/r1.fq, work/r2.fq.  -> (contig names, contigs as 2-bit codes, reads with the pairs interleaved)."""
    rng = np.random.default_rng(12)
    ctgs = []
    for c in range(3):
        g = rng.integers(0, 4, 120_000).astype(np.uint8)
        for _ in range(25):                                   # duplications: 500-bp segments, 1-3 extra copies, ~1 % divergence
            L = 500; src = int(rng.integers(0, len(g) - L)); seg = g[src:src + L]
            for _ in range(int(rng.integers(1, 4))):
                cp = seg.copy(); mut = rng.random(L) < 0.01; cp[mut] = rng.integers(0, 4, int(mut.sum()))
                dst = int(rng.integers(0, len(g) - L)); g[dst:dst + L] = cp
        ctgs.append(g)
    alt = ctgs[0][20_000:60_000].copy(); mut = rng.random(len(alt)) < 0.005; alt[mut] = rng.integers(0, 4, int(mut.sum()))
    ctgs.append(alt)                                          # an ALT contig: a diverged copy of a stretch of the first one
    names = ["c1", "c2", "c3", "c1_alt"]
    with open(work + "/ref.fa", "w") as f:
        for n, g in zip(names, ctgs):
            f.write(f">{n}\n"); s = "".join("ACGT"[b] for b in g)
            f.write("\n".join(s[i:i + 80] for i in range(0, len(s), 80)) + "\n")
    with open(work + "/ref.fa.alt", "w") as f:
        f.write(XA_ALT)
    n_pairs = 1500; L = 151
    reads = np.zeros((2 * n_pairs, L), np.uint8)
    comp = np.array([3, 2, 1, 0, 4], np.uint8)
    for p in range(n_pairs):
        c = int(rng.integers(0, 4)); g = ctgs[c]            # also from the ALT contig: its reads make the primary-assembly hit the secondary (pa tag)
        ins = int(rng.normal(400, 40)); ins = max(ins, L + 10)
        st = int(rng.integers(0, len(g) - ins))
        frag = g[st:st + ins].copy(); mut = rng.random(ins) < 0.01; frag[mut] = rng.integers(0, 4, int(mut.sum()))
        r1 = frag[:L]; r2 = comp[frag[-L:][::-1]]
        if rng.random() < 0.5: r1, r2 = r2, r1
        reads[2 * p] = r1; reads[2 * p + 1] = r2
    for k, name in ((0, "r1.fq"), (1, "r2.fq")):
        with open(os.path.join(work, name), "w") as f:
            for i, r in enumerate(reads[k::2]):
                f.write(f"@p{i}\n{''.join('ACGTN'[c] for c in r)}\n+\n{'I' * L}\n")
    return names, ctgs, reads


def test_sam_text_with_xa_and_alt_tags_matches_the_live_reference(pkg):
    """A genome with 2-4 copy segmental duplications (XA tags) and ALT contigs (pa tag, ALT-aware primary marking): byte-identical text
    against the reference's SAM of the same reads on the same genome (its index written by bwa_mem2_b200.index_build, which writes the
    reference's index bytes)."""
    import importlib
    capi = pkg.capi
    work = tempfile.mkdtemp(prefix="bm2_xa_")
    names, ctgs, reads = xa_dataset(work)
    importlib.import_module("bwa_mem2_b200.index_build").write_index(work + "/ref.fa", list(zip(names, ctgs)), device="cpu")
    L = reads.shape[1]
    want = [ln.rstrip("\n").split("\t", 1)[1] for ln in refgolden.sam_lines("pe/xa_alt")]
    idx = capi.Index(work + "/ref.fa")
    opt = capi.default_opt(); opt.flag |= 0x2
    codes = reads.reshape(-1); offs = (np.arange(len(reads) + 1) * L).astype(np.int64)
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    lh, as_ = _pestat(capi, idx, opt, reads, regs, ro)
    refgolden.assert_sam_text("pe/xa_alt", oracle_sam_text(capi, idx, opt, codes, offs, regs, ro, lh, as_, names))
    assert sum("XA:Z:" in w for w in want) > 30 and sum("pa:f:" in w for w in want) > 5, (sum("XA:Z:" in w for w in want), sum("pa:f:" in w for w in want))
    # the device logic's XA entries (sam_gen_alt_d) against the reference's XA tags, record by record
    e_recs, e_cig, e_md, e_xa, e_aux = emul_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_, xa_names=names)
    assert e_xa == xa_of_lines(want)
    import sam_text                                                  # ... and the whole text from the records: SEQ / QUAL, MC, SA, pa included
    refgolden.assert_sam_text("pe/xa_alt", sam_text.format_lines(e_recs, e_cig, e_md, e_xa, names, codes, offs, is_alt=e_aux[:, 1], n_mc=e_aux[:, 2]))
    pa_want = [([f for f in w.split("\t") if f.startswith("pa:f:")] or [""])[0] for w in want]
    pa_got = [("pa:f:%.3f" % (float(r["score"]) / float(r["_pad"]))) if r["_pad"] > 0 and not (r["flag"] & 0x100) else "" for r in e_recs]
    assert pa_got == pa_want                                         # SamRec::alt_sc
    idx.close()


# ---- the SAM-stage device logic (sam_device.cuh + mate_device.cuh, compiled for the host) against the oracle -----------------------------
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_EMUL = None


def _emul():
    global _EMUL
    if _EMUL is None:
        ol.lib()
        d = os.path.join(ROOT, "tests", "host_emul")
        so = os.path.join(d, "libsamemul.so")
        srcs = [os.path.join(d, "sam_emul.cpp")] + [os.path.join(ROOT, "bwa-mem2_b200", "csrc", f) for f in
                                                     ("../../tests/host_emul/ksw_warp_emul.cpp", "ksw_warp.cuh", "sam_layout.cuh", "sam_device.cuh", "mate_device.cuh", "ksw_device.cuh", "cigar_device.cuh", "ext_device.cuh", "chain_device.cuh", "hd.h")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(s) for s in srcs):
            subprocess.check_call(["g++", "-O2", "-g", "-std=c++17", "-fPIC", "-shared", "-w", "-ffp-contract=off", "-I" + os.path.join(ROOT, "bwa-mem2_b200", "csrc"),
                                   "-I" + os.path.join(ROOT, "include"), srcs[0], os.path.join(d, "ksw_warp_emul.cpp"), "-o", so])
        _EMUL = C.CDLL(so)
    return _EMUL


XA_DT = np.dtype([("read", "<i4"), ("reg", "<i4"), ("rid", "<i4"), ("is_rev", "<i4"), ("nm", "<i4"), ("n_cigar", "<i4"), ("pos", "<i8"), ("cigar_off", "<i8")])


def emul_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_, xa_names=None):
    """-> (recs, cigar, md); with xa_names also the XA string of every record ('' for none), built from the device logic's XA entries."""
    codes = np.ascontiguousarray(codes, np.uint8); offs = np.ascontiguousarray(offs, np.int64)
    regs = np.ascontiguousarray(regs); ro = np.ascontiguousarray(ro, np.int64)
    lh = np.ascontiguousarray(lh, np.int32); as_ = np.ascontiguousarray(as_, np.float64)
    rb = capi.ReadBatch(len(offs) - 1, codes.ctypes.data, offs.ctypes.data)
    rc_ = C.c_void_p(); cg = C.c_void_p(); md = C.c_void_p(); nr = C.c_int64(); no = C.c_int64(); nm = C.c_int64()
    rr = C.c_void_p(); xa = C.c_void_p(); nxa = C.c_int64(); xc = C.c_void_p(); nxc = C.c_int64()
    rc = _emul().emul_sam_pe(C.byref(idx.desc), C.byref(opt), C.byref(rb), regs.ctypes.data_as(C.c_void_p), ro.ctypes.data_as(C.c_void_p),
                             lh.ctypes.data_as(C.c_void_p), as_.ctypes.data_as(C.c_void_p), C.c_int64(0), C.byref(rc_), C.byref(nr), C.byref(cg), C.byref(no),
                             C.byref(md), C.byref(nm), C.byref(rr), C.byref(xa), C.byref(nxa), C.byref(xc), C.byref(nxc))
    assert rc == 0, rc
    def arr(p, n, dt):
        dt = np.dtype(dt)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(n, 1) * dt.itemsize,))[:n * dt.itemsize].view(dt).copy()
    out = arr(rc_, nr.value, REC_DT), arr(cg, no.value, "<u4"), arr(md, nm.value, "u1")
    aux = arr(rr, 3 * nr.value, "<i4").reshape(-1, 3); xas = arr(xa, nxa.value, XA_DT); xops = arr(xc, nxc.value, "<u4")      # (reg, is_alt, n_mc) per record
    rec_reg = aux[:, 0]
    for p in (rc_, cg, md, rr, xa, xc):
        ol.lib().bm2o_free(p)
    if xa_names is None:
        return out
    by_key = {}
    for e in xas:                                                    # entries in emission order (src/bwamem_extra.cpp:153-176)
        ops = xops[e["cigar_off"]:e["cigar_off"] + e["n_cigar"]]
        txt = f"{xa_names[e['rid']]},{'+-'[e['is_rev']]}{e['pos'] + 1}," + "".join(f"{v >> 4}{'MIDSHN'[v & 15]}" for v in ops) + f",{e['nm']};"
        by_key.setdefault((int(e["read"]), int(e["reg"])), []).append(txt)
    strings = ["".join(by_key.get((int(r["read"]), int(g)), [])) if g >= 0 else "" for r, g in zip(out[0], rec_reg)]
    return out + (strings, aux)


def xa_of_lines(lines):
    out = []
    for ln in lines:
        t = [f for f in ln.split("\t") if f.startswith("XA:Z:")]
        out.append(t[0][5:] if t else "")
    return out


@pytest.mark.parametrize("mode", [1, 2], ids=["warp_per_window", "thread_per_window"])
def test_staged_rescue_equals_the_per_pair_block(c0, mode):
    """The shape of the next kernel version: the rescue's local alignments enumerated from the regions before any rescue, computed as a
    batch by the warp formulation (ksw_warp.cuh), looked up by the per-pair block.  Same records; the batch must hold what is asked for."""
    capi, idx, reads, codes, offs, names = c0
    opt = capi.default_opt(); opt.flag |= 0x2
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    lh, as_ = _pestat(capi, idx, opt, reads, regs, ro)
    want = emul_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_)
    L = _emul()
    L.emul_sam_set_staged(mode)
    try:
        got = emul_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_)
        st = (C.c_longlong * 4)(); L.emul_sam_stage_stats(st)
    finally:
        L.emul_sam_set_staged(0)
    _compare(fields(*got, names), fields(*want, names))
    jobs, used, in_place, moved = [int(v) for v in st]
    assert jobs > 50 and used > 50 and in_place == 0 and moved == 0, (jobs, used, in_place, moved)
    assert used <= jobs


def test_records_suffice_for_the_reference_text(c0, golden_dir):
    """tests/golden/c0.sam byte for byte (from FLAG on) out of the device logic's records: the columns, SEQ / QUAL with hard clips, NM MD MC AS XS SA XA."""
    import sam_text
    capi, idx, reads, codes, offs, names = c0
    opt = capi.default_opt(); opt.flag |= 0x2
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    lh, as_ = _pestat(capi, idx, opt, reads, regs, ro)
    recs, cig, md, xa, aux = emul_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_, xa_names=names)
    want = [ln.rstrip("\n").split("\t", 1)[1] for ln in open(golden_dir + "/c0.sam") if not ln.startswith("@")]
    got = sam_text.format_lines(recs, cig, md, xa, names, codes, offs, is_alt=aux[:, 1], n_mc=aux[:, 2])
    assert len(got) == len(want)
    bad = [i for i in range(len(got)) if got[i] != want[i]]
    assert not bad, (len(bad), [(got[i], want[i]) for i in bad[:2]])
    assert sum("MC:Z:" in w for w in want) > 900 and sum("SA:Z:" in w for w in want) >= 6


@pytest.mark.parametrize("flags", [0, 0x8, 0x10, 0x4, 0x20, 0x200, 0x1800, 0x1000, 0x1808], ids=["default", "all", "no_multi", "no_pairing", "no_rescue", "softclip", "primary5", "keep_supp_mapq", "primary5_all"])
def test_sam_stage_device_logic_matches_oracle(c0, flags):
    capi, idx, reads, codes, offs, names = c0
    opt = capi.default_opt(); opt.flag |= 0x2 | flags
    regs, ro, _, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    lh, as_ = _pestat(capi, idx, opt, reads, regs, ro)
    want = oracle_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_)
    got = emul_sam_pe(capi, idx, opt, codes, offs, regs, ro, lh, as_)
    _compare(fields(*got, names), fields(*want, names))
    assert len(got[0]) >= len(reads)
