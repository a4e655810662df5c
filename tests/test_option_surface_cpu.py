"""The mem_opt_t parameter surface of the hot path (`bwa-mem2 mem` options -k -w -A -B -O -E -L -c -d -r -D -s -G -N -W -y -X):
the regs of the UNMODIFIED reference run with the options on the C0 reads (ref_driver's link-time hooks; recorded by
tests/golden/make_live_golden.py), the same options are set in bm2_mem_opt_t the way src/fastmap.cpp does (incl. update_a
and bwa_fill_scmat), and both the oracle and the kernels' device logic (host emulation) must reproduce every field of every
alignment region."""
import os, shutil, tempfile
import numpy as np
import pytest
import oracle_lib as ol
import emul_lib as el
import refgolden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# option sets: (name, CLI arguments)
CASES = [
    ("k15_w50", ["-k", "15", "-w", "50"]),
    ("A2", ["-A", "2"]),                                            # update_a scales B, O, E, L, T, d, U
    ("A2_B3_O5,7_E2,1", ["-A", "2", "-B", "3", "-O", "5,7", "-E", "2,1"]),
    ("L3,7_d50", ["-L", "3,7", "-d", "50"]),
    ("c20_D0.3_r1.0", ["-c", "20", "-D", "0.3", "-r", "1.0"]),
    ("s5_G500_N30_W10", ["-s", "5", "-G", "500", "-N", "30", "-W", "10"]),
    ("y5_X0.3", ["-y", "5", "-X", "0.3"]),
    ("k25_w10_d200_B8", ["-k", "25", "-w", "10", "-d", "200", "-B", "8"]),   # -d >= 128: the 8-bit SIMD class sees a negative threshold
    ("d0", ["-d", "0"]),                                             # the SIMD kernels have no `zdrop > 0` guard
    ("d128", ["-d", "128"]),
    ("A3_d90", ["-A", "3", "-d", "90"]),                             # 8-bit band operands wrap (qlen * a)
    ("x_intractg", ["-x", "intractg"]),                              # B9 O16 L5
    # (-x pacbio on these 2x151 pairs makes the reference itself abort inside worker_sam; -x ont2d covers the same preset code)
    ("x_ont2d_k19", ["-x", "ont2d", "-k", "19"]),
    ("w150_c5", ["-w", "150", "-c", "5"]),
]


def opt_from_cli(capi, args):
    """mem_opt_t after the option parsing of src/fastmap.cpp:640-860 (the options that reach the hot path)."""
    o = capi.default_opt()
    set_ = set()
    it = iter(args)
    def two(v):
        a = v.replace(",", " ").split()
        return int(a[0]), int(a[1]) if len(a) > 1 else int(a[0])
    mode = None
    for k in it:
        v = next(it)
        if k == "-x": mode = v; continue
        if k == "-k": o.min_seed_len = int(v); set_.add("min_seed_len")
        elif k == "-w": o.w = int(v)
        elif k == "-A": o.a = int(v); set_.add("a")
        elif k == "-B": o.b = int(v); set_.add("b")
        elif k == "-O": o.o_del, o.o_ins = two(v); set_.add("o_del"); set_.add("o_ins")
        elif k == "-E": o.e_del, o.e_ins = two(v); set_.add("e_del"); set_.add("e_ins")
        elif k == "-L": o.pen_clip5, o.pen_clip3 = two(v); set_.add("pen_clip5"); set_.add("pen_clip3")
        elif k == "-c": o.max_occ = int(v)
        elif k == "-d": o.zdrop = int(v); set_.add("zdrop")
        elif k == "-r": o.split_factor = float(v); set_.add("split_factor")
        elif k == "-D": o.drop_ratio = float(v)
        elif k == "-s": o.split_width = int(v)
        elif k == "-G": o.max_chain_gap = int(v)
        elif k == "-N": o.max_chain_extend = int(v)
        elif k == "-W": o.min_chain_weight = int(v); set_.add("min_chain_weight")
        elif k == "-y": o.max_mem_intv = int(v)
        elif k == "-X": o.mask_level = float(v)
        else: raise ValueError(k)
    if mode == "intractg":                                           # src/fastmap.cpp:803-811
        for f, v in (("o_del", 16), ("o_ins", 16), ("b", 9), ("pen_clip5", 5), ("pen_clip3", 5)):
            if f not in set_: setattr(o, f, v)
    elif mode in ("pacbio", "pbref", "ont2d"):                       # :812-835
        for f, v in (("o_del", 1), ("e_del", 1), ("o_ins", 1), ("e_ins", 1), ("b", 1)):
            if f not in set_: setattr(o, f, v)
        if "split_factor" not in set_: o.split_factor = 10.0
        for f, v in (("min_chain_weight", 20 if mode == "ont2d" else 40), ("min_seed_len", 14 if mode == "ont2d" else 17), ("pen_clip5", 0), ("pen_clip3", 0)):
            if f not in set_: setattr(o, f, v)
    elif mode is not None:
        raise ValueError(mode)
    if mode is None and "a" in set_:                                 # update_a (src/fastmap.cpp:547-561), only without -x (:843)
        for f in ("b", "T", "o_del", "e_del", "o_ins", "e_ins", "zdrop", "pen_clip5", "pen_clip3", "pen_unpaired"):
            if f not in set_:
                setattr(o, f, getattr(o, f) * o.a)
    k = 0                                                            # bwa_fill_scmat (src/bwa.cpp:246-257)
    for i in range(4):
        for j in range(4):
            o.mat[k] = o.a if i == j else -o.b; k += 1
        o.mat[k] = -1; k += 1
    for j in range(5):
        o.mat[k] = -1; k += 1
    return o


# the .alt file of test_alt_contigs: two of the four C0 contigs are ALT contigs of the first
ALT_FILE = "chr3\t0\tchr1\t1\t60\t100M\t*\t0\t0\t*\t*\nchr4\t0\tchr1\t1\t60\t100M\t*\t0\t0\t*\t*\n"


@pytest.fixture(scope="module")
def c0(pkg, golden_dir):
    idx = pkg.capi.Index(golden_dir + "/c0_index/ref.fa")
    reads = np.load(golden_dir + "/c0_reads.npz")["reads"]
    codes = reads.reshape(-1); offs = (np.arange(len(reads) + 1) * reads.shape[1]).astype(np.int64)
    yield idx, codes, offs, golden_dir + "/c0_index/ref.fa"
    idx.close()


@pytest.mark.parametrize("name,args", CASES, ids=[c[0] for c in CASES])
def test_reference_oracle_and_device_logic_agree(pkg, c0, name, args):
    idx, codes, offs, prefix = c0
    opt = opt_from_cli(pkg.capi, args)
    regs, ro, cells, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    assert rc == 0
    assert refgolden.regs_differ(f"opt/{name}", regs, ro) == [], "oracle differs from the reference"
    eregs, ero = el.seed_chain_extend(idx, opt, codes, offs)
    assert np.array_equal(ero, ro) and eregs.tobytes() == regs.tobytes(), "device logic differs from the oracle"
    assert len(regs) > 1000


def test_alt_contigs(pkg, c0, golden_dir):
    """ALT-aware chaining / marking (src/bwamem.cpp:506-624, :1164-1168): the C0 index with a .alt file naming two of its four contigs."""
    idx0, codes, offs, prefix0 = c0
    d = tempfile.mkdtemp(prefix="bm2_alt_")
    for f in os.listdir(os.path.dirname(prefix0)):
        shutil.copy(os.path.join(os.path.dirname(prefix0), f), os.path.join(d, f))
    with open(os.path.join(d, "ref.fa.alt"), "w") as f:
        f.write(ALT_FILE)
    prefix = os.path.join(d, "ref.fa")
    idx = pkg.capi.Index(prefix)
    opt = pkg.capi.default_opt()
    regs, ro, cells, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    assert rc == 0 and refgolden.regs_differ("opt/alt", regs, ro) == []
    assert (((regs["n_comp_is_alt"] >> 30) & 3) != 0).sum() > 1000
    eregs, ero = el.seed_chain_extend(idx, opt, codes, offs)
    assert np.array_equal(ero, ro) and eregs.tobytes() == regs.tobytes()
    idx.close()
