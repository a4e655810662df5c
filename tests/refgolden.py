"""Outputs of the UNMODIFIED reference that the tests compare against, recorded by tests/golden/make_live_golden.py into
tests/golden/live_ref.xz: one uncompressed .npz inside one xz stream, so that the many option variants of the same data
set (which differ in few lines) cost little.  Keys name the test and its case, e.g. "pe/all" or "opt/k15_w50".

SAM output is stored without its header and with SEQ and QUAL (which follow from the reads) written as "*"; the SHA-256 of
the full text from FLAG on keeps the comparison byte for byte (assert_sam_text).  Alignment regions are stored as their counts
per read and the SHA-256 of every compared field (regs_differ)."""
import hashlib, io, lzma, os
import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "live_ref.xz")
_CACHE = None


def get(key):
    global _CACHE
    if _CACHE is None:
        with open(PATH, "rb") as f:
            z = np.load(io.BytesIO(lzma.decompress(f.read())))
            _CACHE = {k: z[k] for k in z.files}
    return _CACHE[key]


def _reg_columns(regs, from_dump):
    """The fields of alignment regions that oracle_lib.regs_equal_to_dump compares, in the reference dump's types."""
    import oracle_lib as ol, refdump
    cols = {f: np.ascontiguousarray(regs[f], refdump.REG_DT[f]) for f in ol.REG_CMP_FIELDS}
    if from_dump:
        n_comp, is_alt = regs["n_comp"], regs["is_alt"] & 3
    else:
        n_comp, is_alt = (regs["n_comp_is_alt"] << 2) >> 2, (regs["n_comp_is_alt"] >> 30) & 3
    cols["n_comp"] = np.ascontiguousarray(n_comp, "<i4"); cols["is_alt"] = np.ascontiguousarray(is_alt, "<i4")
    return cols


def regs_differ(key, regs, off):
    """Our REG_DT regions against the reference's (stored by put_regs): [] when identical, else the reads whose region counts
    differ or the fields that differ."""
    want_off = get(key + "/off")
    if not np.array_equal(off, want_off):
        return ["reads with other region counts"] + list(np.nonzero(np.diff(off) != np.diff(want_off))[0][:20])
    return [f for f, v in _reg_columns(regs, False).items() if hashlib.sha256(v.tobytes()).hexdigest() != get(f"{key}/sha256/{f}").tobytes().decode()]


def sam_lines(key):
    """The reference's SAM lines of a case (header left out, SEQ and QUAL as "*")."""
    return get(key).tobytes().decode().splitlines(keepends=True)


def _after_qname(lines):
    return [ln.rstrip("\n").split("\t", 1)[1] for ln in lines if not ln.startswith("@")]


def _strip(line):
    f = line.split("\t")
    f[9] = f[10] = "*"
    return "\t".join(f)


def _digest(after_qname):
    return hashlib.sha256("\n".join(after_qname).encode()).hexdigest()


def assert_sam_text(key, got):
    """got: SAM lines from FLAG on (no newline) == the reference's, every character."""
    want = _after_qname(sam_lines(key))
    assert len(got) == len(want), (len(got), len(want))
    bad =[i for i in range(len(got)) if _strip("x\t" + got[i]) != "x\t" + want[i]]
    assert not bad, (len(bad), [(got[i], want[i]) for i in bad[:2]])
    assert _digest(got) == get(key + "/sha256").tobytes().decode(), "SEQ / QUAL differ from the reference's"


# ---- recording (tests/golden/make_live_golden.py) --------------------------------------------------------------------------------------
def put_sam(out, key, text):
    lines = [ln for ln in text.splitlines(keepends=True) if not ln.startswith("@")]
    out[key] = np.frombuffer("".join(_strip(ln.rstrip("\n")) + "\n" for ln in lines).encode(), np.uint8)
    out[key + "/sha256"] = np.frombuffer(_digest(_after_qname(lines)).encode(), np.uint8)


def put_regs(out, key, dump_regs, dump_off):
    out[key + "/off"] = dump_off
    for f, v in _reg_columns(dump_regs, True).items():
        out[f"{key}/sha256/{f}"] = np.frombuffer(hashlib.sha256(v.tobytes()).hexdigest().encode(), np.uint8)


def save(path, arrays):
    buf = io.BytesIO()
    np.savez(buf, **arrays)
    with open(path, "wb") as f:
        f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
