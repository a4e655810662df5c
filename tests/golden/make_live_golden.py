"""Generates tests/golden/live_ref.xz (read by tests/refgolden.py): the outputs of the UNMODIFIED reference that the option,
SAM, ksw_align2, bwa_gen_cigar2 and mate-rescue tests compare against, through `oracle/_ref/<isa>/ref_driver` and
`oracle/_ref/<isa>/bwa-mem2` on the inputs those tests build (C0 reads, seeded request sets, the XA / ALT genome).

Run where the reference sources are present and oracle/_ref is built:  python tests/golden/make_live_golden.py"""
import hashlib, os, struct, subprocess, sys, tempfile
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402
import cigar_util as cu, ksw_util as ku, oracle_lib as ol, refdump, refgolden  # noqa: E402
import test_option_surface_cpu as t_opt, test_oracle_sam_pe as t_pe, test_oracle_sam_se as t_se  # noqa: E402
import test_oracle_ksw as t_ksw, test_oracle_materescue as t_mate, test_cigar_cpu as t_cigar  # noqa: E402


def write_fastq(path, reads):
    with open(path, "w") as f:
        for i, r in enumerate(reads):
            f.write(f"@p{i}\n{''.join('ACGTN'[c] for c in r)}\n+\n{'I' * len(r)}\n")


def mem(prefix, fastqs, args=(), dump=None):
    """`ref_driver mem` (the reference's main_mem) -> SAM text; dump: BM2_DUMP_PREFIX of the link-time stage dumps."""
    env = dict(os.environ, **({"BM2_DUMP_PREFIX": dump} if dump else {}))
    return subprocess.run([cu.refbin(), "mem", "-t", "1", "-K", "100000000"] + list(args) + [prefix] + list(fastqs),
                          check=True, capture_output=True, env=env).stdout.decode()


def main():
    assert cu.refbin(), "oracle/_ref is not built"
    capi = load_package().capi
    out = {}
    work = tempfile.mkdtemp(prefix="bm2_live_")
    prefix = os.path.join(HERE, "c0_index", "ref.fa")
    reads = np.load(os.path.join(HERE, "c0_reads.npz"))["reads"]
    fq = [os.path.join(work, "r1.fq"), os.path.join(work, "r2.fq")]
    write_fastq(fq[0], reads[0::2]); write_fastq(fq[1], reads[1::2])

    # option surface: the regs of every option set, and of the C0 index with two ALT contigs
    for name, args in t_opt.CASES:
        mem(prefix, fq, args, dump=os.path.join(work, name))
        refgolden.put_regs(out, f"opt/{name}", *refdump.read_regs(os.path.join(work, name + ".regs.bin")))
    alt = os.path.join(work, "altidx"); os.makedirs(alt)
    for f in os.listdir(os.path.dirname(prefix)):
        os.symlink(os.path.join(os.path.dirname(prefix), f), os.path.join(alt, f))
    with open(os.path.join(alt, "ref.fa.alt"), "w") as f:
        f.write(t_opt.ALT_FILE)
    mem(os.path.join(alt, "ref.fa"), fq, dump=os.path.join(work, "alt"))
    refgolden.put_regs(out, "opt/alt", *refdump.read_regs(os.path.join(work, "alt.regs.bin")))

    # paired-end SAM with options, and the XA / ALT genome
    for name, args in t_pe.PE_CASES:
        refgolden.put_sam(out, "pe/" + name, mem(prefix, fq, args))
    xa = os.path.join(work, "xa"); os.makedirs(xa)
    t_pe.xa_dataset(xa)
    subprocess.check_call([os.path.join(os.path.dirname(cu.refbin()), "bwa-mem2"), "index", xa + "/ref.fa"],
                          stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    refgolden.put_sam(out, "pe/xa_alt", mem(xa + "/ref.fa", [xa + "/r1.fq", xa + "/r2.fq"]))

    # single-end SAM with options (the r1 file)
    for name, args in t_se.SE_CASES:
        refgolden.put_sam(out, "se/" + name, mem(prefix, fq[:1], args))

    # ksw_align2 on seeded request sets
    for seed, qlens in t_ksw.KSW_CASES:
        out[f"ksw/{seed}"] = ku.reference_ksw(ku.make_requests(np.random.default_rng(seed), 1200, qlens=qlens))

    # bwa_gen_cigar2 on 6000 requests drawn from the oracle's regions of the C0 reads
    idx = capi.Index(prefix)
    codes = reads.reshape(-1); offs = (np.arange(len(reads) + 1) * reads.shape[1]).astype(np.int64)
    reqs = t_cigar.live_requests(capi, idx, codes, offs, reads.shape[1])
    out["cigar/reqs_sha256"] = np.frombuffer(hashlib.sha256(reqs.tobytes()).hexdigest().encode(), np.uint8)
    out["cigar/recs"], out["cigar/cigar"], out["cigar/md"] = cu.reference_gen_cigar(capi, prefix, codes, offs, reqs)

    # mate rescue: mem_pestat of a default run, mem_matesw on the oracle's regs of the C0 reads (== the reference's)
    mem(prefix, fq, dump=os.path.join(work, "d"))
    pestat = open(os.path.join(work, "d.pestat.bin"), "rb").read()
    out["mate/pestat"] = np.frombuffer(pestat, np.uint8)
    regs, ro, _, rc = ol.seed_chain_extend(idx, capi.default_opt(), codes, offs)
    assert rc == 0
    pes = [struct.unpack_from("<iiidd", pestat, 4 + 28 * d) for d in range(4)]
    mate_in = t_mate.mate_input(reads, regs, ro, pes)
    with open(os.path.join(work, "mate_in.bin"), "wb") as f:
        f.write(mate_in)
    subprocess.check_call([cu.refbin(), "matesw", prefix, os.path.join(work, "mate_in.bin"), os.path.join(work, "mate_out.bin")],
                          stderr=subprocess.DEVNULL)
    out["mate/matesw_in_sha256"] = np.frombuffer(hashlib.sha256(mate_in).hexdigest().encode(), np.uint8)
    out["mate/matesw_out"] = np.fromfile(os.path.join(work, "mate_out.bin"), np.uint8)
    idx.close()

    refgolden.save(refgolden.PATH, out)
    print(len(out), "arrays,", os.path.getsize(refgolden.PATH), "bytes")


if __name__ == "__main__":
    main()
