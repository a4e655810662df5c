"""Shared helper: a small long-read (-x ont2d) data set, index written by bwa_mem2_b200.index_build (the reference's file format)."""
import os, tempfile, importlib
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def ont2d_opt(capi):
    """mem_opt_t after `-x ont2d` (reference src/fastmap.cpp:812-826) + bwa_fill_scmat."""
    o = capi.default_opt()
    o.o_del = o.o_ins = 1; o.e_del = o.e_ins = 1; o.b = 1; o.split_factor = 10.0
    o.min_chain_weight = 20; o.min_seed_len = 14; o.pen_clip5 = o.pen_clip3 = 0
    k = 0
    for i in range(4):
        for j in range(4):
            o.mat[k] = o.a if i == j else -o.b; k += 1
        o.mat[k] = -1; k += 1
    for j in range(5):
        o.mat[k] = -1; k += 1
    return o


def make_dataset(n3k=10, n8k=3, ref_bp=1_000_000):
    synth = importlib.import_module("bwa_mem2_b200.synth")
    index_build = importlib.import_module("bwa_mem2_b200.index_build")
    work = tempfile.mkdtemp(prefix="bm2_long_")
    ctg = synth.make_reference(ref_bp, seed=9, n_contigs=3)
    synth.write_fasta(work + "/ref.fa", ctg)
    rng = np.random.default_rng(10)               # N runs become random bases in the index, as `bwa-mem2 index` does
    index_build.write_index(work + "/ref.fa", [(n, np.where(c > 3, rng.integers(0, 4, len(c), dtype=np.uint8), c)) for n, c in ctg], device="cpu")
    reads = synth.make_long_reads(ctg, n3k, read_len=3000, seed=4) + synth.make_long_reads(ctg, n8k, read_len=8000, seed=5)
    reads.append(reads[0][:500])          # a short read in the same batch: below the mem_flt_chained_seeds threshold
    codes = np.concatenate(reads); offs = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.int64)
    return work + "/ref.fa", codes, offs
