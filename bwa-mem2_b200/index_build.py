"""index_build.py — bwa-mem2 index files built with torch (GPU when available).  TEST / BENCH TOOLING.

The hot path takes the reference's on-disk index as an input contract (SURVEY.md §8f-4); the reference's
own builder (`bwa-mem2 index`: single-threaded SA-IS, 28 N bytes of RAM, ~1-2 h for 3 Gbp) cannot run
inside a benchmark, so the 3 Gbp configurations build the SAME files here:

  <prefix>.bwt.2bit.64  int64 N | int64 count[5] | CP_OCC[(N>>6)+1] | int8 sa_ms[(N>>3)+1] |
                        uint32 sa_ls[(N>>3)+1] | int64 sentinel   (writer: reference src/FMI_search.cpp:144-302)
  <prefix>.0123         2*l_pac base codes, forward then reverse complement (src/FMI_search.cpp:325-362)
  <prefix>.pac .ann .amb                                                     (src/bntseq.cpp:73-104, :338-351)

`tests/test_index_build.py` checks byte identity with files written by the reference binary.
Suffix array: MSD bucketing on the first bases, one 31-mer radix sort per bucket, then Larsson-Sadakane
prefix doubling restricted to the still-tied groups (all torch sorts; no Python loops over suffixes).
"""
from __future__ import annotations
import os
import numpy as np
import torch

K = 31  # bases per sort key (62 bits)


def _kmer_keys(Tp: torch.Tensor, pos: torch.Tensor, k: int = K) -> torch.Tensor:
    key = torch.zeros_like(pos)
    for t in range(k):
        key = key * 4 + Tp[pos + t].to(torch.int64)
    return key


def suffix_array(T: torch.Tensor, max_bucket: int = 1 << 27, chunk: int = 1 << 28, log=None) -> torch.Tensor:
    """Suffix array of the base-code text T (uint8, values 0..3), shorter suffix first on ties ($ < A).
    Returns int64[N]."""
    dev = T.device
    N = T.numel()
    Tp = torch.cat([T, torch.zeros(K + 8, dtype=torch.uint8, device=dev)])
    b = 0
    while N / (4 ** b) > max_bucket:
        b += 1
    nb = 4 ** b
    SA = torch.empty(N, dtype=torch.int64, device=dev)
    RANK = torch.empty(N, dtype=torch.int64, device=dev)
    unresolved = []
    base = 0
    for bid in range(nb):
        if b == 0:
            pos = torch.arange(N, dtype=torch.int64, device=dev)
        else:
            parts = []
            for c0 in range(0, N, chunk):
                c1 = min(N, c0 + chunk)
                code = torch.zeros(c1 - c0, dtype=torch.int32, device=dev)
                for t in range(b):
                    code = code * 4 + Tp[c0 + t:c1 + t].to(torch.int32)
                parts.append(torch.nonzero(code == bid).squeeze(1) + c0)
                del code
            pos = torch.cat(parts)
            del parts
        n_b = pos.numel()
        if n_b == 0:
            continue
        keys = _kmer_keys(Tp, pos)
        skeys, perm = torch.sort(keys)
        del keys
        sa_b = pos[perm]
        del pos, perm
        SA[base:base + n_b] = sa_b
        is_start = torch.ones(n_b, dtype=torch.bool, device=dev)
        is_start[1:] = skeys[1:] != skeys[:-1]
        del skeys
        ar = torch.arange(n_b, dtype=torch.int64, device=dev)
        start_idx = torch.cummax(torch.where(is_start, ar, torch.zeros_like(ar)), 0).values
        RANK[sa_b] = start_idx + base
        nxt = torch.ones(n_b, dtype=torch.bool, device=dev)
        nxt[:-1] = is_start[1:]
        multi = ~(is_start & nxt)
        if bool(multi.any()):
            unresolved.append(torch.nonzero(multi).squeeze(1) + base)
        del sa_b, is_start, ar, start_idx, nxt, multi
        base += n_b
        if log and nb > 1:
            log(f"bucket {bid + 1}/{nb}")
    assert base == N
    U = torch.cat(unresolved) if unresolved else torch.empty(0, dtype=torch.int64, device=dev)
    del unresolved
    h = K
    rounds = 0
    piece = 1 << 27
    while U.numel() > 0:
        rounds += 1
        if log:
            log(f"refine round {rounds}: h={h}, unresolved={U.numel()}")
        keep_parts = []
        # pieces end at group boundaries (group = equal RANK of the suffix at that SA slot)
        u0 = 0
        nU = U.numel()
        # the second sort keys of a piece use RANK values that other pieces of the SAME round may already have
        # refined; refined ranks are consistent with the true order, so this is still correct (Larsson-Sadakane)
        while u0 < nU:
            u1 = min(nU, u0 + piece)
            if u1 < nU:
                gl = RANK[SA[U[u1 - 1]]]
                # extend to the end of the group of the last element
                ext = U[u1:min(nU, u1 + (1 << 24))]
                same = RANK[SA[ext]] == gl
                nsame = int(same.to(torch.int64).cumprod(0).sum().item())
                u1 += nsame
            Up = U[u0:u1]
            sfx = SA[Up]
            g = RANK[sfx]
            idx = sfx + h
            key2 = torch.where(idx < N, RANK[torch.clamp(idx, max=N - 1)], -(idx - N) - 1)
            p1 = torch.argsort(key2, stable=True)
            p2 = torch.argsort(g[p1], stable=True)
            perm = p1[p2]
            del p1, p2
            new_sfx = sfx[perm]
            k_s = key2[perm]
            del key2, perm, idx, sfx
            SA[Up] = new_sfx
            is_start = torch.ones(Up.numel(), dtype=torch.bool, device=dev)
            is_start[1:] = (g[1:] != g[:-1]) | (k_s[1:] != k_s[:-1])      # g is already sorted (U ascending)
            start_pos = torch.cummax(torch.where(is_start, Up, torch.zeros_like(Up)), 0).values
            RANK[new_sfx] = start_pos
            nxt = torch.ones(Up.numel(), dtype=torch.bool, device=dev)
            nxt[:-1] = is_start[1:]
            multi = ~(is_start & nxt)
            keep_parts.append(Up[multi])
            del g, k_s, new_sfx, is_start, start_pos, nxt, multi, Up
            u0 = u1
        U = torch.cat(keep_parts) if keep_parts else torch.empty(0, dtype=torch.int64, device=dev)
        h *= 2
        if rounds > 40:
            raise RuntimeError("suffix array refinement did not converge")
    del RANK
    return SA


def build_fm_arrays(T: torch.Tensor, SA: torch.Tensor, chunk_rows: int = 1 << 28):
    """-> dict(N, count[5] (file convention), cp_occ uint8 bytes, sa_ms int8, sa_ls uint32 (as int64 tensor), sentinel)."""
    dev = T.device
    n_txt = T.numel()
    N = n_txt + 1                                     # BWT rows incl. the sentinel suffix
    cnt = torch.bincount(T.to(torch.int64), minlength=4)[:4].cpu().numpy().astype(np.int64)
    count = np.zeros(5, np.int64)
    count[1:] = np.cumsum(cnt)
    n_occ = (N >> 6) + 1
    n_blocks = (N + 63) // 64
    cp = torch.zeros((n_occ, 8), dtype=torch.int64, device=dev)
    sentinel = -1
    run = torch.zeros(4, dtype=torch.int64, device=dev)
    w8 = torch.tensor([128, 64, 32, 16, 8, 4, 2, 1], dtype=torch.int64, device=dev)
    rows_per = max(64, (chunk_rows // 64) * 64)
    for r0 in range(0, n_blocks * 64, rows_per):
        r1 = min(n_blocks * 64, r0 + rows_per)
        rows = torch.arange(r0, r1, dtype=torch.int64, device=dev)
        valid = rows < N
        # full SA: row 0 -> n_txt (sentinel suffix), row i -> SA[i-1]
        p = torch.where(rows == 0, torch.full_like(rows, n_txt), SA[torch.clamp(rows - 1, 0, n_txt - 1)])
        bw = torch.where(p > 0, T[torch.clamp(p - 1, min=0)].to(torch.int64), torch.full_like(p, 4))
        bw = torch.where(valid, bw, torch.full_like(bw, 6))
        z = torch.nonzero((p == 0) & valid)
        if z.numel():
            sentinel = int(z[0, 0].item()) + r0
        blk = bw.view(-1, 64)
        nbk = blk.shape[0]
        for b in range(4):
            m = (blk == b)
            per_block = m.sum(1)
            excl = torch.cumsum(per_block, 0) - per_block + run[b]
            cp[r0 // 64:r0 // 64 + nbk, b] = excl
            run[b] = excl[-1] + per_block[-1]
            by = (m.view(nbk, 8, 8).to(torch.int64) * w8).sum(2)            # 8 bytes, MSB-first bit order
            # big-endian byte string -> little-endian uint64 value: byte 0 is the most significant
            val = torch.zeros(nbk, dtype=torch.int64, device=dev)
            for k in range(8):
                val = val | (by[:, k] << (8 * (7 - k)))
            cp[r0 // 64:r0 // 64 + nbk, 4 + b] = val
        del rows, valid, p, bw, blk
    n_sa = (N >> 3) + 1
    rows = torch.arange(0, N, 8, dtype=torch.int64, device=dev)
    v = torch.where(rows == 0, torch.full_like(rows, n_txt), SA[torch.clamp(rows - 1, 0, n_txt - 1)])
    ms = torch.zeros(n_sa, dtype=torch.int8, device=dev)
    ls = torch.zeros(n_sa, dtype=torch.int64, device=dev)
    ms[:rows.numel()] = ((v >> 32) & 0xff).to(torch.int8)
    ls[:rows.numel()] = v & 0xffffffff
    return dict(N=N, count=count, cp_occ=cp, sa_ms=ms, sa_ls=ls, sentinel=sentinel)


def write_index(prefix: str, contigs, device=None, log=None):
    """contigs: list of (name, uint8 codes 0..3 as numpy or torch) — no ambiguous bases (replace them first).
    Writes the five index files and returns the FM arrays (torch, on `device`)."""
    if device is None:
        device = "cuda" if torch.cuda.is_available() else "cpu"
    parts = [torch.as_tensor(c) for _, c in contigs]
    fwd = torch.cat(parts).to(device=device, dtype=torch.uint8)
    l_pac = fwd.numel()
    T = torch.cat([fwd, (3 - fwd).flip(0)])
    SA = suffix_array(T, log=log)
    fm = build_fm_arrays(T, SA)
    del SA
    with open(prefix + ".bwt.2bit.64", "wb") as f:
        f.write(np.array([fm["N"]], np.int64).tobytes())
        f.write(fm["count"].tobytes())
        cp = fm["cp_occ"]
        step = 1 << 24
        for i in range(0, cp.shape[0], step):
            f.write(cp[i:i + step].cpu().numpy().tobytes())
        f.write(fm["sa_ms"].cpu().numpy().tobytes())
        ls = fm["sa_ls"]
        for i in range(0, ls.numel(), 1 << 26):
            f.write(ls[i:i + (1 << 26)].cpu().numpy().astype(np.uint32).tobytes())
        f.write(np.array([fm["sentinel"]], np.int64).tobytes())
    with open(prefix + ".0123", "wb") as f:
        for i in range(0, T.numel(), 1 << 28):
            f.write(T[i:i + (1 << 28)].cpu().numpy().tobytes())
    # .pac: first base in the two top bits (src/bntseq.cpp:246), trailer bytes (:343-351)
    pad = (-l_pac) % 4
    fp = torch.cat([fwd, torch.zeros(pad, dtype=torch.uint8, device=device)]).view(-1, 4).to(torch.int32)
    packed = ((fp[:, 0] << 6) | (fp[:, 1] << 4) | (fp[:, 2] << 2) | fp[:, 3]).to(torch.uint8)
    with open(prefix + ".pac", "wb") as f:
        f.write(packed.cpu().numpy().tobytes())
        if l_pac % 4 == 0:
            f.write(b"\0")
        f.write(bytes([l_pac % 4]))
    with open(prefix + ".ann", "w") as f:
        f.write(f"{l_pac} {len(contigs)} 11\n")
        off = 0
        for name, c in contigs:
            f.write(f"0 {name} (null)\n{off} {len(c)} 0\n")
            off += len(c)
    with open(prefix + ".amb", "w") as f:
        f.write(f"{l_pac} {len(contigs)} 0\n")
    del T
    return fm


def make_big_reference(total_bp: int, seed: int = 1, n_contigs: int = 24, repeat_frac: float = 0.15, device=None):
    """Torch generator for multi-Gbp synthetic genomes: uniform random bases + planted repeat families (units of
    300..3000 bp, 4..50 copies, divergence 0..10 %, either orientation).  Returns a list of (name, codes)."""
    if device is None:
        device = "cuda" if torch.cuda.is_available() else "cpu"
    g = torch.Generator(device=device); g.manual_seed(seed)
    G = torch.randint(0, 4, (total_bp,), dtype=torch.uint8, device=device, generator=g)
    budget = int(total_bp * repeat_frac)
    for L in (300, 800, 1500, 3000):
        n_units = max(1, budget // 4 // (L * 20))
        units = torch.randint(0, 4, (n_units, L), dtype=torch.uint8, device=device, generator=g)
        copies = torch.randint(4, 50, (n_units,), device=device, generator=g)
        div = torch.tensor([0.0, 0.005, 0.02, 0.05, 0.10], device=device)[torch.randint(0, 5, (n_units,), device=device, generator=g)]
        uid = torch.repeat_interleave(torch.arange(n_units, device=device), copies)
        nc = uid.numel()
        for c0 in range(0, nc, 1 << 16):
            u = uid[c0:c0 + (1 << 16)]
            seqs = units[u].clone()
            mut = torch.rand(seqs.shape, device=device, generator=g) < div[u][:, None]
            seqs = torch.where(mut, (seqs + torch.randint(1, 4, seqs.shape, dtype=torch.uint8, device=device, generator=g)) & 3, seqs)
            rc = torch.rand(len(u), device=device, generator=g) < 0.5
            seqs = torch.where(rc[:, None], (3 - seqs).flip(1), seqs)
            pos = torch.randint(0, total_bp - L - 1, (len(u),), device=device, generator=g)
            idx = pos[:, None] + torch.arange(L, device=device)[None, :]
            # copies overlap, and a scatter with repeated indices keeps an arbitrary writer on the GPU: keep the last copy of
            # each position explicitly, so that the genome (and the bench inputs drawn from it) is the same on every run
            flat = idx.reshape(-1)
            order = torch.argsort(flat, stable=True)
            fs = flat[order]
            last = torch.ones_like(fs, dtype=torch.bool)
            last[:-1] = fs[1:] != fs[:-1]
            G[fs[last]] = seqs.reshape(-1)[order[last]]
    w = np.array([0.8 ** i for i in range(n_contigs)], dtype=np.float64)
    lens = np.maximum((w / w.sum() * total_bp).astype(np.int64), 1000)
    lens[0] += total_bp - lens.sum()
    out = []
    o = 0
    for i, l in enumerate(lens):
        out.append((f"chr{i + 1}", G[o:o + int(l)]))
        o += int(l)
    return out
