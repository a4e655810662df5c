"""GPU parity on long reads (-x ont2d preset): seed SW filter (mem_flt_chained_seeds), extensions with 16-bit and
wide state, doubled-band retries, through the C ABI, against the oracle."""
import numpy as np
import pytest
import oracle_lib as ol
import longread_util as lu

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("coop_min", [None, "0"], ids=["default", "warp_chaining_for_every_heavy_read"])
def test_long_reads_match_oracle(pkg, coop_min, monkeypatch):
    # coop_min = 0: every read of the warp-per-read pass runs its chaining on all 32 lanes (ChainWarp: ballots for the tree scans, block shifts)
    if coop_min is not None:
        monkeypatch.setenv("BM2_CHAIN_COOP_MIN", coop_min)
    prefix, codes, offs = lu.make_dataset(n3k=10, n8k=3, ref_bp=1_000_000)
    idx = pkg.capi.Index(prefix); opt = lu.ont2d_opt(pkg.capi)
    ctx = pkg.capi.Context(0, index=idx, opt=opt)
    got, go = ctx.seed_chain_extend(codes, offs)
    want, wo, cells, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    assert rc == 0 and len(want) > 10 and np.array_equal(go, wo)
    for f in ol.REG_CMP_FIELDS + ("n_comp_is_alt",):
        assert np.array_equal(got[f], want[f]), f
    ctx.close(); idx.close()
