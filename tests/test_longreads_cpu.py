"""Long reads (-x ont2d: mem_flt_chained_seeds with the seed local SW, 16-bit / wide-band extensions): the device
logic compiled for the host must equal the oracle (which is pinned to the reference on long reads, see DESIGN.md)."""
import numpy as np
import oracle_lib as ol
import emul_lib as el
import longread_util as lu


def test_long_read_logic_matches_oracle(pkg):
    prefix, codes, offs = lu.make_dataset(n3k=4, n8k=1, ref_bp=500_000)
    idx = pkg.capi.Index(prefix); opt = lu.ont2d_opt(pkg.capi)
    want, wo, cells, rc = ol.seed_chain_extend(idx, opt, codes, offs)
    got, go = el.seed_chain_extend(idx, opt, codes, offs)
    assert rc == 0 and len(want) > 5 and np.array_equal(go, wo)
    assert got.tobytes() == want.tobytes()
    idx.close()
