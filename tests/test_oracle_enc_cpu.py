"""The restated quant_psnr / bit / rd metrics (oracle/port/orc_enc.c) against the compiled reference: libavcodec/me_cmp.c:621-782 driven
through the table ff_me_cmp_init() fills, with the reference's own ff_dct_quantize_c / ff_convert_matrix / dct_unquantize_*_c
(oracle/refbuild/refapi_enc.c).  CPU only."""
import ctypes as C

import numpy as np
import pytest

import enc_cases


def test_quantiser_matrices_match_ff_convert_matrix(orc, refo):
    port, ref = orc, refo
    T = enc_cases.Tables(1)
    for label, st in enc_cases.states(T):
        got = [np.zeros(64, np.int32), np.zeros(64, np.int32), np.zeros(64, np.uint8)]
        want = [np.zeros(64, np.int32), np.zeros(64, np.int32), np.zeros(64, np.uint8)]
        port.enc_qmatrices(C.byref(st), *[g.ctypes.data for g in got])
        ref.enc_qmatrices(C.byref(st), *[w.ctypes.data for w in want])
        for g, w in zip(got, want):
            assert np.array_equal(g, w), label


@pytest.mark.parametrize("kind", sorted(enc_cases.KINDS))
def test_port_matches_reference(orc, refo, kind):
    port, ref = orc, refo
    T = enc_cases.Tables(2)
    n = 24
    cur, rf = enc_cases.block_pairs(n, seed=kind)
    checked = 0
    for label, st in enc_cases.states(T):
        for sidx, h in ((1, 8), (0, 16), (0, 8)):
            want, wside = enc_cases.oracle_scores(ref, kind, sidx, st, cur, rf, n, h, h263_guard=port)
            got, gside = enc_cases.oracle_scores(port, kind, sidx, st, cur, rf, n, h)
            for i in range(n):
                if want[i] is None:
                    continue
                assert got[i] == want[i] and gside[i] == wside[i], (enc_cases.KINDS[kind], label, sidx, h, i, got[i], want[i], gside[i], wside[i])
                checked += 1
    assert checked > 4000
