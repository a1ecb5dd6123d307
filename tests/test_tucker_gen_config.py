"""The configuration plan creation chooses for the run-time-rank tensor-core kernel (tucker_fit_gen_kernel), read through
nlml_debug_gen_config (no CUDA call: runs without a GPU).

Every rank set with identity / yaw / pitch rank <= 16 and roll rank <= 8 must get a configuration, and each must keep
the budgets and the tiling invariants the kernel's mbarrier rings, tensor-memory column map and shared-memory offsets
rely on.  The configurations `bench.py` measures are pinned.
"""
import ctypes
import itertools

import numpy as np
import pytest

FIELDS = ("rrmax nA KA NA16 nBC nDp BCP NB nblocks resident tslots gslots ypr_tmem tbufs gbufs ybufs "
          "col_g col_a col_t col_y smem_bytes tt_bytes gt_bytes").split()
SMEM_MAX = 232448          # 227 KB of dynamic shared memory per CTA
TMEM_COLS = 512
TILE_BYTES_MAX = 3.0e9     # tile images of the folded Gram tensor kept on the device
SAMPLES = 128              # samples per CTA = TMEM lanes


def tri(r):
    return r * (r + 1) // 2


def gen_config(lib, ranks):
    """dict of the configuration, or (error code, message)."""
    out = np.zeros(len(FIELDS), np.int32)
    rc = lib.nlml_debug_gen_config(*ranks, out.ctypes.data, len(FIELDS))
    if rc:
        return rc, lib.nlml_last_error().decode()
    return dict(zip(FIELDS, out.tolist()))


def check_invariants(ranks, c):
    ri, ry, rp, rr = ranks
    assert c["rrmax"] == (5 if rr <= 5 else 8)
    assert c["nA"] == tri(ri) and c["nBC"] == tri(ry) * tri(rp)
    assert c["nDp"] == (tri(c["rrmax"]) + 7) // 8 * 8
    # identity pairs: K of GEMM-T and N of GEMM-G, 16-deep FP16 MMAs, register accumulators of the 144-pair class
    assert c["NA16"] == c["KA"] >= c["nA"] and c["KA"] % 16 == 0 and c["NA16"] <= 144
    # blocks of the (b,c,d) axis: MMA N granularity, every (b,c) pair in exactly one block
    NB, BCP = c["NB"], c["BCP"]
    assert NB % 16 == 0 and 16 <= NB <= 256
    assert BCP >= 1 and BCP * c["nDp"] <= NB
    assert c["nblocks"] == -(-c["nBC"] // BCP)
    # tensor memory: D_G buffers, UU operand, D_T buffers, YPR operand (when it lives there), disjoint and in budget
    ranges = [(c["col_g"], c["gbufs"] * c["NA16"]), (c["col_a"], c["KA"]), (c["col_t"], c["tbufs"] * NB)]
    if c["ypr_tmem"]:
        ranges.append((c["col_y"], c["ybufs"] * NB))
    cols = c["gbufs"] * c["NA16"] + c["KA"] + c["tbufs"] * NB + c["ypr_tmem"] * c["ybufs"] * NB
    assert cols <= TMEM_COLS and max(a + n for a, n in ranges) <= TMEM_COLS
    ranges.sort()
    assert all(a0 + n0 <= a1 for (a0, n0), (a1, _) in zip(ranges, ranges[1:])), ranges
    assert all(b in (1, 2) for b in (c["tbufs"], c["gbufs"], c["ybufs"])) and c["ypr_tmem"] in (0, 1)
    # tiles: FP16 hi + lo planes; the rings (and the YPR operand when it is in shared memory) fit the CTA's budget
    assert c["tt_bytes"] == NB * c["KA"] * 4 and c["gt_bytes"] == c["NA16"] * NB * 4
    ypr_smem = 0 if c["ypr_tmem"] else c["ybufs"] * NB * SAMPLES * 4
    assert c["tslots"] * (c["tt_bytes"] + c["gt_bytes"]) + ypr_smem < c["smem_bytes"] <= SMEM_MAX
    assert c["tslots"] == c["gslots"]
    if c["resident"]:
        assert c["nblocks"] <= 16 and c["tslots"] == c["nblocks"]
    else:
        assert 1 <= c["tslots"] <= 4
    assert c["nblocks"] * (c["tt_bytes"] + c["gt_bytes"]) <= TILE_BYTES_MAX


def test_every_supported_rank_set_has_a_valid_configuration(cuda_lib):
    """All 32 768 rank sets (ri, ry, rp <= 16, rr <= 8), roll rank 1 included (it used to get none: each of its (b,c)
    pairs fills 1 of 16 columns, so every candidate scored below zero)."""
    missing = []
    for ranks in itertools.product(range(1, 17), range(1, 17), range(1, 17), range(1, 9)):
        c = gen_config(cuda_lib, ranks)
        if isinstance(c, tuple):
            missing.append((ranks, c))
            continue
        try:
            check_invariants(ranks, c)
        except AssertionError as e:
            raise AssertionError(f"ranks {ranks}: {c}") from e
    assert not missing, (len(missing), missing[:5])


def test_roll_rank_1_configurations(cuda_lib):
    """Roll rank 1 runs in the rrmax-5 instance: 1 useful column of the 16 of each (b,c) pair."""
    c = gen_config(cuda_lib, (5, 3, 3, 1))
    assert (c["rrmax"], c["KA"], c["NB"], c["nblocks"], c["resident"], c["tslots"], c["ypr_tmem"]) == (5, 16, 144, 4, 0, 3, 0)
    c = gen_config(cuda_lib, (1, 1, 1, 1))
    assert (c["rrmax"], c["KA"], c["NB"], c["nblocks"], c["resident"], c["tslots"]) == (5, 16, 16, 1, 1, 1)
    c = gen_config(cuda_lib, (2, 13, 13, 1))      # beyond the CTA-per-sample kernel's 8192 folded rows
    assert (c["rrmax"], c["NB"], c["nblocks"], c["resident"], c["tslots"]) == (5, 128, 1036, 0, 4)


# (ranks) -> the configuration bench.py measures: blocks, ring, buffers, column map and shared-memory size
PINNED = {
    (5, 3, 3, 3): dict(rrmax=5, KA=16, NB=144, BCP=9, nblocks=4, resident=0, tslots=3, ypr_tmem=0, tbufs=2, gbufs=2,
                       ybufs=2, col_g=0, col_a=32, col_t=48, col_y=336, smem_bytes=222208),
    (8, 5, 5, 5): dict(rrmax=5, KA=48, NB=128, BCP=8, nblocks=29, resident=0, tslots=4, ypr_tmem=1, tbufs=1, gbufs=1,
                       ybufs=2, col_g=0, col_a=48, col_t=96, col_y=224, smem_bytes=224768),
    (16, 8, 8, 8): dict(rrmax=8, KA=144, NB=80, BCP=2, nblocks=648, resident=0, tslots=2, ypr_tmem=1, tbufs=1, gbufs=1,
                        ybufs=1, col_g=0, col_a=144, col_t=288, col_y=368, smem_bytes=230912),
}


@pytest.mark.parametrize("ranks", list(PINNED))
def test_benchmarked_configurations_are_pinned(cuda_lib, ranks):
    c = gen_config(cuda_lib, ranks)
    assert {k: c[k] for k in PINNED[ranks]} == PINNED[ranks]


@pytest.mark.parametrize("ranks", [(2, 2, 2, 9), (1, 1, 1, 16), (17, 1, 1, 1), (1, 17, 1, 1), (1, 1, 17, 1)])
def test_unsupported_ranks_are_refused_with_the_reason(cuda_lib, ranks):
    rc, msg = gen_config(cuda_lib, ranks)
    assert rc == -3 and "roll ranks <= 8 and other ranks <= 16" in msg


def test_hook_rejects_bad_arguments(cuda_lib):
    out = np.zeros(len(FIELDS), np.int32)
    assert cuda_lib.nlml_debug_gen_config(5, 3, 3, 3, out.ctypes.data, len(FIELDS) - 1) == -1
    assert cuda_lib.nlml_debug_gen_config(0, 3, 3, 3, out.ctypes.data, len(FIELDS)) == -1
    assert cuda_lib.nlml_debug_gen_config(5, 3, 3, 3, ctypes.c_void_p(), len(FIELDS)) == -1
    assert not out.any()
