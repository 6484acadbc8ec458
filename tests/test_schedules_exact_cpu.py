"""Host-only checks of the exact-gradient backward's compile-time schedules (nfb_debug_schedule 5 and 6, csrc/nfb_train.cu): the
exact dX chain loads every hi and every lo half-unit of the hi/lo backward weight stream exactly once per tile, each into one ring
slot, its A operands (hi at +0, lo at +32 of a 64-column slice) stay out of the step's accumulator region, and the exact
weight-gradient kernel's stages hold both halves of both operands and load exactly twice the bytes of the FP16 kernel.  No GPU."""
import ctypes as C

import pytest

STREAM_BWD = 835584          # nfb_layout.h kBwdStreamBytes
REC_LO = 1 << 20             # kRecLo: the lo MiB of a 2 MiB exact-gradient record
SMEM_LIMIT = 232448          # 227 KB per CTA
CHAIN_PROGRAM, CHAIN_PROGRAM_EXACT, DW_JOBS, DW_STAGES_EXACT = 2, 5, 3, 6
FROM_OP, FIRST, COMMIT = 1, 8, 16


@pytest.fixture(scope="module")
def lib(built_lib):
    lb = C.CDLL(built_lib)
    lb.nfb_debug_schedule.restype = C.c_int
    lb.nfb_debug_schedule.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_uint32), C.c_int]
    return lb


def entries(lib, which):
    n = lib.nfb_debug_schedule(which, -1, None, 0)
    assert n > 0
    out = []
    buf = (C.c_uint32 * 10)()
    for i in range(n):
        w = lib.nfb_debug_schedule(which, i, buf, 10)
        assert w > 0
        out.append([int(buf[k]) for k in range(w)])
    assert lib.nfb_debug_schedule(which, n, buf, 10) == -1
    return out


def idesc_n(x):
    return ((x >> 17) & 0x3F) << 3


def test_exact_chain_reads_every_hi_and_lo_half_unit_once(lib):
    fp16 = entries(lib, CHAIN_PROGRAM)
    ents = entries(lib, CHAIN_PROGRAM_EXACT)
    assert len(ents) == 2 * len(fp16) == 56
    spans = sorted(((e[3] & 0xFFFFF) << 4, (e[3] >> 20) * 128, e[4]) for e in ents)
    pos = 0
    for off, nbytes, _ in spans:                        # the loads tile the x3 stream without gap or overlap
        assert off == pos, (off, pos)
        pos += nbytes
    assert pos == 2 * STREAM_BWD
    for k, e in enumerate(ents):
        unit = fp16[k // 2]
        assert e[4] == k % 2                            # hi load, then lo load of the same unit
        assert e[:3] == unit[:3]                        # same MMA shape, TMEM columns and flags as the FP16 program
        off, nbytes = (e[3] & 0xFFFFF) << 4, (e[3] >> 20) * 128
        unit_off = (unit[3] & 0xFFFFF) << 4
        assert nbytes == (unit[3] >> 20) * 128 and off == 2 * unit_off + e[4] * nbytes   # hi image, then its lo image
        assert nbytes <= e[7] and off % 1024 == 0       # one ring slot, swizzle-aligned
        assert idesc_n(e[0]) * 128 == nbytes
    assert sum(1 for e in ents if e[2] & COMMIT) == 2 * 9   # the commit flag rides on both loads of the last unit of each step


def test_exact_chain_fits_shared_memory(lib):
    e = entries(lib, CHAIN_PROGRAM_EXACT)[0]
    smem, slot_bytes, slots, op_buffers = e[6], e[7], e[8], e[9]
    assert op_buffers == 2 and slot_bytes == 32768 and slots >= 2
    assert smem <= SMEM_LIMIT
    assert smem >= slots * slot_bytes + op_buffers * 128 * 128


def test_exact_chain_operands_stay_out_of_the_accumulator(lib):
    for e in entries(lib, CHAIN_PROGRAM_EXACT):
        d_col, a_col, lo_col = e[1] & 0xFFFF, e[1] >> 16, e[5]
        n = idesc_n(e[0])
        acc = range(d_col, d_col + n)
        assert d_col in (0, 256) and d_col + n <= 512
        if e[2] & FROM_OP:
            assert lo_col == 0xFFFFFFFF                 # hi / lo operand from the two shared-memory buffers
            continue
        assert lo_col == a_col + 32 and a_col % 64 == 0
        for c0 in (a_col, lo_col):                      # 32 columns each (64 FP16 of K)
            assert c0 + 32 <= 512
            assert not any(c in acc for c in range(c0, c0 + 32)), (e, c0)
            assert (c0 & 256) != d_col                  # the other region


def test_exact_weight_gradient_stages(lib):
    jobs = entries(lib, DW_JOBS)
    stages = entries(lib, DW_STAGES_EXACT)
    assert len(stages) == len(jobs) == 21
    for job, st in zip(jobs, stages):
        a_hi, b_hi, a_lo, b_lo, stage_bytes, n_stages, tile_bytes, tile_bytes_fp16, smem, rec_lo = st
        b_rows = job[4]
        assert rec_lo == REC_LO
        a_bytes, b_bytes = 128 * 128, b_rows * 128     # per r-atom: A [128 features x 64 rows], B [b_rows x 64 rows]
        parts = sorted([(a_hi, a_bytes), (b_hi, 256 * 128), (a_lo, a_bytes), (b_lo, 256 * 128)])
        for (o0, n0), (o1, _) in zip(parts, parts[1:]):
            assert o0 + n0 <= o1                        # A and B, hi and lo: four disjoint buffers inside the stage
        assert parts[0][0] >= 0 and parts[-1][0] + parts[-1][1] <= stage_bytes
        assert all(o % 1024 == 0 for o, _ in parts)
        assert n_stages == 2 and stage_bytes == 2 * 49152
        assert n_stages * stage_bytes + 2048 <= smem <= SMEM_LIMIT
        today = 2 * (a_bytes + b_bytes)                 # two r-atoms per 128-row tile
        assert tile_bytes_fp16 == today
        assert tile_bytes == 2 * today
