"""GPU parity: libloexec (through the C ABI) vs the CPU oracle, bit for bit.

Sizes here are ones the oracle finishes in seconds; full BASELINE.json sizes are covered in
test_gpu_fullsize.py through the streaming oracle and size-independent properties.
"""
import numpy as np
import pytest

from oracle import bsem_numpy as bn
from oracle import cport

pytestmark = pytest.mark.gpu

SEED = 20260921
TILE = 61440


def _bits(a):
    return a.view({4: np.uint32, 8: np.uint64, 1: np.uint8}[a.dtype.itemsize])


def _check_project_cast_hist(engine, table_np, col_idx, nbins, lo, hi, with_out=True, out_dtype="f32"):
    t = engine.table_from_numpy(table_np)
    k = len(col_idx)
    out = engine.table(out_dtype, t.nrows, k) if with_out else None
    counts = engine.project_cast_hist(t, col_idx, nbins, lo, hi, out=out).to_numpy()
    exp_out, exp_counts = bn.project_cast_hist(table_np, col_idx, nbins, np.broadcast_to(np.float32(lo), (k,)),
                                               np.broadcast_to(np.float32(hi), (k,)))
    assert counts.dtype == np.uint64 and counts.shape == (k, nbins)
    np.testing.assert_array_equal(counts, exp_counts)
    if with_out:
        for j in range(k):
            got = out.to_numpy(j)
            if out_dtype == "f32":
                np.testing.assert_array_equal(_bits(got), _bits(exp_out[j]))
            else:
                np.testing.assert_array_equal(_bits(got), _bits(np.ascontiguousarray(table_np[col_idx[j]])))
        out.free()
    t.free()
    return counts


@pytest.mark.parametrize("nrows", [1, 3, 4, 5, 255, 1024, 4099, TILE - 1, TILE, TILE + 1, 3 * TILE + 17])
def test_project_cast_hist_ragged_sizes(engine, nrows):
    table = bn.synth_table_f64(1, SEED, 5, 0, nrows)
    _check_project_cast_hist(engine, table, [4, 0, 2], 256, -1000.0, 1000.0)


@pytest.mark.parametrize("nbins", [1, 2, 3, 4, 5, 10, 64, 100, 255, 256])
def test_nbins(engine, nbins):
    table = bn.synth_table_f64(1, SEED + 1, 3, 1000, 200_000)
    _check_project_cast_hist(engine, table, [0, 1, 2], nbins, -1000.0, 1000.0)


@pytest.mark.parametrize("nbins", [257, 512, 1000, 4096, 16384, 16385, 40000, 57344, 57345, 65536])
def test_nbins_above_the_tile_kernel(engine, nbins):
    """More than 256 bins (the REST ``bins`` key has no 256 ceiling): the chunk kernel with 32-bit shared-memory lane slots
    (<= 16 Ki bins) or L2 counters (above), same binning arithmetic, bit-exact against the oracle; fp32 out, histogram
    only, fp64 copy, special values, per-column ranges, a constant column and a ragged row count."""
    table = bn.synth_table_f64(1, SEED + 31, 4, 1000, 333_337)
    _check_project_cast_hist(engine, table, [0, 1, 2, 3], nbins, -1000.0, 1000.0)
    _check_project_cast_hist(engine, table, [3, 0], nbins, np.array([-1000, -3.5], np.float32), np.array([7.25, 1000], np.float32),
                             with_out=False)
    _check_project_cast_hist(engine, table, [2], nbins, -1e30, 1e30, out_dtype="f64")
    const = bn.synth_table_f64(2, SEED, 2, 0, 70_001)
    c = _check_project_cast_hist(engine, const, [0, 1], nbins, -1000.0, 1000.0)
    assert c[0].max() >= 70_001 - 100


def test_nbins_above_the_tile_kernel_unaligned_and_host(engine):
    nrows, ncols, nbins = 100_003, 3, 1000
    table = bn.synth_table_f64(1, SEED, ncols, 0, nrows)
    big = engine.table("f64", (nrows + 1) * ncols + 8, 1)
    flat = np.zeros((nrows + 1) * ncols + 8)
    for c in range(ncols):
        flat[1 + c * (nrows + 1): 1 + c * (nrows + 1) + nrows] = table[c]
    big.upload(0, flat)
    view = engine.wrap("f64", nrows, ncols, big.base_ptr + 8, (nrows + 1) * 8)
    out = engine.table("f32", nrows, ncols)
    counts = engine.project_cast_hist(view, [2, 0, 1], nbins, -1000.0, 1000.0, out=out).to_numpy()
    exp_out, exp_counts = bn.project_cast_hist(table, [2, 0, 1], nbins, [-1000.0] * 3, [1000.0] * 3)
    np.testing.assert_array_equal(counts, exp_counts)
    for j in range(3):
        np.testing.assert_array_equal(_bits(out.to_numpy(j)), _bits(exp_out[j]))
    view.free(); out.free(); big.free()
    outs = [np.empty(nrows, dtype=np.float32) for _ in range(ncols)]
    lo = np.full(ncols, -1000, np.float32); hi = np.full(ncols, 1000, np.float32)
    hc, _ = engine.project_cast_hist_host([table[j] for j in range(ncols)], 5000, lo, hi, out=outs)
    exp_out, exp_counts = bn.project_cast_hist(table, range(ncols), 5000, lo, hi)
    np.testing.assert_array_equal(hc, exp_counts)
    for j in range(ncols):
        np.testing.assert_array_equal(_bits(outs[j]), _bits(exp_out[j]))


def test_special_values_and_per_column_ranges(engine):
    nrows = 300_000
    table = bn.synth_table_f64(1, SEED + 2, 8, 0, nrows)
    lo = np.array([-1000, -500, 0, -1, -1e30, 1, -0.0, 999], dtype=np.float32)
    hi = np.array([1000, 500, 1000, 1, 1e30, 2, 1e-38, 1000], dtype=np.float32)
    c = _check_project_cast_hist(engine, table, list(range(8)), 256, lo, hi)
    assert c.sum() > 0


def test_constant_column_contention(engine):
    table = bn.synth_table_f64(2, SEED, 4, 0, 500_000)
    c = _check_project_cast_hist(engine, table, [0, 1, 0, 3], 256, -1000.0, 1000.0)
    assert c[0].max() >= 500_000 - 600      # one hot bin (minus the special-value rows)


def test_histogram_only_and_f64_copy(engine):
    table = bn.synth_table_f64(1, SEED + 3, 6, 77, 150_001)
    _check_project_cast_hist(engine, table, [5, 1], 10, -1000.0, 1000.0, with_out=False)
    _check_project_cast_hist(engine, table, [5, 1, 3], 16, -250.0, 750.0, out_dtype="f64")


def test_projection_cast_only_matches_c_oracle(engine):
    nrows = 1_000_003
    table = bn.synth_table_f64(1, SEED, 16, 0, nrows)
    perm = [3, 15, 0, 7, 7, 12]
    t = engine.table_from_numpy(table)
    out = engine.project_cast(t, perm)
    for j, c in enumerate(perm):
        exp = cport.cast_f64_f32(table[c])
        np.testing.assert_array_equal(_bits(out.to_numpy(j)), _bits(exp))
        assert out.checksum(j, 5) == cport.checksum(exp, 5) == bn.checksum(exp, 5)
    out.free(); t.free()


def test_known_answer_casts(engine):
    # SURVEY.md §8c known answers for fp64 -> fp32 RNE
    x = np.array([0.1, 16777217.0, 1e39, -1e-46, 3.4028235677973366e38, 1e-40, -0.0, np.nan, 1 + 2.0 ** -24],
                 dtype=np.float64)
    want = np.array([0x3DCCCCCD, 0x4B800000, 0x7F800000, 0x80000000, 0x7F800000, 0x000116C2, 0x80000000, 0x7FC00000,
                     0x3F800000], dtype=np.uint32)
    t = engine.table_from_numpy(x[None, :])
    out = engine.project_cast(t, [0])
    np.testing.assert_array_equal(_bits(out.to_numpy(0)), want)
    out.free(); t.free()


def test_counts_accumulate_over_row_shards(engine):
    # linearity: histogram of the whole == sum of histograms of row shards accumulated in one buffer
    nrows = 400_000
    table = bn.synth_table_f64(1, SEED + 4, 4, 0, nrows)
    whole = _check_project_cast_hist(engine, table, [0, 1, 2, 3], 256, -1000.0, 1000.0, with_out=False)
    acc = engine.counts(4, 256)
    for r0, r1 in [(0, 100_001), (100_001, 100_002), (100_002, 399_999), (399_999, nrows)]:
        t = engine.table_from_numpy(table[:, r0:r1])
        engine.project_cast_hist(t, [0, 1, 2, 3], 256, -1000.0, 1000.0, counts=acc)
        t.free()
    np.testing.assert_array_equal(acc.to_numpy(), whole)
    acc.free()


def test_device_generator_matches_oracle(engine):
    for kind in (0, 1, 2):
        t = engine.table("f64", 70_001, 5).fill_synthetic(kind, SEED, row_offset=123_456_789)
        for c in range(5):
            exp = cport.synth_f64(kind, SEED, c, 123_456_789, 70_001)
            np.testing.assert_array_equal(_bits(t.to_numpy(c)), _bits(exp))
        t.free()
    t = engine.table("u8", 100_003, 150).fill_synthetic(3, SEED, row_offset=99)
    for c in (0, 4 * 28 + 4, 39, 149):
        np.testing.assert_array_equal(t.to_numpy(c), cport.synth_u8(SEED, c, 99, 100_003))
    t.free()


@pytest.mark.parametrize("nrows", [1, 15, 16, 17, 4097, TILE - 3, TILE, 2 * TILE + 5])
def test_hist_u8_cols(engine, nrows):
    ncols = 784 if nrows <= 4097 else 150
    table = bn.synth_table_u8(SEED, ncols, 0, nrows)
    t = engine.table_from_numpy(table)
    cols = list(range(ncols))[::-1]
    got = engine.hist_u8_cols(t, cols).to_numpy()
    np.testing.assert_array_equal(got, bn.hist_u8_cols(table, cols))
    assert (got.sum(axis=1) == nrows).all()
    t.free()


def test_hist_u8_all_values_and_constant(engine):
    rng = np.random.default_rng(5)
    table = np.stack([rng.integers(0, 256, 300_000, dtype=np.uint8), np.full(300_000, 255, np.uint8),
                      np.arange(300_000, dtype=np.uint64).astype(np.uint8)])
    t = engine.table_from_numpy(table)
    got = engine.hist_u8_cols(t, [0, 1, 2]).to_numpy()
    np.testing.assert_array_equal(got, cport.hist_u8_cols(list(table)))
    t.free()


@pytest.mark.parametrize("mode", ["2", "4", "5", "6", "7", "8", "9", "10", "11", "12", "13", "14"])
def test_hist_u8_every_kernel_variant(engine, monkeypatch, mode):
    """Every selectable form of the byte-histogram kernel (LOEXEC_U8_MODE; 8 = the 512-thread shared-histogram kernel
    with its own tile size) gives the oracle's counts: ragged sizes, full tiles, constant columns, every byte value."""
    monkeypatch.setenv("LOEXEC_U8_MODE", mode)
    wide_tile = 512 * 7 * 16 if mode != "9" else 1024 * 3 * 16
    rng = np.random.default_rng(int(mode))
    for nrows in (1, 17, 4097, TILE, TILE + 1, wide_tile, 2 * wide_tile + 777, 3 * TILE + 5):
        table = np.stack([rng.integers(0, 256, nrows, dtype=np.uint8), np.full(nrows, 0, np.uint8), np.full(nrows, 200, np.uint8),
                          np.arange(nrows, dtype=np.uint64).astype(np.uint8), bn.synth_u8(SEED, 300, 0, nrows),
                          np.where(np.arange(nrows) < nrows // 2, 7, 9).astype(np.uint8)])
        t = engine.table_from_numpy(table)
        got = engine.hist_u8_cols(t, range(6)).to_numpy()
        np.testing.assert_array_equal(got, bn.hist_u8_cols(table, range(6)), err_msg=f"mode {mode} nrows {nrows}")
        t.free()


def test_unaligned_wrapped_tables(engine):
    # foreign device memory with an odd element offset / pitch takes the scalar kernel variant
    nrows, ncols = 100_003, 3
    table = bn.synth_table_f64(1, SEED, ncols, 0, nrows)
    big = engine.table("f64", (nrows + 1) * ncols + 8, 1)
    flat = np.zeros((nrows + 1) * ncols + 8)
    for c in range(ncols):
        flat[1 + c * (nrows + 1): 1 + c * (nrows + 1) + nrows] = table[c]
    big.upload(0, flat)
    view = engine.wrap("f64", nrows, ncols, big.base_ptr + 8, (nrows + 1) * 8)
    out = engine.table("f32", nrows, ncols)
    counts = engine.project_cast_hist(view, [2, 0, 1], 256, -1000.0, 1000.0, out=out).to_numpy()
    exp_out, exp_counts = bn.project_cast_hist(table, [2, 0, 1], 256, [-1000.0] * 3, [1000.0] * 3)
    np.testing.assert_array_equal(counts, exp_counts)
    for j in range(3):
        np.testing.assert_array_equal(_bits(out.to_numpy(j)), _bits(exp_out[j]))
    view.free(); out.free(); big.free()


def test_host_buffer_entry_points(engine):
    nrows, k = 1_500_007, 6
    table = bn.synth_table_f64(1, SEED + 9, k, 0, nrows)
    cols = [np.ascontiguousarray(table[j]) for j in range(k)]
    outs = [np.empty(nrows, dtype=np.float32) for _ in range(k)]
    lo = np.linspace(-1000, -900, k).astype(np.float32)
    hi = np.linspace(900, 1000, k).astype(np.float32)
    counts, timing = engine.project_cast_hist_host(cols, 256, lo, hi, out=outs)
    exp_out, exp_counts = bn.project_cast_hist(table, range(k), 256, lo, hi)
    np.testing.assert_array_equal(counts, exp_counts)
    for j in range(k):
        np.testing.assert_array_equal(_bits(outs[j]), _bits(exp_out[j]))
    assert timing["h2d_bytes"] == nrows * k * 8 and timing["launches"] >= 1
    # pinned buffers, histogram only
    pin = engine.pinned_empty((k, nrows), np.float64)
    pin[:] = table
    counts2, _ = engine.project_cast_hist_host([pin[j] for j in range(k)], 256, lo, hi)
    np.testing.assert_array_equal(counts2, exp_counts)
    # bytes
    tb = bn.synth_table_u8(SEED, 30, 0, 200_001)
    c8, _ = engine.hist_u8_cols_host([np.ascontiguousarray(tb[j]) for j in range(30)])
    np.testing.assert_array_equal(c8, bn.hist_u8_cols(tb, range(30)))


def test_host_columns_in_every_memory_arrangement(engine):
    """The host pipeline moves runs of equally strided columns as one 2-D copy and everything else column by column:
    rows of one matrix (in order, every other row, reversed), separately allocated arrays and a mix must all give the
    oracle's answer, inputs and outputs alike."""
    nrows, k = 700_003, 8
    table = bn.synth_table_f64(1, SEED + 21, k, 0, nrows)
    lo = np.full(k, -1000, np.float32); hi = np.full(k, 1000, np.float32)
    exp_out, exp_counts = bn.project_cast_hist(table, range(k), 64, lo, hi)
    wide = np.zeros((2 * k, nrows + 5), dtype=np.float64)          # row stride != nrows * 8; every other row used
    wide[::2, :nrows] = table
    out_mat = np.empty((k, nrows), dtype=np.float32)
    arrangements = {
        "matrix rows": ([table[j] for j in range(k)], [out_mat[j] for j in range(k)]),
        "every other row of a wider matrix": ([wide[2 * j, :nrows] for j in range(k)], [np.empty(nrows, np.float32) for _ in range(k)]),
        "separate arrays": ([table[j].copy() for j in range(k)], [out_mat[k - 1 - j] for j in range(k)]),      # outputs reversed
        "mixed": ([table[0], table[1], table[2].copy(), table[3], wide[8, :nrows], wide[10, :nrows], table[6], table[7].copy()],
                  [np.empty(nrows, np.float32) if j % 3 == 0 else out_mat[j] for j in range(k)]),
    }
    for name, (cols, outs) in arrangements.items():
        counts, timing = engine.project_cast_hist_host(cols, 64, lo, hi, out=outs)
        np.testing.assert_array_equal(counts, exp_counts, err_msg=name)
        for j in range(k):
            np.testing.assert_array_equal(_bits(outs[j]), _bits(exp_out[j]), err_msg=f"{name}, column {j}")
        assert timing["h2d_bytes"] == nrows * k * 8
    rev, _ = engine.project_cast_hist_host([table[k - 1 - j] for j in range(k)], 64, lo, hi)       # negative stride
    np.testing.assert_array_equal(rev, exp_counts[::-1])
    tb = bn.synth_table_u8(SEED, 40, 0, 300_001)                    # bytes: 40 columns of one matrix, then scattered
    want = bn.hist_u8_cols(tb, range(40))
    np.testing.assert_array_equal(engine.hist_u8_cols_host([tb[j] for j in range(40)])[0], want)
    np.testing.assert_array_equal(engine.hist_u8_cols_host([tb[j].copy() if j % 5 == 0 else tb[j] for j in range(40)])[0], want)


def test_error_reporting(engine):
    from learningorchestra_b200._native import LoexecError, LO_ERR_INVALID
    t = engine.table("f64", 100, 2)
    with pytest.raises(LoexecError) as e:
        engine.project_cast_hist(t, [0, 2], 256, -1.0, 1.0)
    assert e.value.code == LO_ERR_INVALID and "col_idx" in e.value.message
    with pytest.raises(LoexecError):
        engine.project_cast_hist(t, [0], 65537, -1.0, 1.0)
    with pytest.raises(LoexecError):
        engine.project_cast_hist(t, [0], 10, 1.0, 1.0)
    with pytest.raises(LoexecError):
        engine.hist_u8_cols(t, [0])
    t.free()


@pytest.mark.parametrize("lo,hi,nbins", [
    (-1000.0, 1000.0, 256), (-1000.0, 1000.0, 10), (0.0, 1.0, 256), (0.0, 255.0, 255), (-3.0, 7.0, 3),
    (1e-30, 2e-30, 100), (-1e30, 1e30, 256), (0.1, 0.7, 7), (-123.456, 789.012, 177), (5.0, 5.000001, 2),
    (0.0, 512.0, 256), (-1.0, 80.0, 10),
])
def test_fast_divide_is_ieee_divide_exhaustively(engine, lo, hi, nbins):
    """All 2^32 fp32 bit patterns: the branch-free divide of the fast kernels bins exactly like __fdiv_rn."""
    used, bad = engine.selftest_fastdiv(lo, hi, nbins)
    if used:
        assert bad == 0


def test_unsafe_divisors_take_the_ieee_kernel(engine):
    # w with an all-ones significand (Markstein's exception) and w outside the safe exponent window
    w_bad = np.float32(np.uint32(0x3FFFFFFF).view(np.float32))          # 1.9999999
    for lo, hi, nbins in [(0.0, float(w_bad * np.float32(4)), 4), (0.0, 1e-37, 8), (-1e38, 1e38, 2)]:
        used, _ = engine.selftest_fastdiv(lo, hi, nbins)
        assert not used
        rng = np.random.default_rng(3)
        x = rng.uniform(lo, hi, 200_000)
        x[::7] = hi; x[::11] = lo
        t = engine.table_from_numpy(x[None, :])
        got = engine.project_cast_hist(t, [0], nbins, lo, hi).to_numpy()
        _, exp = bn.project_cast_hist(x[None, :], [0], nbins, [lo], [hi])
        np.testing.assert_array_equal(got, exp)
        t.free()


def test_empty_inputs(engine):
    t = engine.table("f64", 0, 3)
    out = engine.table("f32", 0, 3)
    c = engine.project_cast_hist(t, [0, 1, 2], 16, -1.0, 1.0, out=out).to_numpy()
    assert c.sum() == 0
    counts, timing = engine.project_cast_hist_host([np.empty(0), np.empty(0)], 8, -1.0, 1.0, out=[np.empty(0, np.float32)] * 2)
    assert counts.shape == (2, 8) and counts.sum() == 0 and timing["launches"] == 0
    c8, _ = engine.hist_u8_cols_host([np.empty(0, np.uint8)])
    assert c8.sum() == 0
    vals, st = engine.parse_number_host([])
    assert vals.shape == (0,) and st.shape == (0,)
    k, n = engine.value_counts_f64_host(np.empty(0))
    assert k.size == 0 and n.size == 0
    t.free(); out.free()


def test_concurrent_callers_share_one_engine(engine):
    """The C ABI is documented re-entrant: four Python threads (ctypes drops the GIL) hammer one context."""
    import threading
    errors = []

    def work(seed):
        try:
            table = bn.synth_table_f64(1, SEED + seed, 3, seed * 1000, 150_000 + seed)
            _, exp = bn.project_cast_hist(table, [2, 0], 64, [-1000.0] * 2, [1000.0] * 2)
            for _ in range(5):
                t = engine.table_from_numpy(table)
                got = engine.project_cast_hist(t, [2, 0], 64, -1000.0, 1000.0).to_numpy()
                np.testing.assert_array_equal(got, exp)
                t.free()
                cols = [np.ascontiguousarray(table[2]), np.ascontiguousarray(table[0])]
                got_h, _ = engine.project_cast_hist_host(cols, 64, -1000.0, 1000.0)
                np.testing.assert_array_equal(got_h, exp)
        except Exception as exc:      # noqa: BLE001
            errors.append(exc)

    threads = [threading.Thread(target=work, args=(s,)) for s in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors


def test_plain_c_consumer_runs_the_hot_path(engine):
    import subprocess
    from test_abi_cpu import _build_c_consumer
    out = subprocess.run([str(_build_c_consumer())], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "abi_smoke ok" in out.stdout, out.stderr


def test_tma_staged_variant_has_the_same_results(engine):
    """LOEXEC_TMA=1 routes full tiles through the cp.async.bulk + mbarrier ring kernel (DESIGN.md §3.8); the switch
    is read once per process, so the parity subset is re-run in a child process with it set."""
    import os
    import subprocess
    import sys
    env = dict(os.environ, LOEXEC_TMA="1")
    out = subprocess.run([sys.executable, "-m", "pytest", __file__, "-m", "gpu", "-q", "-x", "-k",
                          "ragged_sizes or test_nbins or special_values or constant_column or histogram_only or "
                          "projection_cast_only or accumulate or host_buffer"],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert " passed" in out.stdout


def test_more_projected_columns_than_one_launch_holds(engine):
    """k > 128 (f64) and k > 1024 (u8) are split over several launches; counts / outputs line up per column."""
    table = bn.synth_table_f64(1, SEED + 21, 7, 0, 70_000)
    cols = [(3 * j + 1) % 7 for j in range(300)]
    lo = np.linspace(-1000, -900, 300).astype(np.float32)
    hi = np.linspace(900, 1000, 300).astype(np.float32)
    t = engine.table_from_numpy(table)
    out = engine.table("f32", 70_000, 300)
    got = engine.project_cast_hist(t, cols, 100, lo, hi, out=out).to_numpy()
    exp_out, exp = bn.project_cast_hist(table, cols, 100, lo, hi)
    np.testing.assert_array_equal(got, exp)
    for j in (0, 127, 128, 129, 255, 256, 299):
        np.testing.assert_array_equal(_bits(out.to_numpy(j)), _bits(exp_out[j]))
    out.free(); t.free()
    tb = bn.synth_table_u8(SEED, 1300, 0, 5000)
    t8 = engine.table_from_numpy(tb)
    idx = list(range(1300)) + [5, 700]
    got8 = engine.hist_u8_cols(t8, idx).to_numpy()
    np.testing.assert_array_equal(got8, bn.hist_u8_cols(tb, idx))
    t8.free()


def test_bench_dumps_the_last_timed_steps_outputs(built, tmp_path):
    """``bench.py --dump-outputs``: the merged counts and the sampled fp32 output rows of the last timed step equal the
    oracle's, and ``--steps`` is the number of timed launches."""
    import json
    import subprocess
    import sys
    from pathlib import Path
    rows, ncols = 300_007, 32
    bench = Path(__file__).resolve().parent.parent / "bench.py"
    res = subprocess.run([sys.executable, str(bench), "--rows", str(rows), "--steps", "7", "--warmup", "1", "--no-e2e",
                          "--no-cpu", "--executor-rows", "0", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == 7 and line["gpu_launches"] == 7
    counts = np.load(tmp_path / "counts.npy")
    sample = np.load(tmp_path / "out_f32_sample.npy")
    assert counts.dtype == np.float64 and sample.dtype == np.float32 and sample.shape[0] == ncols
    assert counts.nbytes + sample.nbytes <= 64 * 10 ** 6
    cols = [(7 * j + 3) % ncols for j in range(ncols)]
    lo, hi = np.full(ncols, -1000.0, np.float32), np.full(ncols, 1000.0, np.float32)
    exp_counts, _ = cport.synth_project_cast_hist(0, SEED, 0, rows, -1000.0, 1000.0, cols, 256, lo, hi)
    np.testing.assert_array_equal(counts, exp_counts.astype(np.float64))
    picked = np.sort(np.random.default_rng(SEED).choice(rows, size=sample.shape[1], replace=False))
    for j, c in enumerate(cols):
        exp = cport.cast_f64_f32(cport.synth_f64(0, SEED, c, 0, rows))[picked]
        np.testing.assert_array_equal(_bits(sample[j]), _bits(exp))
