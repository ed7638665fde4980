"""The launch arithmetic of beast_minmax_f32 (csrc/bounds.cu) restated on the CPU, and the argument checks of the
bound entry points that return before any device work.

`minmax_launch` restates the host side of beast_minmax_f32: the column groups (4 columns on the float4 path, taken when
cols % 4 == 0 and x is 16-byte aligned, else 1), their cut into chunks of at most 1024 groups, the rows per block and
the block budget.  `owners` restates how minmax_kernel maps (chunk, thread) to columns.  Every column count 1..8192,
aligned and not, must give launches the device accepts and own every column exactly once; up to 1024 groups the launch
must be the one the kernel had before wide rows were accepted (one chunk, same grid, block and shared memory).
"""
import ctypes as C

import numpy as np
import pytest

B200_SMS = 148
MAX_THREADS = 1024
MAX_STATIC_SMEM = 48 * 1024


def minmax_launch(cols, aligned, rows, sms=B200_SMS):
    vec = 4 if cols % 4 == 0 and aligned else 1
    groups = cols // vec
    chunks = -(-groups // 1024)
    chunk_groups = -(-groups // chunks)
    rpb = max(1, 512 // chunk_groups)
    row_blocks = min(-(-rows // rpb), max(1, sms * 4 // chunks))
    return dict(vec=vec, chunks=chunks, chunk_groups=chunk_groups, rpb=rpb, row_blocks=row_blocks,
                grid=row_blocks * chunks, block=chunk_groups * rpb, smem=2 * rpb * chunk_groups * vec * 4)


def single_chunk_launch(cols, aligned, rows, sms=B200_SMS):
    """The launch of the one-chunk kernel (every column group in one block); None where it returned
    BEAST_E_UNSUPPORTED (more than 1024 groups)."""
    vec = 4 if cols % 4 == 0 and aligned else 1
    groups = cols // vec
    if groups > 1024:
        return None
    rpb = max(1, 512 // groups)
    return dict(grid=min(-(-rows // rpb), sms * 4), block=groups * rpb, smem=2 * rpb * cols * 4)


def owners(cols, launch):
    """Column index of every (chunk, group, vector lane) that reads one, as minmax_kernel computes it."""
    vec, cg = launch["vec"], launch["chunk_groups"]
    ccols = cg * vec
    out = []
    for chunk in range(launch["chunks"]):
        c0 = chunk * ccols
        ncols = min(ccols, cols - c0)
        assert ncols > 0 and ncols % vec == 0, (cols, chunk, ncols)
        g = np.arange(cg)
        g = g[g * vec < ncols]                       # groups past the end of a short last chunk read nothing
        out.append((c0 + g[:, None] * vec + np.arange(vec)[None, :]).ravel())
    return np.concatenate(out)


@pytest.mark.parametrize("aligned", [True, False])
def test_minmax_launch_covers_every_column_count(aligned):
    for cols in range(1, 8193):
        for rows in (1, 10 ** 6):
            L = minmax_launch(cols, aligned, rows)
            assert 257 <= L["block"] <= MAX_THREADS, (cols, L)            # >= 8 full warps finish the columns
            assert L["smem"] <= MAX_STATIC_SMEM and L["smem"] <= 32 * 1024, (cols, L)
            assert 1 <= L["grid"] < 2 ** 31 and L["row_blocks"] >= 1, (cols, L)
            assert L["chunks"] * L["chunk_groups"] * L["vec"] >= cols
            assert (L["chunks"] - 1) * L["chunk_groups"] * L["vec"] < cols      # no empty chunk
        own = owners(cols, L)
        assert own.size == cols and np.array_equal(np.sort(own), np.arange(cols)), cols


def test_minmax_launch_unchanged_up_to_1024_groups():
    """One chunk: the grid, block and shared memory of the single-chunk kernel, at every row count where its grid
    changes (the 4 * SMs cap) and for every column count it accepted."""
    for aligned in (True, False):
        for cols in range(1, 4097):
            old = single_chunk_launch(cols, aligned, 1)
            if old is None:
                continue
            rpb = minmax_launch(cols, aligned, 1)["rpb"]
            for rows in (1, 31, 32, 33, 511, 512, 513, (4 * B200_SMS - 1) * rpb, 4 * B200_SMS * rpb,
                         4 * B200_SMS * rpb + 1, 10 ** 6):
                new = minmax_launch(cols, aligned, rows)
                assert new["chunks"] == 1
                assert {k: new[k] for k in ("grid", "block", "smem")} == single_chunk_launch(cols, aligned, rows)
    # the shipped shape, 14 DoF x 10 basis functions
    assert minmax_launch(140, True, 10 ** 6) == dict(vec=4, chunks=1, chunk_groups=35, rpb=14, row_blocks=592,
                                                     grid=592, block=490, smem=15680)
    assert minmax_launch(140, False, 10 ** 6)["block"] == 420


def test_minmax_launch_wide_rows():
    """Column counts the single-chunk kernel refused: 14 x 75 and 30 x 35 (not a multiple of 4), 64 x 65 (over 4096),
    32 x 50 through an offset view (scalar path, 1600 groups)."""
    for cols, aligned, chunks in ((1050, True, 2), (1050, False, 2), (1600, False, 2), (4160, True, 2),
                                  (4097, True, 5), (5120, True, 2), (5120, False, 5), (8192, False, 8)):
        assert single_chunk_launch(cols, aligned, 1) is None
        L = minmax_launch(cols, aligned, 10 ** 6)
        assert L["chunks"] == chunks, (cols, aligned, L)
        assert L["grid"] <= 4 * B200_SMS                                  # the block budget is shared by the chunks
    # the largest int32 column count still gives a launchable 1-D grid
    L = minmax_launch(2 ** 31 - 1, False, 10 ** 6)
    assert L["grid"] < 2 ** 31 and L["block"] <= MAX_THREADS


def test_minmax_rows_owned_once():
    """Within a chunk, block rb and thread row rl read rows rb * rpb + rl + j * row_blocks * rpb: every row once."""
    for cols, aligned in ((1, True), (140, True), (1050, False), (5120, True)):
        for rows in (1, 33, 513, 4 * B200_SMS * 512 + 1):
            L = minmax_launch(cols, aligned, rows)
            rpb, rb = L["rpb"], L["row_blocks"]
            seen = np.zeros(rows, np.int64)
            for b in range(rb):
                for rl in range(rpb):
                    seen[b * rpb + rl::rb * rpb] += 1
            assert (seen == 1).all(), (cols, rows)


# ---------------------------------------------------------------- argument checks (no device work)
def _lib():
    from beast_tokenizer_b200 import _lib as L
    return L.load()


def test_colselect_argument_errors():
    lib = _lib()
    fake = C.c_void_p(256)          # never dereferenced: every check below returns before a launch

    def call(rows, cols, ks, nk=None, scratch=fake, x=fake, out=fake):
        arr = (C.c_int64 * max(len(ks), 1))(*ks)
        return lib.beast_colselect_f32(x, rows, cols, arr, len(ks) if nk is None else nk, out, scratch, None)

    assert call(10, 3, [0], scratch=None) == -1
    assert call(10, 3, [0], x=None) == -1
    assert call(10, 3, [0], out=None) == -1
    assert lib.beast_colselect_f32(fake, 10, 3, None, 1, fake, fake, None) == -1
    assert call(10, 3, [], nk=0) == -2
    assert call(10, 3, [0] * 9) == -2
    assert call(10, 3, [-1]) == -2
    assert call(10, 3, [10]) == -2
    assert call(10, 3, [0, 1, 2, 3, 4, 5, 6, 10]) == -2          # the last of eight out of range
    assert call(10, 65536, [0]) == -2
    assert call(0, 3, [0]) == -2
    assert call(10, 0, [0]) == -2


def test_colselect_scratch_bytes_edges():
    lib = _lib()
    f = lib.beast_colselect_scratch_bytes
    assert f(0, 0, 1) == 0 and f(0, 5, 1) == 0 and f(5, 0, 1) == 0
    assert f(-1, 5, 1) == 0 and f(5, -1, 1) == 0
    assert f(1, 1, 1) == 256 and f(64, 1, 8) == 256 and f(65, 1, 1) == 512
    assert f(2 ** 20 + 3, 1600, 2) == -(-((2 ** 20 + 3) * 1600 * 4) // 256) * 256
    assert f(2 ** 31, 65535, 1) == 2 ** 31 * 65535 * 4                   # 64-bit size, no overflow


def test_minmax_and_expand_argument_errors():
    lib = _lib()
    fake = C.c_void_p(256)
    assert lib.beast_minmax_f32(None, 1, 3, fake, fake, 1, None) == -1
    assert lib.beast_minmax_f32(fake, 1, 3, None, fake, 1, None) == -1
    assert lib.beast_minmax_f32(fake, -1, 3, fake, fake, 1, None) == -2
    assert lib.beast_minmax_f32(fake, 1, 0, fake, fake, 1, None) == -2
    assert lib.beast_minmax_f32(None, 0, 3, fake, fake, 1, None) == 0      # rows = 0 with accumulate: nothing to do
    assert lib.beast_bounds_expand_f32(fake, fake, fake, None, 3, 1e-4, None) == -1
    assert lib.beast_bounds_expand_f32(fake, fake, fake, fake, -1, 1e-4, None) == -2
    assert lib.beast_bounds_expand_f32(fake, fake, fake, fake, 0, 1e-4, None) == 0
