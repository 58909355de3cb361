"""CPU model of how the fused head's epilogue (csrc/ppn_head.cu, head_epilogue) cuts the channels of a cell tile.

The epilogue never sees a limb window whole: every channel tile (acc_n columns) is cut into one run of whole 8-column
groups per sub-warp, a run crosses windows, and each stretch of one window inside a run is a piece that publishes its
own (sigmoid, position) key.  The arg-max map is right only if the pieces of every window cover its S positions
exactly once, if every piece knows its window and the position it starts at, and if the walk ends.  That is plain
integer bookkeeping, so it is restated here line by line and checked over far more geometries than a GPU run could
take — including the 1 x 1 window, where a window-index division without an identity case never leaves the second
limb column, and the large windows where a 32-bit magic division is inexact.
"""
import numpy as np
import pytest


# ---- the kernel's window-index division (HeadArgs::magic_S, fill_common and begin() in ppn_head.cu) --------------
def magic_S(S):
    return ((1 << 40) + S - 1) // S                         # fill_common: a.magic_S


def window_index(p, magic):
    return (p * magic) >> 40                                  # begin(): ei = (p * magic_S) >> 40


# the formula it replaced: ceil(2^32 / S), 0 for S = 1, >> 32 (kept to show that the checks below have teeth)
def magic_S_32(S):
    return 0 if S <= 1 else ((1 << 32) + S - 1) // S


def window_index_32(p, magic):
    return (p * magic) >> 32


KERNEL_DIV = (magic_S, window_index)
OLD_DIV = (magic_S_32, window_index_32)


# ---- plan_items (ppn_head.cu, host side) and head_item (device side) ------------------------------------------------
def plan_items(n_tiles, n_ntiles, sms):
    chunks = 1
    if n_tiles < sms:
        chunks = min(n_ntiles, max(1, sms // n_tiles))
    chunk_tiles = (n_ntiles + chunks - 1) // chunks
    n_chunks = (n_ntiles + chunk_tiles - 1) // chunk_tiles
    return chunk_tiles, n_chunks, n_tiles * n_chunks


def head_item(item, n_chunks, chunk_tiles, n_ntiles):
    tile = item // n_chunks
    nt0 = (item - tile * n_chunks) * chunk_tiles
    return tile, nt0, min(nt0 + chunk_tiles, n_ntiles)


class Stuck(Exception):
    pass


def walk_run(n_dec, S, C, r_lo, r_hi, emit, div, decode, pieces):
    """One sub-warp's run [r_lo, r_hi) of one channel tile: head_epilogue from `begin(r_lo)` to the end of the
    `while (c0 < r_hi)` loop.  Appends each decode stretch (c_lo, c_hi) to `decode` and each published piece
    (ei, wbase, positions scanned in order) to `pieces`."""
    make_magic, index = div
    magic = make_magic(S)
    st = {}
    scanned = []                                              # window positions the current piece has scanned

    def begin(c):                                             # the `begin` lambda
        if c < n_dec:
            st.update(limb=False, seg_end=min(n_dec, r_hi))
            return
        p = c - n_dec
        ei = index(p, magic)
        aw = p - ei * S
        st.update(limb=True, ei=ei, wbase=c - aw, seg_end=min(c - aw + S, r_hi), idx=aw)
        scanned.clear()

    def scan(c0, j_lo, j_hi):                                 # spec_scan / limb_column / decode_group on [j_lo, j_hi)
        if j_hi <= j_lo:
            return
        if st["limb"]:
            aw0 = c0 - st["wbase"]
            scanned.append((aw0 + j_lo, aw0 + j_hi))
        else:
            decode.append((c0 + j_lo, c0 + j_hi))

    def publish():                                            # publish_piece: (ei, the position the piece started at)
        pieces.append((st["ei"], st["wbase"], st["idx"], list(scanned)))

    budget = 4 * (r_hi - r_lo) + 16                           # every pass below scans at least one column when all is well
    begin(r_lo)
    c0 = r_lo
    while c0 < r_hi:                                          # :398
        budget -= 1
        if budget < 0:
            raise Stuck(c0)
        if st["limb"] and not emit and c0 + 8 <= st["seg_end"]:
            while True:                                       # the hot loop, :405-410
                scan(c0, 0, 8)
                c0 += 8
                if not c0 + 8 <= st["seg_end"]:
                    break
            if c0 == st["seg_end"]:                           # :411-414
                publish()
                if st["seg_end"] < r_hi:
                    begin(st["seg_end"])
            continue
        j_lo = 0                                              # the generic group, :419-447
        while True:
            budget -= 1
            if budget < 0:
                raise Stuck(c0)
            j_hi = min(8, st["seg_end"] - c0)
            scan(c0, j_lo, j_hi)
            j_lo = j_hi
            if c0 + j_hi == st["seg_end"]:
                if st["limb"]:
                    publish()
                if st["seg_end"] < r_hi:
                    begin(st["seg_end"])
            if not (j_lo < 8 and c0 + j_lo < r_hi):
                break
        c0 += 8


def walk_tile(K, E, S, acc_n, subs, emit=False, div=KERNEL_DIV):
    """Every channel tile of one cell tile, every sub-warp's run (:263-269) -> (decode stretches, pieces)."""
    n_dec = 6 * K
    C = n_dec + S * E
    decode, pieces = [], []
    for nt in range((C + acc_n - 1) // acc_n):
        c_tile = nt * acc_n
        n_cols = min(acc_n, C - c_tile)
        n8 = (n_cols + 7) >> 3
        per = (n8 + subs - 1) // subs
        for sub in range(subs):
            r_lo = c_tile + min(sub * per, n8) * 8
            r_hi = min(c_tile + min((sub + 1) * per, n8) * 8, c_tile + n_cols)
            if r_lo < r_hi:
                walk_run(n_dec, S, C, r_lo, r_hi, emit, div, decode, pieces)
    return decode, pieces


def coverage_errors(K, E, S, acc_n, subs, emit=False, div=KERNEL_DIV):
    """None when the walk ends and its pieces tile every window exactly once, else what went wrong."""
    n_dec = 6 * K
    try:
        decode, pieces = walk_tile(K, E, S, acc_n, subs, emit, div)
    except Stuck as e:
        return f"walk stuck at column {e.args[0]}"
    cols = sorted(decode)
    at = 0
    for lo, hi in cols:
        if lo != at:
            return f"decode channels: gap or overlap at {at}"
        at = hi
    if at != n_dec:
        return f"decode channels end at {at}, want {n_dec}"
    by_window = {}
    for ei, wbase, start, scanned in pieces:
        if not 0 <= ei < E or wbase != n_dec + ei * S:
            return f"piece of window {ei} based at channel {wbase}"
        if not scanned or scanned[0][0] != start:
            return f"window {ei}: piece starts at {start} but scans {scanned[:1]}"
        for (a, b), (c, _) in zip(scanned, scanned[1:]):
            if b != c:
                return f"window {ei}: piece scans {scanned}, not one stretch"
        by_window.setdefault(ei, []).append((scanned[0][0], scanned[-1][1]))
    if sorted(by_window) != list(range(E)):
        return f"pieces for windows {sorted(by_window)[:8]}..., want 0..{E - 1}"
    for ei, spans in by_window.items():
        at = 0
        for lo, hi in sorted(spans):
            if lo != at:
                return f"window {ei}: positions {at}.. covered {'twice' if lo < at else 'never'}"
            at = hi
        if at != S:
            return f"window {ei}: pieces end at {at}, want {S}"
    return None


# ---------------------------------------------------------------------------------------------------------------
SMALL_S = [1, 2, 3, 9, 15, 25]
PRESET_S = [49, 81, 121, 441]
# K: 6K on both sides of 128 (K = 21, 22) and 256 (K = 42, 43), where the decode planes cross an accumulator tile
K_AT_EDGES = [1, 2, 5, 16, 18, 21, 22, 42, 43, 44, 50]


@pytest.mark.parametrize("S", SMALL_S)
def test_pieces_tile_every_window_small_windows(S):
    for K in range(1, 51):
        for E in (0, 1, 2, 17):
            for subs in (1, 2, 4, 6):
                for acc_n in (256, 128):
                    for emit in (False, True):
                        err = coverage_errors(K, E, S, acc_n, subs, emit)
                        assert err is None, f"K={K} E={E} S={S} subs={subs} acc_n={acc_n} emit={emit}: {err}"


@pytest.mark.parametrize("S", PRESET_S)
def test_pieces_tile_every_window_preset_windows(S):
    for K in K_AT_EDGES:
        for E in (0, 1, 2, 17):
            for subs in (1, 2, 4, 6):
                for acc_n in (256, 128):
                    err = coverage_errors(K, E, S, acc_n, subs)
                    assert err is None, f"K={K} E={E} S={S} subs={subs} acc_n={acc_n}: {err}"


@pytest.mark.parametrize("S,E", [(5041, 3), (5041, 171), (65535, 2), (65535, 3), (255 * 255, 5)])
def test_pieces_tile_every_window_large_windows(S, E):
    for K in (1, 18, 44):
        for subs, acc_n in ((1, 256), (6, 128)):
            err = coverage_errors(K, E, S, acc_n, subs)
            assert err is None, f"K={K} E={E} S={S} subs={subs} acc_n={acc_n}: {err}"


def test_work_items_cover_every_channel_tile_once():
    for n_ntiles in (1, 2, 3, 5, 6, 9, 30, 60):
        for n_tiles in (1, 2, 5, 29, 147, 148, 149, 450):
            chunk_tiles, n_chunks, n_items = plan_items(n_tiles, n_ntiles, 148)
            seen = [(tile, nt) for item in range(n_items)
                    for tile, nt0, nt1 in [head_item(item, n_chunks, chunk_tiles, n_ntiles)] for nt in range(nt0, nt1)]
            assert sorted(seen) == [(t, nt) for t in range(n_tiles) for nt in range(n_ntiles)], (n_tiles, n_ntiles)


def division_failures(div, S_max=65535, E_max=255):
    """Every S <= S_max against every p < S * E_max: the first (S, p) where div's window index is not p // S.  Per
    quotient q the worst p are q * S (the smallest) and q * S + S - 1 (the largest, where a rounded-up magic
    overshoots first), so those two are all that is checked."""
    make_magic, index = div
    S = np.arange(1, S_max + 1, dtype=np.uint64)
    magic = np.array([make_magic(int(s)) for s in S], dtype=np.uint64)
    bad = []
    for q in range(E_max):
        for r in (np.zeros_like(S), S - np.uint64(1)):
            p = np.uint64(q) * S + r
            got = index(p, magic)
            wrong = np.nonzero(got != np.uint64(q))[0]
            bad += [(int(S[i]), int(p[i])) for i in wrong]
    return sorted(bad)


def test_window_index_division_is_exact_over_every_accepted_shape():
    """check_shape accepts sH * sW <= 65535 and E <= 255, so every limb channel p < S * E is below 2^24."""
    assert division_failures(KERNEL_DIV) == []


def test_the_checks_catch_the_32_bit_division():
    """The formula the kernel used before: 0 for S = 1 (no identity case: the walk never leaves the second limb
    column), and inexact for large windows — 255 x 257 from E = 2, 71 x 71 from E = 170.  (At 255 x 257 and E = 2
    the only wrong channel is the odd p = 2S - 1, where no run starts; from E = 3 runs start on wrong channels.)"""
    assert coverage_errors(16, 15, 1, 256, 4, div=OLD_DIV).startswith("walk stuck")
    assert coverage_errors(18, 17, 1, 128, 6, div=OLD_DIV).startswith("walk stuck")
    assert coverage_errors(2, 3, 65535, 256, 2, div=OLD_DIV) is not None
    assert coverage_errors(2, 3, 65535, 256, 2) is None
    bad = division_failures(OLD_DIV)
    first = {}
    for S, p in bad:
        first.setdefault(S, p // S + 1)                       # the smallest E whose channels include p
    assert first[1] == 2 and first[65535] == 2 and first[5041] == 170
