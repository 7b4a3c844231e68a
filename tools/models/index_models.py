"""Index models of the round-2 kernels, restated index for index in Python so that the arithmetic the kernels rely on can be
checked exhaustively on the CPU (tests/test_cpu_oracle.py):

* `ook_fold_index` / `sorted_key_pair` -- the block-sum kernel's folded envelope table (k_ook.cu): one PRMT + VIMNMX.U16x2 sort
  the byte pairs of two samples, `max(key, 65279 - key)` folds the triangle {lo <= hi} into rows 127..255, `k2 + (k2 >> 5)` skews
  the rows 8 banks apart.
* `ook_rank_slot` -- the slicer's rank table indexed from the raw halfword.
* `gen_tile_offsets` / `chunk_plan` -- the padded-chunk tile of the generic fused chain and FIR tile kernel
  (chain_generic.cuh: GenTile, load_sub): where sample j of a thread window lives, which bulk copies a tile takes, and that
  every sample a tap can reach was either copied or lies in the zeroed tail.
"""
import numpy as np

OOK_FOLD_C = 65279
OOK_FOLD_MIN = 32640 + (32640 >> 5)
OOK_FOLD_MAX = 65535 + (65535 >> 5)


def sorted_key_pair(w: int) -> tuple[int, int]:
    """w = b0 | b1 << 8 | b2 << 16 | b3 << 24 (two samples): (key0, key1) with key = hi << 8 | lo of each sample's byte pair"""
    swapped = ((w & 0x00FF00FF) << 8) | ((w >> 8) & 0x00FF00FF)          # PRMT 0x2301
    lo = max(w & 0xFFFF, swapped & 0xFFFF)                                # VIMNMX.U16x2
    hi = max(w >> 16, swapped >> 16)
    return lo, hi


def ook_fold_index(key: int) -> int:
    alt = OOK_FOLD_C - key                                               # negative for hi = 255: loses the SIGNED max
    k2 = max(alt, key)
    return k2 + (k2 >> 5)                                                # LEA.HI


def ook_rank_slot(raw: int) -> int:
    return raw + (raw >> 5)


def gen_tile(ntaps_max: int, decim: int, r: int):
    step = r * decim
    win = (r - 1) * decim + ntaps_max
    winl = (win + 1) & ~1
    padb = 16 if (step // 2) % 2 == 0 else 0
    pitch = step * 8 + padb
    return step, win, winl, padb, pitch


def gen_tile_offsets(ntaps_max: int, decim: int, r: int):
    """byte offset of sample j of a thread window, from the window start"""
    step, win, winl, padb, pitch = gen_tile(ntaps_max, decim, r)
    return [j * 8 + padb * (j // step) for j in range(winl)]


def chunk_plan(tile_in: int, step: int):
    """(chunk, first sample, samples by bulk copy, hand-copied sample or None) as load_sub issues them"""
    n_chunks = (tile_in + step - 1) // step
    tma = tile_in & ~1
    out = []
    for c in range(n_chunks):
        s0 = c * step
        ns = min(step, tma - s0)
        hand = tile_in - 1 if (tile_in & 1) and s0 + step >= tile_in and s0 < tile_in else None
        out.append((c, s0, max(ns, 0), hand))
    return out


# ---- OOK trigger kernel, round 2: book-keeping from the walker's masks ------------------------------------------------------
# The walker leaves, per stream and tile of 32 blocks, cm (bit u: block u is collected, bitfount.rs:73) and sm (bit u: block u
# sends, :78).  keeper_blockwise is the reference's statements taken block by block (the kernel's slow path, used where the OOM
# guard :52-54 could fire); keeper_send_to_send / tags_from_masks are the fast path: the keeper steps from send to send counting
# collected blocks with popc, the helpers expand tags as "burst index at the start of the tile + sends before the block".
OOK_BLOCK_SAMPLES = 512


def _keeper_tile_blockwise(cm, sm, nb, t, state, guard_samples, max_bursts, tags, events):
    buf_len, lead0, burst, dropped = state
    for u in range(nb):
        if buf_len > guard_samples:                              # :52-54
            if burst < max_bursts:
                events.append((burst, 0, t * 32 + u - 1))
            burst += 1; dropped = True; buf_len = 1; lead0 = True
        collect = (cm >> u) & 1                                  # :73-75
        buf_len += OOK_BLOCK_SAMPLES if collect else 0
        tags.append(burst if (collect and burst < max_bursts) else -1)
        if (sm >> u) & 1:                                        # :78-81
            if burst < max_bursts:
                events.append((burst, 1 | (2 if lead0 else 0), t * 32 + u))
            burst += 1; buf_len = 0; lead0 = False
    return buf_len, lead0, burst, dropped


def keeper_blockwise(tiles, guard_samples, max_bursts):
    """tiles: list of (cm, sm, nb).  Returns (tags per block, [(burst, flags, end block)], (buf_len, lead0, burst, dropped))."""
    state, tags, events = (1, True, 0, False), [], []
    for t, (cm, sm, nb) in enumerate(tiles):
        state = _keeper_tile_blockwise(cm, sm, nb, t, state, guard_samples, max_bursts, tags, events)
    return tags, events, state


def keeper_send_to_send(tiles, guard_samples, max_bursts):
    """The kernel's keeper: per tile the fast path unless the guard could fire in it (then block by block)."""
    state, tags, events = (1, True, 0, False), [], []
    popc = lambda x: bin(x & 0xFFFFFFFF).count("1")
    for t, (cm, sm, nb) in enumerate(tiles):
        buf_len, lead0, burst, dropped = state
        if buf_len + 32 * OOK_BLOCK_SAMPLES > guard_samples:
            state = _keeper_tile_blockwise(cm, sm, nb, t, state, guard_samples, max_bursts, tags, events)
            continue
        b0 = burst
        rem, done = sm, 0
        while rem:
            u = (rem & -rem).bit_length() - 1
            rem &= rem - 1
            upto = (1 << u) - 1
            buf_len += OOK_BLOCK_SAMPLES * popc(cm & upto & ~done)
            done = upto | (1 << u)
            if burst < max_bursts:
                events.append((burst, 1 | (2 if lead0 else 0), t * 32 + u))
            burst += 1; buf_len = 0; lead0 = False
        buf_len += OOK_BLOCK_SAMPLES * popc(cm & ~done)
        for u in range(nb):                                     # tags_out of the helpers
            bi = b0 + popc(sm & ((1 << u) - 1))
            tags.append(bi if ((cm >> u) & 1 and bi < max_bursts) else -1)
        state = (buf_len, lead0, burst, dropped)
    return tags, events, state


# ---- OOK slicer: summaries -> scan -> scatter ---------------------------------------------------------------------------------
# A stream is a list of blocks (tag, bits): tag = index of the burst the block is collected into (-1: not collected), bits = its
# 512 slicer outputs.  flags[j] of burst j: bit 0 sent, bit 1 the burst starts with the 0.0 of vec!(0.0) (one 0 bit); a burst with
# flags 3 and no tagged block is the lone [0.0] the OOM guard leaves behind (bitfount.rs:52-54, :78-81).  rle_split restates
# ook_slice_kernel's summaries, ook_scan_kernel's 32-block steps with their carry and ook_scatter_kernel; the result is kpn::rle on
# the flattened bit stream (kpn.rs:17-29: a position is recorded where the value changes).
def rle_split(blocks, flags, n_bursts):
    # C1: per collected block {transitions between its own bits, first bit, last bit}
    summ = [None if t < 0 else (sum(1 for i in range(1, len(b)) if b[i] != b[i - 1]), b[0], b[-1]) for t, b in blocks]
    lone = lambda frm, to: sum(1 for j in range(frm, to) if flags[j] & 3 == 3)
    # C2: 32 blocks per step, everything inside a step from prefix sums, (pos, ntr, prev, cur) carried between steps
    pos, ntr, prev, cur = 0, 0, 0, -1
    info = [None] * len(blocks)
    tail = []
    for g0 in range(0, len(blocks), 32):
        grp = range(g0, min(g0 + 32, len(blocks)))
        col = [k for k in grp if blocks[k][0] >= 0]
        if not col:
            continue
        n_ins, ptag, plast = {}, {}, {}
        for i, k in enumerate(col):                               # the collected block before this one: in the group, or the carry
            ptag[k] = blocks[col[i - 1]][0] if i else cur
            plast[k] = summ[col[i - 1]][2] if i else prev
            tg = blocks[k][0]
            n_ins[k] = (lone(ptag[k] + 1, tg) + (1 if flags[tg] & 2 else 0)) if tg != ptag[k] else 0
        excl_bits, excl_tr = 0, 0
        for k in col:
            cnt, first, last = summ[k]
            pos_ins = pos + excl_bits
            pos_base = pos_ins + n_ins[k]
            before = 0 if n_ins[k] else plast[k]
            pre = n_ins[k] > 0 and pos_ins > 0 and plast[k] != 0
            first_t = pos_base > 0 and first != before
            info[k] = (pos_base, ntr + excl_tr, pos_ins, pre, first_t)
            excl_bits += 512 + n_ins[k]
            excl_tr += cnt + int(pre) + int(first_t)
        pos += excl_bits
        ntr += excl_tr
        cur = blocks[col[-1]][0]
        prev = summ[col[-1]][2]
    n = lone(cur + 1, n_bursts)
    if n:
        if pos > 0 and prev != 0:
            tail.append((ntr, pos))
            ntr += 1
        pos += n
    # C3: every block writes its transitions at its place
    trans = [None] * ntr
    for k, (t, b) in enumerate(blocks):
        if t < 0:
            continue
        pos_base, o, pos_ins, pre, first_t = info[k]
        if pre:
            trans[o] = pos_ins; o += 1
        if first_t:
            trans[o] = pos_base; o += 1
        for i in range(1, len(b)):
            if b[i] != b[i - 1]:
                trans[o] = pos_base + i; o += 1
    for o, p in tail:
        trans[o] = p
    return trans, pos
