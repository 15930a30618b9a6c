"""Generate csrc/cube_tables.cuh: every constant table the sm_100a kernels use.

    python rubiks_cube_solver_b200/csrc/gen_tables.py            # rewrite the header
    python rubiks_cube_solver_b200/csrc/gen_tables.py --check    # verify it is current + self-test

The header is committed; build() only compiles it.  This script is product code
and deliberately does NOT import ``oracle/`` -- it restates the reference's
constants independently (the tests then compare the two restatements and the
reference dump in tests/golden/reference_tables.npz):

* face turns            gym-cube/gym_cube/envs/assets/py333.py:46-138 (``moveDefs``),
                        action order cube_env.py:24-28
* one-hot hash tables   py333.py:140-198 (``corner_pieceDefs`` .. ``edge_pieceInds``), as
                        shipped, including the mirrored corner row 6 and the zero-default
                        holes of ``corner_pieceInds``
* 2x2x2                 the un-vendored assets/py222.py (MeepMoop/py222), SURVEY.md Appendix A

Internal cubie model (used only by the fused scramble kernel; never visible at
the boundary).  A cube reached from solved is tracked as 8 corner bytes
``piece | twist_sum << 3`` and 12 edge bytes ``piece | flip << 4``.  A face turn m
is  ``new[q] = old[src_m[q]] + delta_m[q]``  which is one PRMT (byte permute) per
output register plus one add / xor, with the per-move selector words fetched
from shared memory -- no branch on the move, so lanes holding different moves
do not diverge.  Edge slots are ordered F/B-layer-aware so that only U and D
turns flip edges:

    slot order   corners: the 8 rows of corner_pieceDefs (row 6 un-mirrored)
                 edges  : reg0 = U layer (UB UL UF UR), reg1 = middle layer
                          (FL FR BR BL), reg2 = D layer (DB DL DF DR)
    edge reference sticker: the F/B sticker for the 8 edges touching F or B,
                 the U/D sticker for UL UR DL DR  ->  F, B, R, L never flip.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "cube_tables.cuh")

ACTIONS_3 = ["U", "U'", "F", "F'", "R", "R'", "D", "D'", "B", "B'", "L", "L'"]

# clockwise quarter turns as sticker 4-cycles (a b c d): new[a] = old[b], new[b] = old[c], ...
CW = {
    "U": "0 6 8 2 | 1 3 7 5 | 9 45 36 18 | 10 46 37 19 | 11 47 38 20",
    "F": "6 44 29 9 | 7 41 28 12 | 8 38 27 15 | 18 24 26 20 | 19 21 25 23",
    "R": "2 20 29 51 | 5 23 32 48 | 8 26 35 45 | 9 15 17 11 | 10 12 16 14",
    "D": "15 24 42 51 | 16 25 43 52 | 17 26 44 53 | 27 33 35 29 | 28 30 34 32",
    "B": "0 11 35 42 | 1 14 34 39 | 2 17 33 36 | 45 51 53 47 | 46 48 52 50",
    "L": "0 53 27 18 | 3 50 30 21 | 6 47 33 24 | 36 42 44 38 | 37 39 43 41",
}


def cycles_of(name):
    return [[int(x) for x in c.split()] for c in CW[name].split("|")]


def gather_row(n, cycles, inverse=False):
    row = list(range(n))
    for c in cycles:
        for k, a in enumerate(c):
            if inverse:
                row[c[(k + 1) % 4]] = a
            else:
                row[a] = c[(k + 1) % 4]
    return row


MOVES_3 = []          # [12][54] gather rows
CYCLES_3 = []         # [12][5][4] : new[c[k]] = old[c[k+1]]
for _name in ACTIONS_3[0::2]:
    _cyc = cycles_of(_name)
    MOVES_3.append(gather_row(54, _cyc))
    CYCLES_3.append(_cyc)
    MOVES_3.append(gather_row(54, _cyc, inverse=True))
    CYCLES_3.append([[c[0], c[3], c[2], c[1]] for c in _cyc])
MOVES_3 = np.array(MOVES_3)

# 2x2x2 sticker 4f+k <-> 3x3x3 corner sticker 9f+(0,2,6,8)[k]
TO3 = [9 * (i // 4) + (0, 2, 6, 8)[i % 4] for i in range(24)]
TO2 = {s3: i for i, s3 in enumerate(TO3)}
MOVES_2 = np.array([[TO2[MOVES_3[a][s3]] for s3 in TO3] for a in range(6)])
CYCLES_2 = [[[TO2[s] for s in c] for c in CYCLES_3[a] if c[0] in TO2] for a in range(6)]

# ---- reference one-hot tables (as shipped) ---------------------------------
CORNER_DEFS_REF = [[0, 47, 36], [6, 38, 18], [8, 20, 9], [2, 11, 45],
                   [33, 42, 53], [27, 24, 44], [29, 26, 15], [35, 51, 17]]
EDGE_DEFS_REF = [[1, 46], [3, 37], [7, 19], [5, 10], [34, 52], [30, 43],
                 [28, 25], [32, 16], [21, 41], [23, 12], [48, 14], [50, 39]]
CORNER_HASHES_REF = [(50, 54, 13), (28, 8, 42), (14, 5, 12), (52, 11, 15),
                     (61, 44, 51), (47, 30, 40), (17, 35, 18), (23, 56, 21)]
PIECE_DEFS_2 = [[0, 21, 16], [2, 17, 8], [3, 9, 4], [1, 5, 20],
                [12, 10, 19], [13, 6, 11], [15, 22, 7]]

CORNER_COL_3 = [0] * 128        # hash -> 3*piece+ori (0 where the shipped table has a hole)
for _p, _hs in enumerate(CORNER_HASHES_REF):
    for _o, _h in enumerate(_hs):
        CORNER_COL_3[_h] = 3 * _p + _o
EDGE_COL_3 = [0] * 128          # hash -> 2*piece+ori
for _p, (_s0, _s1) in enumerate(EDGE_DEFS_REF):
    _a, _b = _s0 // 9, _s1 // 9
    EDGE_COL_3[_a + 10 * _b] = 2 * _p
    EDGE_COL_3[_b + 10 * _a] = 2 * _p + 1
PIECE_CODE_2 = [0] * 128        # hash -> cubelet | ori << 4
for _p in range(7):
    _c = [s // 4 for s in PIECE_DEFS_2[_p]]
    for _o in range(3):
        _r = _c[-_o:] + _c[:-_o] if _o else _c          # np.roll(c, o)
        PIECE_CODE_2[_r[0] + 2 * _r[1] + 10 * _r[2]] = _p | (_o << 4)

# ---- internal cubie model ---------------------------------------------------
CORNER_SLOTS_3 = [list(r) for r in CORNER_DEFS_REF]
CORNER_SLOTS_3[6] = [29, 15, 26]                       # un-mirrored: same chirality as the rest
EDGE_SLOTS_3 = [[46, 1], [3, 37], [19, 7], [5, 10],    # UB UL UF UR   (reference sticker first)
                [21, 41], [23, 12], [48, 14], [50, 39],  # FL FR BR BL
                [52, 34], [30, 43], [25, 28], [32, 16]]  # DB DL DF DR
CORNER_SLOTS_2 = [[TO2[s] for s in r] for r in CORNER_SLOTS_3]   # slot 4 = the fixed DBL cubie


def cubie_action(moves, slots):
    """src[m][q], rot[m][q] with new[q] = old[src] twisted by rot."""
    where = {}
    for q, st in enumerate(slots):
        for k, s in enumerate(st):
            where[s] = (q, k)
    n = len(slots[0])
    src = np.zeros((len(moves), len(slots)), dtype=int)
    rot = np.zeros((len(moves), len(slots)), dtype=int)
    for m, row in enumerate(moves):
        for q, st in enumerate(slots):
            q2, k2 = where[row[st[0]]]
            for k, s in enumerate(st):
                assert where[row[s]] == (q2, (k + k2) % n), "slot stickers must share chirality"
            src[m][q], rot[m][q] = q2, k2
    return src, rot


C_SRC_3, C_ROT_3 = cubie_action(MOVES_3, CORNER_SLOTS_3)
E_SRC_3, E_ROT_3 = cubie_action(MOVES_3, EDGE_SLOTS_3)
C_SRC_2, C_ROT_2 = cubie_action(MOVES_2, CORNER_SLOTS_2)
assert all(E_ROT_3[m].sum() == 0 for m in (2, 3, 4, 5, 8, 9, 10, 11)), "only U/D may flip edges"
assert all(E_ROT_3[m][4:8].sum() == 0 for m in range(12)), "middle-layer edges never flip"

# 2x2x2 distance table (csrc/cube_distance.cuh): the cubies in py222 getOP's own terms -- slot q = the stickers
# PIECE_DEFS_2[q], byte = cubelet | ori << 4 (kPieceCode2's format), a cubelet at ori o showing np.roll(home, o).
# A turn moves the byte of slot src into slot q and adds (3 - rot) mod 3 to its ori.
_D_SRC_2, _D_ROT_2 = cubie_action(MOVES_2, PIECE_DEFS_2)
DIST_MOVE_2 = [int(_D_SRC_2[a][q]) | ((3 - int(_D_ROT_2[a][q])) % 3) << 4 for a in range(6) for q in range(7)]
CUBIE_COLOURS_2 = [0] * 21      # 3 * cubelet + ori -> the colours the slot's stickers k = 0..2 show, one per byte
for _p in range(7):
    _c = [s // 4 for s in PIECE_DEFS_2[_p]]
    for _o in range(3):
        CUBIE_COLOURS_2[3 * _p + _o] = sum(_c[(k - _o) % 3] << (8 * k) for k in range(3))

N_MOVE_ROWS = 16          # rows 0..A-1 = moves, the rest = identity (row 12 doubles as "no-op")
W3 = 10                   # words per 3x3x3 move
W2 = 4                    # words per 2x2x2 move


def _sel(nibbles):
    v = 0
    for i, nb in enumerate(nibbles):
        assert 0 <= nb < 8
        v |= nb << (4 * i)
    return v


def _bytes(vals):
    v = 0
    for i, b in enumerate(vals):
        assert 0 <= b < 256
        v |= b << (8 * i)
    return v


def move_words_3(m):
    """10 words: selC0 selC1 dC0 dC1 selE0 selE2 selEt selE1 fE0 fE2 (identity when m >= 12)."""
    if m >= 12:
        return [0x3210, 0x7654, 0, 0, 0x3210, 0x3210, 0x3210, 0x3210, 0, 0]
    cs, cr, es, er = C_SRC_3[m], C_ROT_3[m], E_SRC_3[m], E_ROT_3[m]
    selc0 = _sel([cs[q] for q in range(0, 4)])                       # prmt(c0, c1, .)
    selc1 = _sel([cs[q] for q in range(4, 8)])
    dc0 = _bytes([cr[q] << 3 for q in range(0, 4)])
    dc1 = _bytes([cr[q] << 3 for q in range(4, 8)])
    s0, s2, st, s1 = [], [], [], []
    for q in range(0, 4):                                            # out0 = prmt(e0, e1, s0)
        s = es[q]
        assert s < 8
        s0.append(s if s < 4 else 4 + (s - 4))
    for q in range(8, 12):                                           # out2 = prmt(e2, e1, s2)
        s = es[q]
        assert s >= 4
        s2.append(s - 8 if s >= 8 else 4 + (s - 4))
    for i, q in enumerate(range(4, 8)):                              # t = prmt(e0, e2, st); out1 = prmt(e1, t, s1)
        s = es[q]
        if 4 <= s < 8:
            st.append(0)
            s1.append(s - 4)
        else:
            st.append(s if s < 4 else 4 + (s - 8))
            s1.append(4 + i)
    f0 = _bytes([er[q] << 4 for q in range(0, 4)])
    f2 = _bytes([er[q] << 4 for q in range(8, 12)])
    return [selc0, selc1, dc0, dc1, _sel(s0), _sel(s2), _sel(st), _sel(s1), f0, f2]


def move_words_2(m):
    if m >= 6:
        return [0x3210, 0x7654, 0, 0]
    cs, cr = C_SRC_2[m], C_ROT_2[m]
    return [_sel([cs[q] for q in range(0, 4)]), _sel([cs[q] for q in range(4, 8)]),
            _bytes([cr[q] << 3 for q in range(0, 4)]), _bytes([cr[q] << 3 for q in range(4, 8)])]


def packed_words_3(m):
    """5 words the kernel actually loads: A = selC0 | selC1 << 16, B = dC0, D = selE0 | selE2 << 16,
    E = selEt | selE1 << 16, F = fE0 | fE2 << 1 (bit 4 / bit 5 per byte; an edge is flipped when
    bits 4 and 5 of its byte differ).
    PRMT reads only the low 16 bits of its selector, so A, D, E are used as they are for the
    first permute and shifted right by 16 for the second.  The D-layer corner twists need no
    word of their own: corner slot q+4 sits directly below slot q and a side-face turn twists
    the two in opposite senses, so dC1 == 2 * dC0 (mod 3) byte for byte (asserted here)."""
    w = move_words_3(m)
    for q in range(4):
        d0, d1 = (w[2] >> (8 * q + 3)) & 3, (w[3] >> (8 * q + 3)) & 3
        assert d1 == (2 * d0) % 3, "D-layer twist must be the negative of the U-layer twist"
    return [w[0] | w[1] << 16, w[2], w[4] | w[5] << 16, w[6] | w[7] << 16, w[8] | w[9] << 1]


def packed_words_2(m):
    w = move_words_2(m)
    for q in range(4):
        d0, d1 = (w[2] >> (8 * q + 3)) & 3, (w[3] >> (8 * q + 3)) & 3
        assert d1 == (2 * d0) % 3
    return [w[0] | w[1] << 16, w[2]]



# ---- pair tables: two face turns per table row (fused scramble kernel K1p) ---------------
# Row p = m0 + 13 * m1 applies m0 and then m1 (index 12 = no move), so a byte pair of the move
# stream is one table lookup:  new[q] = old[src[q]] + delta[q]  with src = src_m0 o src_m1 and
# delta[q] = delta_m0[src_m1[q]] + delta_m1[q] (twists mod 3, flips mod 2).
PAIR_BASE = 13
PAIR_ROWS = PAIR_BASE * PAIR_BASE


def _ident_or(table, m, n):
    return list(table[m]) if m < len(table) else list(range(n))


def _zero_or(table, m, n):
    return list(table[m]) if m < len(table) else [0] * n


def compose(src_t, rot_t, m0, m1, n, mod):
    s0, r0 = _ident_or(src_t, m0, n), _zero_or(rot_t, m0, n)
    s1, r1 = _ident_or(src_t, m1, n), _zero_or(rot_t, m1, n)
    return [s0[s1[q]] for q in range(n)], [(r0[s1[q]] + r1[q]) % mod for q in range(n)]


def pair_words_3(p):
    """8 words of one 3x3x3 pair row, as the kernel loads them (two 16-byte vectors):
    P = [selC0 | selC1 << 16, T0, T1, F]      c0' = prmt(c0, c1, selC0) + T0, c1' likewise with T1;
                                              F = flips of e0 at bit 4 | flips of e2 at bit 5
    Q = [st0 | so0 << 16, st1 | so1 << 16, st2 | so2 << 16, F1]
        t_k = prmt(e_x, e_y, st_k) gathers the bytes output register k takes from the two OTHER
        registers ((x, y) = (1,2), (0,2), (0,1)); e_k' = prmt(e_k, t_k, so_k) ^ flips; F1 = flips of
        e1 at bit 4.  An edge is flipped when bits 4 and 5 of its byte differ."""
    m0, m1 = p % PAIR_BASE, p // PAIR_BASE
    cs, cr = compose(C_SRC_3, C_ROT_3, m0, m1, 8, 3)
    es, er = compose(E_SRC_3, E_ROT_3, m0, m1, 12, 2)
    P = [_sel(cs[0:4]) | _sel(cs[4:8]) << 16,
         _bytes([r << 3 for r in cr[0:4]]), _bytes([r << 3 for r in cr[4:8]]),
         _bytes([r << 4 for r in er[0:4]]) | _bytes([r << 5 for r in er[8:12]])]
    Q = []
    for k, (x, y) in enumerate(((1, 2), (0, 2), (0, 1))):
        st, so = [], []
        for i in range(4):
            s = es[4 * k + i]
            if s // 4 == k:
                st.append(0)
                so.append(s - 4 * k)
            else:
                st.append(s - 4 * x if s // 4 == x else 4 + s - 4 * y)
                so.append(4 + i)
        Q.append(_sel(st) | _sel(so) << 16)
    Q.append(_bytes([r << 4 for r in er[4:8]]))
    return P + Q


def pair_words_2(p):
    """4 words of one 2x2x2 pair row: [selC0 | selC1 << 16, T0, T1, 0]; indices 6..12 = no move.
    (Measured and rejected: T0 | T1 << 2 in one word, i.e. one 64-bit load per pair instead of a 64- and a
    32-bit one -- a third fewer table wavefronts, but the two ANDs of the unpacking cost more: -6 %.)"""
    m0, m1 = p % PAIR_BASE, p // PAIR_BASE
    cs, cr = compose(C_SRC_2, C_ROT_2, m0, m1, 8, 3)
    return [_sel(cs[0:4]) | _sel(cs[4:8]) << 16,
            _bytes([r << 3 for r in cr[0:4]]), _bytes([r << 3 for r in cr[4:8]]), 0]


def fold_twist(c):
    return (c & 0x1f1f1f1f) + ((c >> 2) & 0x38383838)


PW3 = 5
PW2 = 2


def colour_lut(slots, per_face, n_or):
    """lut[piece | ori << sh] = colours seen at slot sticker positions k=0.. (one byte each).
    Position k of the slot shows home sticker (k + ori) % n of the piece."""
    sh = 3 if n_or == 3 else 4
    lut = [0] * 32
    for p, st in enumerate(slots):
        for o in range(n_or):
            lut[p | (o << sh)] = _bytes([st[(k + o) % n_or] // per_face for k in range(n_or)])
    return lut


C_LUT_3 = colour_lut(CORNER_SLOTS_3, 9, 3)
# Edge flip is the PARITY of bits 4 and 5 of the edge byte: U-layer flips toggle bit 4 and
# D-layer flips toggle bit 5, so the packed flip word F = fE0 | fE2 << 1 is applied with two fused
# and-xor LOP3s and no shift.  The edge colour LUT therefore has 64 entries.
_E_LUT_32 = colour_lut(EDGE_SLOTS_3, 9, 2)
E_LUT_3 = [_E_LUT_32[(i & 15) | ((((i >> 4) ^ (i >> 5)) & 1) << 4)] for i in range(64)]
C_LUT_2 = colour_lut(CORNER_SLOTS_2, 4, 3)
# K1p's finishing pass reads the edge colours from one LUT PER SLOT (32 canonical entries each: piece | flip << 4).
# Bytes 0, 1 are the two colours as above; bytes 2, 3 are the CENTRE colours of the faces that the slot's sticker
# positions 0 and 1 lie on -- constants of the slot.  A centre sticker always shares its output word with an edge
# sticker of its own face, so the row assembly takes it from that edge's LUT word instead of from an immediate:
# one source register fewer, i.e. one byte permute fewer, in six words of a row.
E_LUT_SLOT_3 = [[_E_LUT_32[i] | (st[0] // 9) << 16 | (st[1] // 9) << 24 for i in range(32)] for st in EDGE_SLOTS_3]
CENTRE_ALTERNATIVES_3 = {f: [(8 + s_, 2 + k) for s_, st in enumerate(EDGE_SLOTS_3) for k in range(2) if st[k] // 9 == f]
                         for f in range(6)}


def sticker_sources(slots_list, n_stickers, centres):
    """For every sticker position: (slot_register_index, byte) or a constant colour.
    Register index: 0..len-1 in the order slots are listed."""
    src = [None] * n_stickers
    idx = 0
    for slots in slots_list:
        for st in slots:
            for k, s in enumerate(st):
                src[s] = (idx, k)
            idx += 1
    for s, col in centres.items():
        src[s] = ("const", col)
    assert all(v is not None for v in src)
    return src


# ---- sticker-level tables for the walk (step) and expand kernels ------------
def cycle_words(cycles):
    """5 (3x3x3) / 3 (2x2x2) words per move, bytes (a,b,c,d): new[a]=old[b] ... new[d]=old[a]."""
    return [[_bytes(c) for c in mv] for mv in cycles]


def hash_defs_3():
    """[20] words: bytes = the sticker positions feeding each slot's hash (corner_pieceDefs /
    edge_pieceDefs as shipped); byte 3 = 1 for edge slots."""
    words = [_bytes([d[0], d[1], d[2], 0]) for d in CORNER_DEFS_REF]
    words += [_bytes([d[0], d[1], d[1], 1]) for d in EDGE_DEFS_REF]
    return words


# ---- opt-in EXACT 3x3x3 encoding (SURVEY.md section 8f4) ---------------------------------------
# The shipped corner table is lossy: row 6 of corner_pieceDefs is mirrored (read anticlockwise where the
# other seven slots are read clockwise) and corner_pieceInds was patched by hand, so reachable states fall
# into unassigned hashes.  The exact encoding keeps the reference's layout ([20, 24], corners: column =
# 3 * piece + ori, edges: 2 * piece + ori, same hash weights) but reads slot 6 the right way round and
# assigns every rotation of every corner the py222 way, (piece, ori) <- np.roll(home colours, ori):
# a bijection between cube states and one-hot observations, which the shipped one is not.
CORNER_DEFS_EXACT = [list(r) for r in CORNER_SLOTS_3]                  # slot 6 = [29, 15, 26]
CORNER_COL_3X = [0] * 128       # hash -> 3*piece+ori, all 24 rotations assigned
CORNER_HOME_3X = [0] * 24       # column -> the three colours the slot's stickers show, one per byte
for _p in range(8):
    _c = [s_ // 9 for s_ in CORNER_DEFS_EXACT[_p]]
    for _o in range(3):
        _r = _c[-_o:] + _c[:-_o] if _o else _c                          # np.roll(c, o)
        assert CORNER_COL_3X[_r[0] + 2 * _r[1] + 10 * _r[2]] == 0 or (_p, _o) == (0, 0)
        CORNER_COL_3X[_r[0] + 2 * _r[1] + 10 * _r[2]] = 3 * _p + _o
        CORNER_HOME_3X[3 * _p + _o] = _r[0] | _r[1] << 8 | _r[2] << 16
EDGE_HOME_3 = [0] * 24          # column -> the two colours (the shipped edge table is already a bijection)
for _p, (_s0, _s1) in enumerate(EDGE_DEFS_REF):
    _a, _b = _s0 // 9, _s1 // 9
    EDGE_HOME_3[2 * _p] = _a | _b << 8
    EDGE_HOME_3[2 * _p + 1] = _b | _a << 8
# sticker -> (slot, position inside the slot) for decoding: slot | k << 5; centres: 0x80 | colour
STICKER_SLOT_3X = [0] * 54
for _f in range(6):
    STICKER_SLOT_3X[9 * _f + 4] = 0x80 | _f
for _q, _d in enumerate(CORNER_DEFS_EXACT):
    for _k, _s in enumerate(_d):
        STICKER_SLOT_3X[_s] = _q | _k << 5
for _q, _d in enumerate(EDGE_DEFS_REF):
    for _k, _s in enumerate(_d):
        STICKER_SLOT_3X[_s] = (8 + _q) | _k << 5


# 3x3x3 pattern databases (csrc/cube_pattern.cuh): the cubies of the exact encoding -- corner slot q = the stickers
# CORNER_DEFS_EXACT[q], edge slot q = EDGE_DEFS_REF[q], byte = piece | ori << 4, a piece at ori o showing
# np.roll(home colours, o).  A turn moves the byte of slot src into slot q and adds (n - rot) mod n to its ori.
_P_CSRC_3, _P_CROT_3 = cubie_action(MOVES_3, CORNER_DEFS_EXACT)
_P_ESRC_3, _P_EROT_3 = cubie_action(MOVES_3, EDGE_DEFS_REF)
PAT_MOVE_3 = [[int(_P_CSRC_3[a][q]) | ((3 - int(_P_CROT_3[a][q])) % 3) << 4 for q in range(8)]
              + [int(_P_ESRC_3[a][q]) | ((2 - int(_P_EROT_3[a][q])) % 2) << 4 for q in range(12)] for a in range(12)]


def hash_defs_3x():
    words = [_bytes([d[0], d[1], d[2], 0]) for d in CORNER_DEFS_EXACT]
    words += [_bytes([d[0], d[1], d[1], 1]) for d in EDGE_DEFS_REF]
    return words


def hash_defs_2():
    return [_bytes([d[0], d[1], d[2], 0]) for d in PIECE_DEFS_2]


def assemble_fn(name, src, n_words):
    """Straight-line code: out word j = stickers 4j..4j+3, each a byte of L[slot] or a constant."""
    lines = ["CUBE_HD void %s(const uint32_t* L, uint32_t* w)\n{\n" % name]
    for j in range(n_words):
        ops = []
        for b in range(4):
            s_ = 4 * j + b
            if s_ >= len(src) or src[s_][0] == "const":
                col = 0 if s_ >= len(src) else src[s_][1]
                ops.append(("0x%02xu" % col, 0))
            else:
                ops.append(("L[%d]" % src[s_][0], src[s_][1]))
        lo = "cube_prmt(%s, %s, 0x%04xu)" % (ops[0][0], ops[1][0], 0x4400 | ops[0][1] | ((4 + ops[1][1]) << 4))
        hi = "cube_prmt(%s, %s, 0x%04xu)" % (ops[2][0], ops[3][0], 0x4400 | ops[2][1] | ((4 + ops[3][1]) << 4))
        lines.append("    w[%d] = cube_prmt(%s, %s, 0x5410u);\n" % (j, lo, hi))
    lines.append("}\n\n")
    return "".join(lines)



def _prmt_expr(ops):
    """Fewest byte permutes that put ops[i] = (operand, byte) into output byte i (None = don't care).
    Operands are C expressions (L[slot] or an immediate); at most four distinct ones."""
    regs = []
    for o in ops:
        if o is not None and o[0] not in regs:
            regs.append(o[0])

    def sel(pair, want, passthrough=None):
        v = 0
        for i, o in enumerate(want):
            if o is None:
                nb = 0
            elif passthrough is not None and o[0] not in pair:
                nb = passthrough[i]
            else:
                nb = (0 if o[0] == pair[0] else 4) + o[1]
            v |= nb << (4 * i)
        return v

    if len(regs) <= 2:
        pair = (regs + regs + ["0u"])[:2]
        return "cube_prmt(%s, %s, 0x%04xu)" % (pair[0], pair[1], sel(pair, ops)), 1
    if len(regs) == 3:
        # t holds the bytes of regs[0:2] in place, then regs[2] fills the rest
        pair = regs[:2]
        lo = [o if (o is not None and o[0] in pair) else None for o in ops]
        t = "cube_prmt(%s, %s, 0x%04xu)" % (pair[0], pair[1], sel(pair, lo))
        final = 0
        for i, o in enumerate(ops):
            final |= (i if (o is None or o[0] in pair) else 4 + o[1]) << (4 * i)
        return "cube_prmt(%s, %s, 0x%04xu)" % (t, regs[2], final), 2
    lo_pair, hi_pair = regs[:2], regs[2:]
    lo = [o if (o is not None and o[0] in lo_pair) else None for o in ops]
    hi = [o if (o is not None and o[0] in hi_pair) else None for o in ops]
    final = sum(((i if (ops[i] is None or ops[i][0] in lo_pair) else 4 + i) << (4 * i)) for i in range(4))
    return ("cube_prmt(cube_prmt(%s, %s, 0x%04xu), cube_prmt(%s, %s, 0x%04xu), 0x%04xu)"
            % (lo_pair[0], lo_pair[1], sel(lo_pair, lo), hi_pair[0], hi_pair[1], sel(hi_pair, hi), final)), 3


def assemble_row_fn(name, src, first, n_words, half_at, centre_alt=None):
    """Straight-line code for one alignment of a 54-byte row in shared memory: w[j] = stickers
    first+4j .. first+4j+3 and *h = the two stickers half_at, half_at+1 (low 16 bits).
    centre_alt[f] = [(L index, byte), ...]: LUT words that also carry the centre colour of face f; a centre is
    taken from one that the word reads anyway, else from an immediate."""
    def ops_of(positions):
        regs = {src[s_][0] for s_ in positions if s_ is not None and src[s_][0] != "const"}
        out = []
        for s_ in positions:
            if s_ is None:
                out.append(None)
            elif src[s_][0] == "const":
                alt = [a for a in (centre_alt or {}).get(src[s_][1], []) if a[0] in regs]
                out.append(("L[%d]" % alt[0][0], alt[0][1]) if alt else ("0x%02xu" % src[s_][1], 0))
            else:
                out.append(("L[%d]" % src[s_][0], src[s_][1]))
        return out
    lines = ["CUBE_HD void %s(const uint32_t* L, uint32_t* w, uint32_t* h)\n{\n" % name]
    total = 0
    for j in range(n_words):
        e, k = _prmt_expr(ops_of([first + 4 * j + b for b in range(4)]))
        total += k
        lines.append("    w[%d] = %s;\n" % (j, e))
    e, k = _prmt_expr(ops_of([half_at, half_at + 1, None, None]))
    total += k
    lines.append("    *h = %s;\n}   // %d byte permutes\n\n" % (e, total))
    return "".join(lines)


def gather_words_fn(name, moves, n_words):
    """Straight-line code: c = child `a` of the parent row held as words p[]; every child word is a
    byte gather from at most four parent words (compile-time PRMT selectors)."""
    lines = ["template <int A> CUBE_HD void %s(const uint32_t* p, uint32_t* c)\n{\n" % name]
    for a, row in enumerate(moves):
        lines.append("    if (A == %d) {\n" % a)
        for j in range(n_words):
            srcs = [int(row[4 * j + b]) if 4 * j + b < len(row) else 4 * j + b for b in range(4)]
            if srcs == [4 * j + b for b in range(4)]:
                lines.append("        c[%d] = p[%d];\n" % (j, j))
                continue
            words = []
            for s_ in srcs:
                if s_ // 4 not in words:
                    words.append(s_ // 4)
            def pick(pair, want):
                # selector over (pair[0], pair[1]) giving `want` = list of (word, byte) or None per output byte
                sel = 0
                for i, wb in enumerate(want):
                    if wb is None:
                        continue
                    w_, b_ = wb
                    sel |= ((0 if w_ == pair[0] else 4) + b_) << (4 * i)
                return sel
            want = [(s_ // 4, s_ % 4) for s_ in srcs]
            if len(words) <= 2:
                pair = (words + words)[:2]
                lines.append("        c[%d] = cube_prmt(p[%d], p[%d], 0x%04xu);\n" % (j, pair[0], pair[1], pick(pair, want)))
            else:
                lo_pair, hi_pair = words[:2], (words[2:] + words[2:])[:2]
                lo = [wb if wb[0] in lo_pair else None for wb in want]
                hi = [wb if wb[0] not in lo_pair else None for wb in want]
                final = sum(((i if lo[i] is not None else 4 + i) << (4 * i)) for i in range(4))
                lines.append("        c[%d] = cube_prmt(cube_prmt(p[%d], p[%d], 0x%04xu), cube_prmt(p[%d], p[%d], 0x%04xu), 0x%04xu);\n"
                             % (j, lo_pair[0], lo_pair[1], pick(lo_pair, lo), hi_pair[0], hi_pair[1], pick(hi_pair, hi), final))
        lines.append("    }\n")
    lines.append("}\n\n")
    return "".join(lines)


def _c_array(ctype, name, values, per_line=8, fmt="0x%08xu"):
    flat = list(values)
    lines = []
    for i in range(0, len(flat), per_line):
        lines.append("    " + ", ".join(fmt % v for v in flat[i:i + per_line]))
    return "CUBE_TABLE %s %s[%d] = {\n%s\n};\n" % (ctype, name, len(flat), ",\n".join(lines))


def render():
    o = []
    o.append("// GENERATED by csrc/gen_tables.py -- do not edit; run the script instead.\n"
             "// Constant tables of the B200 cube kernels (reference citations are in gen_tables.py).\n"
             "#pragma once\n#include <cstdint>\n\n"
             "// device-resident in .cu translation units, plain host arrays elsewhere (test emulation)\n"
             "#if defined(__CUDACC__)\n#define CUBE_TABLE static __device__ const\n#else\n"
             "#define CUBE_TABLE static const\n#endif\n\n")
    o.append("#define CUBE_MOVE_ROWS %d   // table rows per word: 0..A-1 moves, rest identity\n" % N_MOVE_ROWS)
    o.append("#define CUBE_NOOP_MOVE 12   // identity row used for padded / rejected moves\n")
    o.append("#define CUBE_W3 %d\n#define CUBE_W2 %d\n\n" % (PW3, PW2))
    # fused-scramble move words, layout [word][row]
    t3 = [[packed_words_3(m)[w] for m in range(N_MOVE_ROWS)] for w in range(PW3)]
    t2 = [[packed_words_2(m)[w] for m in range(N_MOVE_ROWS)] for w in range(PW2)]
    o.append("// [word][move] : A = selC0 | selC1 << 16, B = dC0 (dC1 == 2*B mod 3), D = selE0 | selE2 << 16,\n"
             "//                 E = selEt | selE1 << 16, F = fE0 | fE2 << 1\n")
    o.append(_c_array("uint32_t", "kMoveWords3", [v for r in t3 for v in r]))
    o.append("// [word][move] : A = selC0 | selC1 << 16, B = dC0 (dC1 == 2*B mod 3)\n")
    o.append(_c_array("uint32_t", "kMoveWords2", [v for r in t2 for v in r]))
    o.append("#define CUBE_PAIR_BASE %d    // pair row = m0 + CUBE_PAIR_BASE * m1 (m0 first; index 12 = no move)\n" % PAIR_BASE)
    o.append("#define CUBE_PAIR_ROWS %d\n" % PAIR_ROWS)
    o.append("// [row][8]: P = selC0|selC1<<16, T0, T1, F(e0 bit 4 | e2 bit 5); Q = st0|so0<<16, st1|so1<<16, st2|so2<<16, F1\n")
    o.append(_c_array("uint32_t", "kPairWords3", [v for p in range(PAIR_ROWS) for v in pair_words_3(p)]))
    o.append("// [row][4]: selC0|selC1<<16, T0, T1, 0\n")
    o.append(_c_array("uint32_t", "kPairWords2", [v for p in range(PAIR_ROWS) for v in pair_words_2(p)]))
    o.append("// colour LUTs: index = cubie byte (piece | twist << 3 corners; piece | a << 4 | b << 5 edges, flip = a ^ b)\n")
    o.append(_c_array("uint32_t", "kCornerColour3", C_LUT_3))
    o.append(_c_array("uint32_t", "kEdgeColour3", E_LUT_3))
    o.append("// K1p finishing pass: one 32-entry edge LUT per slot, bytes 2 / 3 = the centre colours of the slot's two faces\n")
    o.append(_c_array("uint32_t", "kEdgeColourSlot3", [v for lut in E_LUT_SLOT_3 for v in lut]))
    o.append(_c_array("uint32_t", "kCornerColour2", C_LUT_2))
    src3 = sticker_sources([CORNER_SLOTS_3, EDGE_SLOTS_3], 54, {4 + 9 * f: f for f in range(6)})
    src2 = sticker_sources([CORNER_SLOTS_2], 24, {})
    o.append("// sticker rows from per-slot colour words L[slot] (bytes k = 0..2), generated straight-line\n")
    o.append("#ifdef CUBE_HD\n")
    o.append(assemble_fn("cube_assemble3", src3, 14))
    o.append(assemble_fn("cube_assemble2", src2, 6))
    o.append("// the same row for the two alignments of a 54-byte row on the word grid (K1p): even rows start on\n"
             "// a word (13 words + trailing half), odd rows two bytes later (leading half + 13 words)\n")
    o.append(assemble_row_fn("cube_assemble3_even", src3, 0, 13, 52, CENTRE_ALTERNATIVES_3))
    o.append(assemble_row_fn("cube_assemble3_odd", src3, 2, 13, 0, CENTRE_ALTERNATIVES_3))
    o.append("// sticker positions of 2x2x2 slot `pos` (py222 pieceDefs), usable as compile-time constants\n")
    o.append("CUBE_HD constexpr int cube_piece_def2(int pos, int k)\n{\n    constexpr int t[21] = {%s};\n"
             "    return t[pos * 3 + k];\n}\n\n" % ", ".join(str(v) for r in PIECE_DEFS_2 for v in r))
    o.append("// child A of a 2x2x2 parent row held as six words (new[i] = old[moveDefs[A][i]])\n")
    o.append(gather_words_fn("cube_child2", MOVES_2, 6))
    o.append("#endif\n\n")
    # sticker-level tables
    cyc3 = cycle_words(CYCLES_3)
    cyc2 = cycle_words(CYCLES_2)
    o.append("// sticker 4-cycles per move, bytes (a,b,c,d): new[a]=old[b], new[b]=old[c], new[c]=old[d], new[d]=old[a]\n")
    o.append("// layout [cycle][move row] (rows >= A hold the trivial cycle 0,0,0,0)\n")
    o.append(_c_array("uint32_t", "kCycles3", [(cyc3[m][c] if m < 12 else 0) for c in range(5) for m in range(N_MOVE_ROWS)]))
    o.append(_c_array("uint32_t", "kCycles2", [(cyc2[m][c] if m < 6 else 0) for c in range(3) for m in range(N_MOVE_ROWS)]))
    o.append("// full gather rows new[i] = old[row[i]] ([12][56] / [6][24])\n")
    g3 = [list(MOVES_3[a]) + [54, 55] for a in range(12)]
    g2 = [list(MOVES_2[a]) for a in range(6)]
    o.append(_c_array("uint8_t", "kGather3", [v for r in g3 for v in r], per_line=28, fmt="%d"))
    o.append(_c_array("uint8_t", "kGather2", [v for r in g2 for v in r], per_line=24, fmt="%d"))
    o.append("// one-hot hash definitions: [slot] -> the sticker positions whose colours are hashed\n")
    o.append(_c_array("uint32_t", "kHashDef3", hash_defs_3()))
    o.append(_c_array("uint32_t", "kHashDef2", hash_defs_2()))
    o.append("// hash -> one-hot column (3x3x3, holes = 0 as shipped) / cubelet | ori << 4 (2x2x2)\n")
    o.append(_c_array("uint8_t", "kCornerCol3", CORNER_COL_3, per_line=32, fmt="%d"))
    o.append(_c_array("uint8_t", "kEdgeCol3", EDGE_COL_3, per_line=32, fmt="%d"))
    o.append(_c_array("uint8_t", "kPieceCode2", PIECE_CODE_2, per_line=32, fmt="%d"))
    o.append("// opt-in exact 3x3x3 encoding: un-mirrored slot 6, every corner rotation assigned (gen_tables.py)\n")
    o.append(_c_array("uint32_t", "kHashDef3x", hash_defs_3x()))
    o.append(_c_array("uint8_t", "kCornerCol3x", CORNER_COL_3X, per_line=32, fmt="%d"))
    o.append(_c_array("uint32_t", "kCornerHome3x", CORNER_HOME_3X))
    o.append(_c_array("uint32_t", "kEdgeHome3", EDGE_HOME_3))
    o.append(_c_array("uint8_t", "kStickerSlot3x", STICKER_SLOT_3X, per_line=27, fmt="%d"))
    o.append("// 2x2x2 decode (py222 getStickers): sticker positions of each slot, home colours of each cubelet\n")
    o.append(_c_array("uint8_t", "kPieceDefs2", [v for r in PIECE_DEFS_2 for v in r] + [14, 18, 23], per_line=24, fmt="%d"))
    o.append(_c_array("uint8_t", "kHomeColour2", [v // 4 for r in PIECE_DEFS_2 for v in r] + [3, 4, 5], per_line=24, fmt="%d"))
    o.append("// 2x2x2 distance table (cube_distance.cuh): [move][slot] = source slot | ori added << 4, and\n"
             "// [3 * cubelet + ori] = the colours of the slot's stickers k = 0..2, one per byte\n")
    o.append(_c_array("uint8_t", "kDistMove2", DIST_MOVE_2, per_line=21, fmt="%d"))
    o.append(_c_array("uint32_t", "kCubieColours2", CUBIE_COLOURS_2, per_line=7))
    o.append("// 3x3x3 pattern databases (cube_pattern.cuh): [move][slot] = source slot | ori added << 4, corner slots\n"
             "// 0..7 then edge slots 0..11, in the cubies of the exact encoding\n")
    o.append(_c_array("uint8_t", "kPatMove3", [v for r in PAT_MOVE_3 for v in r], per_line=20, fmt="%d"))
    return "".join(o)


# ---- self-test: emulate the register algorithm against sticker-level gathers --
def prmt(x, y, s):
    b = [(x >> (8 * i)) & 255 for i in range(4)] + [(y >> (8 * i)) & 255 for i in range(4)]
    return sum(b[(s >> (4 * i)) & 7] << (8 * i) for i in range(4))


def emulate_3(seq):
    c0, c1, e0, e1, e2 = 0x03020100, 0x07060504, 0x03020100, 0x07060504, 0x0b0a0908
    for i, m in enumerate(seq):
        A, B, D, E, F = packed_words_3(m)              # exactly what the kernel does
        n0, n1 = prmt(c0, c1, A) + B, prmt(c0, c1, A >> 16) + 2 * B
        if i % 4 == 3:
            n0, n1 = fold_twist(n0), fold_twist(n1)
        assert all(((n >> 8 * k) & 255) >> 3 <= 31 for n in (n0, n1) for k in range(4)) and n0 < 2 ** 32 and n1 < 2 ** 32
        t = prmt(e0, e2, E)
        m0, m2, m1 = prmt(e0, e1, D) ^ (F & 0x10101010), prmt(e2, e1, D >> 16) ^ (F & 0x20202020), prmt(e1, t, E >> 16)
        c0, c1, e0, e1, e2 = n0, n1, m0, m1, m2
    regs = [(c0 >> 8 * i) & 255 for i in range(4)] + [(c1 >> 8 * i) & 255 for i in range(4)]
    regs = [(b & 7) | (((b >> 3) % 3) << 3) for b in regs]
    regs += [(r >> 8 * i) & 255 for r in (e0, e1, e2) for i in range(4)]
    src = sticker_sources([CORNER_SLOTS_3, EDGE_SLOTS_3], 54, {4 + 9 * f: f for f in range(6)})
    out = []
    for s in range(54):
        if src[s][0] == "const":
            out.append(src[s][1])
        else:
            slot, k = src[s]
            lut = C_LUT_3 if slot < 8 else E_LUT_3
            out.append((lut[regs[slot]] >> (8 * k)) & 255)
    return out


def emulate_2(seq):
    c0, c1 = 0x03020100, 0x07060504
    for i, m in enumerate(seq):
        A, B = packed_words_2(m)
        c0, c1 = prmt(c0, c1, A) + B, prmt(c0, c1, A >> 16) + 2 * B
        if i % 4 == 3:
            c0, c1 = fold_twist(c0), fold_twist(c1)
    regs = [(c0 >> 8 * i) & 255 for i in range(4)] + [(c1 >> 8 * i) & 255 for i in range(4)]
    regs = [(b & 7) | (((b >> 3) % 3) << 3) for b in regs]
    src = sticker_sources([CORNER_SLOTS_2], 24, {})
    return [(C_LUT_2[regs[src[s][0]]] >> (8 * src[s][1])) & 255 for s in range(24)]



def emulate_pairs_3(seq):
    """The K1p register algorithm: pairs of moves through pair_words_3, odd tail padded with 12."""
    c0, c1, e0, e1, e2 = 0x03020100, 0x07060504, 0x03020100, 0x07060504, 0x0b0a0908
    seq = list(seq) + [12] * (len(seq) % 2)
    for i in range(0, len(seq), 2):
        P0, T0, T1, F, Q0, Q1, Q2, F1 = pair_words_3(seq[i] + PAIR_BASE * seq[i + 1])
        n0, n1 = prmt(c0, c1, P0) + T0, prmt(c0, c1, P0 >> 16) + T1
        if (i // 2) % 10 == 9:
            n0, n1 = fold_twist(n0), fold_twist(n1)
        assert all(((n >> 8 * k) & 255) >> 3 <= 31 for n in (n0, n1) for k in range(4)) and n0 < 2 ** 32 and n1 < 2 ** 32
        t0, t1, t2 = prmt(e1, e2, Q0), prmt(e0, e2, Q1), prmt(e0, e1, Q2)
        m0 = prmt(e0, t0, Q0 >> 16) ^ (F & 0x10101010)
        m1 = prmt(e1, t1, Q1 >> 16) ^ F1
        m2 = prmt(e2, t2, Q2 >> 16) ^ (F & 0x20202020)
        c0, c1, e0, e1, e2 = n0, n1, m0, m1, m2
    regs = [(c0 >> 8 * i) & 255 for i in range(4)] + [(c1 >> 8 * i) & 255 for i in range(4)]
    regs = [(b & 7) | (((b >> 3) % 3) << 3) for b in regs]
    regs += [(r >> 8 * i) & 255 for r in (e0, e1, e2) for i in range(4)]
    src = sticker_sources([CORNER_SLOTS_3, EDGE_SLOTS_3], 54, {4 + 9 * f: f for f in range(6)})
    out = []
    for s in range(54):
        if src[s][0] == "const":
            out.append(src[s][1])
        else:
            slot, k = src[s]
            lut = C_LUT_3 if slot < 8 else E_LUT_3
            out.append((lut[regs[slot]] >> (8 * k)) & 255)
    return out


def emulate_pairs_2(seq):
    c0, c1 = 0x03020100, 0x07060504
    seq = list(seq) + [12] * (len(seq) % 2)
    for i in range(0, len(seq), 2):
        P0, T0, T1, _ = pair_words_2(seq[i] + PAIR_BASE * seq[i + 1])
        c0, c1 = prmt(c0, c1, P0) + T0, prmt(c0, c1, P0 >> 16) + T1
        if (i // 2) % 10 == 9:
            c0, c1 = fold_twist(c0), fold_twist(c1)
    regs = [(c0 >> 8 * i) & 255 for i in range(4)] + [(c1 >> 8 * i) & 255 for i in range(4)]
    regs = [(b & 7) | (((b >> 3) % 3) << 3) for b in regs]
    src = sticker_sources([CORNER_SLOTS_2], 24, {})
    return [(C_LUT_2[regs[src[s][0]]] >> (8 * src[s][1])) & 255 for s in range(24)]


def selftest(n=300, depth=37):
    rng = np.random.RandomState(0)
    for _ in range(n):
        seq = rng.randint(12, size=depth)
        s = np.repeat(np.arange(6), 9)
        for m in seq:
            s = s[MOVES_3[m]]
        assert list(s) == emulate_3(seq), "3x3x3 cubie model disagrees with sticker gathers"
        assert list(s) == emulate_pairs_3(seq), "3x3x3 pair tables disagree with sticker gathers"
        seq = rng.randint(6, size=depth)
        s = np.repeat(np.arange(6), 4)
        for m in seq:
            s = s[MOVES_2[m]]
        assert list(s) == emulate_2(seq), "2x2x2 cubie model disagrees with sticker gathers"
        assert list(s) == emulate_pairs_2(seq), "2x2x2 pair tables disagree with sticker gathers"
    for _ in range(60):                                   # the no-move index inside a sequence
        for moves, n_act, per_face, emu in ((MOVES_3, 12, 9, emulate_pairs_3), (MOVES_2, 6, 4, emulate_pairs_2)):
            seq = rng.randint(n_act + 1, size=depth)
            seq[seq == n_act] = 12
            s = np.repeat(np.arange(6), per_face)
            for m in seq:
                if m < n_act:
                    s = s[moves[m]]
            assert list(s) == emu(seq), "pair tables mishandle the no-move index"
    # distance-table cubies: a turn through kDistMove2 equals getOP (hash -> kPieceCode2) of the turned stickers,
    # and kCubieColours2 rebuilds the stickers
    for _ in range(n):
        s = np.repeat(np.arange(6), 4)
        codes = list(range(7))
        for m in rng.randint(6, size=depth):
            s = s[MOVES_2[m]]
            codes = [(codes[DIST_MOVE_2[7 * m + q] & 15] & 15)
                     | (((codes[DIST_MOVE_2[7 * m + q] & 15] >> 4) + (DIST_MOVE_2[7 * m + q] >> 4)) % 3) << 4
                     for q in range(7)]
        assert codes == [PIECE_CODE_2[s[d[0]] + 2 * s[d[1]] + 10 * s[d[2]]] for d in PIECE_DEFS_2], \
            "2x2x2 distance cubies disagree with getOP"
        assert all(CUBIE_COLOURS_2[3 * (c & 15) + (c >> 4)] == sum(int(s[d[k]]) << (8 * k) for k in range(3))
                   for c, d in zip(codes, PIECE_DEFS_2)), "kCubieColours2 does not rebuild the stickers"
    # pattern-database cubies: a turn through kPatMove3 equals the exact encoding of the turned stickers
    def exact_cubies(s):
        c = [CORNER_COL_3X[s[d[0]] + 2 * s[d[1]] + 10 * s[d[2]]] for d in CORNER_DEFS_EXACT]
        e = [EDGE_COL_3[s[d[0]] + 10 * s[d[1]]] for d in EDGE_DEFS_REF]
        return [v // 3 | (v % 3) << 4 for v in c] + [v // 2 | (v % 2) << 4 for v in e]
    for _ in range(n):
        s = np.repeat(np.arange(6), 9)
        cub = exact_cubies(s)
        assert cub == list(range(8)) + list(range(12)), "the solved cube must be piece q in slot q, ori 0"
        for m in rng.randint(12, size=depth):
            s = s[MOVES_3[m]]
            row = PAT_MOVE_3[m]
            cub = [(cub[row[q] & 15] & 15) | (((cub[row[q] & 15] >> 4) + (row[q] >> 4)) % 3) << 4 for q in range(8)] + \
                  [(cub[8 + (row[q] & 15)] & 15) | (((cub[8 + (row[q] & 15)] >> 4) + (row[q] >> 4)) % 2) << 4
                   for q in range(8, 20)]
        assert cub == exact_cubies(s), "3x3x3 pattern cubies disagree with the exact encoding"
    # cycles reproduce the gather rows
    for moves, cycles, n_s in ((MOVES_3, CYCLES_3, 54), (MOVES_2, CYCLES_2, 24)):
        for m in range(len(moves)):
            row = list(range(n_s))
            for c in cycles[m]:
                for k in range(4):
                    row[c[k]] = c[(k + 1) % 4]
            assert row == list(moves[m])
    return True


if __name__ == "__main__":
    selftest()
    text = render()
    if "--check" in sys.argv:
        with open(OUT) as f:
            if f.read() != text:
                sys.exit("cube_tables.cuh is stale: run gen_tables.py")
        print("cube_tables.cuh is current; self-test passed")
    else:
        with open(OUT, "w") as f:
            f.write(text)
        print("wrote", OUT)
