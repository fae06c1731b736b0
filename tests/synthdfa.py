"""Generated automata for the scan kernels (TEST INFRASTRUCTURE).

``SynthDfa`` is a complete DFA over letter classes in the reference's numbering; ``image()`` writes it as a
serialised Pire::Scanner (NoShortcuts) that pire_b200/csrc/pire_image.cpp and oracle/pire_oracle.c both read,
and ``walk()`` is a numpy walk of the same table that shares no code with either.  The generator families make
automata a regexp front end does not: state tables above 65 536 states (the u32 complete table), walks that stay
outside the hot rows, one letter or ~258 letters, long and repeated accept lists, absorbing states.

Image layout (pire/scanners/common.h:44-63, multi.h:297-388, mirrored by pire_image.cpp:10-160):
    stream header   magic 0x45524950, version 7, ptr 8, word 16, type 1 (Scanner), header 48
    Locals          states, letters, regexps, initial (byte offset of its row), final table size, relocation 1
                    (Relocatable), shortcutting 0x1000 (NoShortcuts)
    empty flag      8 bytes
    letter table    264 u16: row cell of each character's class (2 header cells + class)
    final table     u64 regexp ids, each accept list closed by ~0
    final index     one u64 per state: where its list starts
    rows            RoundUp(letters + 2, 4) u32 cells: u64 Flags (bit 0 Final, bit 1 Dead), then one int32 byte
                    shift per letter, relative to the row
"""
import struct

import numpy as np

BEGIN_MARK, END_MARK = 258, 259
MAX_CHAR = 264                 # pire/defs.h MaxChar: 260 rounded up to 8
WIDE_STATES = 65536            # more states than this: the complete table is u32 (dfa_tables.cpp BuildScanTables)
_HEADER_CELLS = 2              # NoShortcuts row header: the u64 Flags


def _round_up(v, b):
    return (v + b - 1) // b * b


class SynthDfa:
    """next[states, letters] (u32), class_of[260] (bytes 0..255, 256 unused, 257 Epsilon = 0, BeginMark, EndMark),
    initial, accept[state] = list of regexp ids (final <=> non-empty), dead = non-final and every letter loops back."""

    def __init__(self, name, next_, class_of, initial, accept, regexps):
        self.name = name
        self.next = np.ascontiguousarray(next_, dtype=np.uint32)
        self.states, self.letters = self.next.shape
        self.class_of = np.asarray(class_of, dtype=np.int64)
        assert self.class_of.shape == (260,) and self.class_of.min() >= 0 and self.class_of.max() < self.letters
        assert self.class_of[257] == 0
        assert int(self.next.max()) < self.states and 0 <= initial < self.states
        self.initial = int(initial)
        self.accept = accept                       # dict state -> list of ids; absent = empty
        self.regexps = int(regexps)
        self.final = np.zeros(self.states, bool)
        for s, ids in accept.items():
            self.final[s] = len(ids) > 0
        loops = (self.next == np.arange(self.states, dtype=np.uint32)[:, None]).all(axis=1)
        self.dead = loops & ~self.final
        self.mask = np.zeros(self.states, np.uint32)
        for s, ids in accept.items():
            for i in ids:
                if i < 32:
                    self.mask[s] |= np.uint32(1 << i)
        self._flat = self.next.reshape(-1)

    def __repr__(self):
        return "SynthDfa(%s: %d states, %d letters, %d regexps)" % (self.name, self.states, self.letters, self.regexps)

    @property
    def wide(self):
        return self.states > WIDE_STATES

    def step(self, states, ch):
        """Next state of each of `states` on character `ch` (a byte or a mark)."""
        return self._flat[np.asarray(states, np.int64) * self.letters + self.class_of[ch]]

    # --------------------------------------------------------------------- image
    def image(self):
        S, L = self.states, self.letters
        row_cells = _round_up(L + _HEADER_CELLS, 4)
        row_bytes = row_cells * 4
        assert S * row_bytes < 2 ** 31, "byte shifts are int32"
        # accept lists: one shared empty list at 0, then one list per final state
        final_tab = [~0 & 0xFFFFFFFFFFFFFFFF]
        final_idx = np.zeros(S, np.uint64)
        for s in sorted(self.accept):
            ids = self.accept[s]
            if ids:
                final_idx[s] = len(final_tab)
                final_tab.extend(int(i) for i in ids)
                final_tab.append(0xFFFFFFFFFFFFFFFF)
        head = struct.pack("<6I", 0x45524950, 7, 8, 16, 1, 48)
        head += struct.pack("<4IQ2I2Q", S, L, self.regexps, 0, self.initial * row_bytes, len(final_tab), 0, 1, 0x1000)
        head += b"\0" * 8                                                # not empty
        cols = np.full(MAX_CHAR, _HEADER_CELLS, np.uint16)
        cols[:260] = self.class_of + _HEADER_CELLS
        rows = np.zeros((S, row_cells), np.uint32)
        flags = self.final.astype(np.uint32) | (self.dead.astype(np.uint32) << 1)
        rows[:, 0] = flags
        shift = (self.next.astype(np.int64) - np.arange(S, dtype=np.int64)[:, None]) * row_bytes
        rows[:, _HEADER_CELLS:_HEADER_CELLS + L] = shift.astype(np.int32).view(np.uint32)
        return b"".join([head, cols.tobytes(), np.array(final_tab, np.uint64).tobytes(), final_idx.tobytes(),
                         rows.tobytes()])

    # ---------------------------------------------------------------------- walk
    def walk(self, corpus, offsets=None, fixed_len=0, n=None, begin=True, end=True, track_max=False):
        """Runner(sc).[Begin()].Run(s).[End()] per string: (final[n] bool, mask[n] u32 of ids < 32, state[n] u32),
        plus the largest state each walk entered when `track_max`.  Strings of one length step together, one numpy
        gather per position; long strings are walked one by one."""
        corpus = np.asarray(corpus, np.uint8)
        if offsets is None:
            n = len(corpus) // fixed_len if n is None else n
            starts = np.arange(n, dtype=np.int64) * fixed_len
            lens = np.full(n, fixed_len, np.int64)
        else:
            offsets = np.asarray(offsets, np.int64)
            n = len(offsets) - 1 if n is None else n
            starts, lens = offsets[:n], offsets[1:n + 1] - offsets[:n]
        st = np.full(n, self.initial, np.int64)
        if begin:
            st = self.step(st, BEGIN_MARK).astype(np.int64)
        top = st.copy()
        cls = self.class_of[:256]
        L, flat = self.letters, self._flat
        long_ = lens > 4096
        order = np.argsort(-np.where(long_, 0, lens), kind="stable")
        order = order[~long_[order]]
        olen = lens[order]
        for p in range(int(olen[0]) if len(olen) else 0):
            k = int(np.searchsorted(-olen, -p, side="left"))        # strings longer than p lead the order
            idx = order[:k]
            st[idx] = flat[st[idx] * L + cls[corpus[starts[idx] + p]]]
            if track_max:
                top[idx] = np.maximum(top[idx], st[idx])
        clsl = cls.tolist()
        for i in np.nonzero(long_)[0]:
            s, hi = int(st[i]), int(top[i])
            for b in corpus[starts[i]:starts[i] + lens[i]].tolist():
                s = flat.item(s * L + clsl[b])
                if s > hi:
                    hi = s
            st[i], top[i] = s, hi
        if end:
            st = self.step(st, END_MARK).astype(np.int64)
            top = np.maximum(top, st)
        out = (self.final[st], self.mask[st], st.astype(np.uint32))
        return out + (top,) if track_max else out


def _class_table(letters, rng, marks=None):
    """Bytes spread over `letters` classes (each class gets at least one byte while there are bytes enough); the
    marks get `marks` = (begin class, end class) or random classes."""
    cls = np.zeros(260, np.int64)
    if letters == 258:                               # every byte and both marks a letter of their own
        cls[:256] = rng.permutation(256)
        cls[BEGIN_MARK], cls[END_MARK] = 256, 257
        return cls
    assert letters < 258
    perm = rng.permutation(256)
    cls[perm] = np.arange(256) % letters
    cls[256] = 0
    if marks is None:
        marks = rng.integers(0, letters, 2)
    cls[BEGIN_MARK], cls[END_MARK] = marks
    return cls


def _accept_lists(final_states, rng, regexps, shape="plain"):
    acc = {}
    for s in final_states.tolist():
        if shape == "many":          # long lists of distinct ids, up to `regexps` (64) of them
            k = int(rng.integers(1, regexps + 1))
            acc[s] = sorted(rng.choice(regexps, k, replace=False).tolist())
        elif shape == "repeat":      # one id listed 16..20 times (turns packed counting off)
            r = int(rng.integers(0, regexps))
            acc[s] = [r] * int(rng.integers(16, 21)) + sorted(rng.choice(regexps, 2).tolist())
        else:
            acc[s] = sorted(set(rng.choice(regexps, int(rng.integers(1, 4))).tolist()))
    return acc


def shift_register(k):
    """"The (k+1)-th byte from the end is `a`" over {a, b}, as (a|b)*a(a|b){k} determinises: 2^(k+1) register
    states (the last k+1 bytes, newest in bit 0, initial = all b) plus one dead state for any other byte.  The marks
    loop.  Closed form: final <=> only a/b bytes, length > k, and byte len-k-1 is `a`."""
    R = 1 << (k + 1)
    dead = R
    nxt = np.empty((R + 1, 4), np.uint32)
    r = np.arange(R, dtype=np.uint32)
    nxt[:R, 0] = ((r << 1) | 1) & (R - 1)         # a
    nxt[:R, 1] = (r << 1) & (R - 1)               # b
    nxt[:R, 2] = dead                             # any other byte
    nxt[:R, 3] = r                                # marks
    nxt[dead] = dead
    cls = np.full(260, 2, np.int64)
    cls[ord("a")], cls[ord("b")] = 0, 1
    cls[256] = cls[257] = 0
    cls[BEGIN_MARK] = cls[END_MARK] = 3
    acc = {int(s): [0] for s in np.nonzero(r >> k & 1)[0]}
    return SynthDfa("shift_register(%d)" % k, nxt, cls, 0, acc, 1)


def shift_register_answer(k, strings):
    """The closed form of shift_register(k) for a list of byte strings."""
    return np.array([len(s) > k and s[len(s) - k - 1] == ord("a") and not s.strip(b"ab") for s in strings], bool)


def ring(N, seed=0, regexps=64):
    """A ring of N states: letter 0 steps i -> i+1, letters 1 and 2 jump by a hash, letter 3 jumps into the top 512
    states (so walks end deep in the high ids even when only a few states lie above 65 535), the marks step by 7 and
    11.  About a ninth of the states are final with 1..3 of `regexps` ids (ids >= 32 included)."""
    rng = np.random.default_rng(seed)
    i = np.arange(N, dtype=np.int64)
    nxt = np.empty((N, 6), np.uint32)
    nxt[:, 0] = (i + 1) % N
    nxt[:, 1] = (i * 40503 + 17) % N
    nxt[:, 2] = (i * 2654435761 + 99991) % N
    nxt[:, 3] = N - 1 - (i * 97 + 5) % min(N, 512)
    nxt[:, 4] = (i + 7) % N
    nxt[:, 5] = (i + 11) % N
    cls = _class_table(4, rng, marks=(4, 5))
    finals = np.nonzero((i * 2654435761 >> 7) % 9 == 0)[0]
    return SynthDfa("ring(%d)" % N, nxt, cls, 0, _accept_lists(finals, rng, regexps), regexps)


def search(states, letters=24, seed=0, regexps=8):
    """A search automaton: state 0 keeps most bytes (letter 0); the other letters lead from it into states 1..letters-1,
    which go on through hashed transitions anywhere in the table and fall back to 0 on letter 0.  Every exit of the
    resting state is hot, so the look-ahead filter applies.  State `states-1` is a final absorbing state and
    `states-2` a dead one, both reached from state 1 on the last letter."""
    rng = np.random.default_rng(seed)
    nxt = rng.integers(1, states, (states, letters)).astype(np.uint32)
    nxt[:, 0] = 0
    nxt[0, 1:] = np.arange(1, letters)
    nxt[0, 0] = 0
    nxt[1, letters - 1] = states - 1
    nxt[2, letters - 1] = states - 2
    nxt[states - 1] = states - 1
    nxt[states - 2] = states - 2
    cls = np.zeros(260, np.int64)
    per = max(1, min(4, 128 // (letters - 1)))
    trig = rng.choice(256, per * (letters - 1), replace=False)
    cls[trig] = 1 + np.arange(per * (letters - 1)) % (letters - 1)   # up to four bytes per trigger letter, the rest 0
    cls[BEGIN_MARK], cls[END_MARK] = 0, int(rng.integers(1, letters))
    finals = np.nonzero(rng.random(states) < 0.2)[0]
    finals = finals[(finals != 0) & (finals != states - 2)]
    acc = _accept_lists(np.append(finals, states - 1), rng, regexps)
    return SynthDfa("search(%d,%d)" % (states, letters), nxt, cls, 0, acc, regexps)


def dense_random(states, letters, seed=0, regexps=8, accept="plain", final_share=0.3, absorbing=0):
    """Uniform random transitions over every state: most steps are cold, the look-ahead set is incomplete.
    `absorbing` states loop on every letter (half of them final, the others dead)."""
    rng = np.random.default_rng(seed)
    nxt = rng.integers(0, states, (states, letters)).astype(np.uint32)
    cls = _class_table(letters, rng)
    final = rng.random(states) < final_share
    if absorbing:
        ab = rng.choice(np.arange(1, states), min(absorbing, states - 1), replace=False)
        nxt[ab] = ab[:, None]
        final[ab[: len(ab) // 2]] = True
        final[ab[len(ab) // 2:]] = False
    acc = _accept_lists(np.nonzero(final)[0], rng, regexps, accept)
    return SynthDfa("dense_random(%d,%d,%s)" % (states, letters, accept), nxt, cls, int(rng.integers(0, states)), acc,
                    regexps)


def from_host_scanner(sc, name="host"):
    """Rebuild a SynthDfa from a host Scanner handle's Next / AcceptedRegexps: characters whose columns agree over all
    states share a letter.  Used to check the writer against images the reference wrote."""
    info = sc.info()
    S = info.states
    chars = list(range(256)) + [256, BEGIN_MARK, END_MARK]
    cols = np.array([[sc.Next(s, c) for c in chars] for s in range(S)], np.uint32)   # [S, 259]
    uniq, inv = np.unique(cols.T, axis=0, return_inverse=True)
    cls = np.zeros(260, np.int64)
    cls[chars] = inv.reshape(-1)
    acc = {s: sc.AcceptedRegexps(s) for s in range(S) if sc.Final(s)}
    return SynthDfa(name, uniq.T, cls, sc.Initialize(), acc, info.regexps)
