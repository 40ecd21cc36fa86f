"""A DEFLATE bit writer for tests: hand-built streams whose every field can be set from outside, including the ones no
encoder writes (BTYPE 3, litlen 286/287, distance 30/31, incomplete / over-subscribed / Q5-shaped code tables, repeat
codes across the litlen/dist boundary and past the end, stored LEN/NLEN mismatches, data after the final block).

    s = write([dynamic(cat(lits(b"abc"), match(258, 3, lsym=284, lx=31)), final=True)])
    s.data        the bytes
    s.offsets     bit offset of every litlen symbol (per Huffman block, in stream order)
    s.expect(cap) ("good" | "fail" | "ub", bytes): what the reference does with it (rules Q2, Q3, Q5, inflate.c:1809,
                  :1843, :826/:836, LEN/NLEN); "ub" = undefined behaviour in the reference (over-subscribed code, 286/287,
                  a repeat with no predecessor, reading past the input, output overflow): every decoder must fail there.

Bits are packed vectorised: one uint64 value and a bit count per symbol, a cumsum of positions, two ORs into a word
array. Plain Python + numpy; test scaffolding only.
"""
import heapq
from dataclasses import dataclass

import numpy as np

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_XB = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_XB = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
HOLE = -2  # a litlen "symbol" that writes the canonical hole of an incomplete code (the stream hits an unassigned code)

_LXB = np.array(LEN_XB + [6, 6, 0], np.int64)      # 286/287: the 6 extra bits a decoder that extended the length table would read
_DXB = np.array(DIST_XB + [0, 0], np.int64)        # 30/31 likewise
_LSYM = np.zeros(259, np.int64)
for _s in range(28, -1, -1):
    _LSYM[LEN_BASE[_s]:] = np.where(_LSYM[LEN_BASE[_s]:] == 0, 257 + _s, _LSYM[LEN_BASE[_s]:])
_LSYM[258] = 285
_DBASE = np.array(DIST_BASE, np.int64)


def fixed_litlen_lengths():
    return [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8


# ----------------------------------------------------------------------------------------------------- codes ----
def canonical(lengths):
    """RFC 1951 3.2.2 codes for any set of lengths -- incomplete and over-subscribed sets too (codes of an
    over-subscribed set simply run past 2^len and are taken modulo it)."""
    lengths = [int(x) for x in lengths]
    bl = [0] * 17
    for x in lengths:
        bl[x] += 1
    bl[0] = 0
    nxt, code = [0] * 17, 0
    for b in range(1, 17):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    out = [0] * len(lengths)
    for s, x in enumerate(lengths):
        if x:
            out[s] = nxt[x] & ((1 << x) - 1)
            nxt[x] += 1
    return out


def kraft(lengths):
    """Kraft sum in units of 2^-15: 32768 = complete, less = incomplete, more = over-subscribed."""
    return sum(1 << (15 - int(x)) for x in lengths if x)


def q5_range(lengths):
    """(min, max) lengths the reference probes (inflate.c:528-539: the first non-zero length sets only the minimum,
    and later ones update the maximum only when they do not lower the minimum)."""
    mn, mx = 9999, 1
    for x in lengths:
        if not x:
            continue
        if x < mn:
            mn = x
        elif x > mx:
            mx = x
    return mn, mx


def rev(v, n):
    return int(format(v, "0%db" % n)[::-1], 2) if n else 0


def limited_lengths(freqs, limit=15):
    """Length-limited Huffman code lengths (package-merge) for the symbols with non-zero frequency; a lone symbol gets 1."""
    syms = [s for s, f in enumerate(freqs) if f]
    out = [0] * len(freqs)
    if len(syms) == 1:
        out[syms[0]] = 1
        return out
    leaves = sorted((int(freqs[s]), [s]) for s in syms)
    cur = list(leaves)
    for _ in range(limit - 1):
        pk = [(cur[i][0] + cur[i + 1][0], cur[i][1] + cur[i + 1][1]) for i in range(0, len(cur) - 1, 2)]
        cur = list(heapq.merge(leaves, pk, key=lambda t: t[0]))
    for _, members in cur[: 2 * len(syms) - 2]:
        for s in members:
            out[s] += 1
    return out


# ---------------------------------------------------------------------------------------------------- tokens ----
@dataclass
class Tokens:
    """A run of symbols of one Huffman block: litlen symbol (HOLE for an unassigned code), its extra-bit value,
    distance symbol (-1: none) and its extra-bit value."""
    sym: np.ndarray
    lx: np.ndarray
    dsym: np.ndarray
    dx: np.ndarray

    def __len__(self):
        return len(self.sym)


def _tok(sym, lx=None, dsym=None, dx=None):
    sym = np.asarray(sym, np.int64).reshape(-1)
    z = np.zeros(len(sym), np.int64)
    return Tokens(sym, z if lx is None else np.asarray(lx, np.int64).reshape(-1),
                  z - 1 if dsym is None else np.asarray(dsym, np.int64).reshape(-1),
                  z if dx is None else np.asarray(dx, np.int64).reshape(-1))


def lits(data):
    return _tok(np.frombuffer(bytes(data), np.uint8).astype(np.int64))


def matches(lengths, dists):
    """(len, dist) pairs with the usual symbol choice (vectorised)."""
    L = np.asarray(lengths, np.int64).reshape(-1)
    D = np.asarray(dists, np.int64).reshape(-1)
    ls = _LSYM[L]
    ds = np.searchsorted(_DBASE, D, side="right") - 1
    return _tok(ls, L - np.array(LEN_BASE, np.int64)[ls - 257], ds, D - _DBASE[ds])


def match(length, dist, lsym=None, lx=None):
    """One match; `lsym`/`lx` pick the length symbol explicitly (258 = 284 + 31 or 285)."""
    t = matches([length], [dist])
    if lsym is not None:
        t.sym[0], t.lx[0] = lsym, (length - LEN_BASE[lsym - 257] if lx is None else lx)
    return t


def raw(sym, lx=0, dsym=-1, dx=0):
    """A raw symbol: litlen 286/287, or a length symbol with distance symbol 30/31."""
    return _tok([sym], [lx], [dsym], [dx])


def hole():
    return _tok([HOLE])


def cat(*ts):
    ts = [t for t in ts if len(t)]
    if not ts:
        return _tok([])
    return Tokens(*(np.concatenate([getattr(t, f) for t in ts]) for f in ("sym", "lx", "dsym", "dx")))


def token_out_len(t):
    """Output bytes of every token (0 for symbols that do not produce any)."""
    n = np.where((t.sym >= 0) & (t.sym < 256), 1, 0)
    m = (t.sym >= 257) & (t.sym <= 285)
    n[m] = np.array(LEN_BASE, np.int64)[t.sym[m] - 257] + t.lx[m]
    n[t.sym == HOLE] = 0
    return n


# ---------------------------------------------------------------------------------------------------- blocks ----
@dataclass
class Block:
    btype: int
    final: bool = False
    tokens: Tokens = None
    eob: bool = True
    data: bytes = b""
    stored_len: int = None
    stored_nlen: int = None
    lit_lens: list = None
    dist_lens: list = None
    hlit: int = None
    hdist: int = None
    hclen: int = None
    cl_lens: list = None
    plan: list = None


def stored(data, final=False, len_=None, nlen=None):
    return Block(0, final, data=bytes(data), stored_len=len_, stored_nlen=nlen)


def fixed(tokens, final=False, eob=True):
    return Block(1, final, tokens=tokens, eob=eob)


def btype3(final=False):
    return Block(3, final)


def dynamic(tokens, final=False, eob=True, lit_lens=None, dist_lens=None, hlit=None, hdist=None, hclen=None,
            cl_lens=None, plan=None):
    """A dynamic block. Code lengths are explicit, or length-limited (<= 15) from the tokens' frequencies. `plan` is an
    explicit code-length sequence: a list of (symbol, repeat count) with symbol 0-15 (count ignored) or 16/17/18;
    when given, the lengths are what the plan decodes to (it may run across the litlen/dist boundary or past the end)."""
    return Block(2, final, tokens=tokens, eob=eob, lit_lens=lit_lens, dist_lens=dist_lens, hlit=hlit, hdist=hdist,
                 hclen=hclen, cl_lens=cl_lens, plan=plan)


def rle_plan(lens):
    """The usual code-length sequence: 16 repeats the previous length 3-6 times, 17/18 write 3-10 / 11-138 zeros."""
    plan, i, n = [], 0, len(lens)
    while i < n:
        v, j = lens[i], i
        while j < n and lens[j] == v:
            j += 1
        run = j - i
        if v == 0:
            while run >= 11:
                k = min(run, 138)
                plan.append((18, k))
                run -= k
            if run >= 3:
                plan.append((17, run))
                run = 0
            plan += [(0, 1)] * run
        else:
            plan.append((v, 1))
            run -= 1
            while run >= 3:
                k = min(run, 6)
                plan.append((16, k))
                run -= k
            plan += [(v, 1)] * run
        i = j
    return plan


def plan_lengths(plan, total):
    """What a plan decodes to: (lengths[:total], ub) -- ub when a 16 comes first (the reference reads table[-1])."""
    out = []
    for s, k in plan:
        if len(out) >= total:
            break
        if s <= 15:
            out.append(s)
        elif s == 16:
            if not out:
                return None, True
            out += [out[-1]] * k
        else:
            out += [0] * k
    return out[:total], False


# ------------------------------------------------------------------------------------------------- the stream ----
class _Bits:
    def __init__(self):
        self.vals, self.nbits, self.pos = [], [], 0

    def add(self, vals, nbits):
        vals = np.asarray(vals, np.uint64).reshape(-1)
        nbits = np.asarray(nbits, np.int64).reshape(-1)
        self.vals.append(vals)
        self.nbits.append(nbits)
        start = self.pos + np.concatenate([[0], np.cumsum(nbits)[:-1]]) if len(nbits) else np.zeros(0, np.int64)
        self.pos += int(nbits.sum())
        return start

    def pack(self, tail=b""):
        v = np.concatenate(self.vals) if self.vals else np.zeros(0, np.uint64)
        n = np.concatenate(self.nbits) if self.nbits else np.zeros(0, np.int64)
        keep = n > 0
        v, n = v[keep], n[keep]
        p = np.concatenate([[0], np.cumsum(n)[:-1]]).astype(np.int64)
        words = np.zeros((self.pos + 127) // 64 + 1, np.uint64)
        sh = (p & 63).astype(np.uint64)
        np.bitwise_or.at(words, p >> 6, v << sh)
        hi = (sh + n.astype(np.uint64)) > 64
        np.bitwise_or.at(words, (p >> 6)[hi] + 1, v[hi] >> (np.uint64(64) - sh[hi]))
        return words.astype("<u8").tobytes()[: (self.pos + 7) // 8] + bytes(tail)


@dataclass
class Stream:
    data: bytes
    blocks: list
    offsets: list        # per Huffman block: bit offset of every litlen symbol (EOB included)
    plans: list          # per block: what the decoder meets, in order (see expect)
    spec_valid: bool     # zlib must decode it to the intended output
    end_bits: int = 0

    def expect(self, cap=None, in_size=None):
        return expect(self, cap, in_size)

    @property
    def max_out(self):
        """Output bytes of every symbol and stored byte written (an upper bound of what a decoder produces)."""
        return sum(int(token_out_len(p[4]).sum()) if p[0] == "huff" else len(p[6]) if p[0] == "stored" else 0
                   for p in self.plans)

    @property
    def output(self):
        return self.expect(1 << 40)[1]


def _code_of(sym, codes, lens):
    return rev(codes[sym], lens[sym]), lens[sym]


def write(blocks, tail=b""):
    """Writes the blocks (and `tail` after them) and returns a Stream."""
    B = _Bits()
    offsets, plans = [], []
    spec_valid = not tail
    for bk in blocks:
        hdr_at = B.pos
        B.add([int(bk.final) | (bk.btype << 1)], [3])
        if bk.btype == 3:
            plans.append(("btype3", hdr_at, bk.final))
            spec_valid = False
            continue
        if bk.btype == 0:
            B.add([0], [(-B.pos) & 7])
            ln = len(bk.data) if bk.stored_len is None else bk.stored_len
            nl = (~ln & 0xFFFF) if bk.stored_nlen is None else bk.stored_nlen
            B.add([ln, nl], [16, 16])
            at = B.pos // 8
            B.add(np.frombuffer(bk.data, np.uint8), np.full(len(bk.data), 8))
            plans.append(("stored", hdr_at, bk.final, ln, nl, at, bk.data))
            spec_valid &= ln == len(bk.data) and nl == (~ln & 0xFFFF)
            continue
        t = bk.tokens if bk.tokens is not None else _tok([])
        if bk.eob:
            t = cat(t, _tok([256]))
        header_verdict = "ok"
        if bk.btype == 1:
            ll, dl, hlit, hdist = fixed_litlen_lengths(), [5] * 32, 288, 32
        else:
            ll, dl = bk.lit_lens, bk.dist_lens
            if ll is None:
                f = np.bincount(t.sym[t.sym >= 0], minlength=286)[:286]
                f[256] = max(f[256], 1)
                ll = limited_lengths(f, 15)
            if dl is None:
                used = t.dsym[t.dsym >= 0]
                if len(used):
                    f = np.bincount(used, minlength=30)[:30]
                    dl = limited_lengths(f, 15)
                    if sum(1 for x in dl if x) == 1:  # a lone code is 1 bit long: HDIST >= 2 keeps it clear of rule Q3
                        dl = dl + [0] if len(dl) < 2 else dl
                else:
                    dl = [0]
            ll, dl = list(ll), list(dl)
            hlit = bk.hlit if bk.hlit is not None else max(257, max(s for s, x in enumerate(ll) if x) + 1)
            nzd = [s for s, x in enumerate(dl) if x]
            hdist = bk.hdist if bk.hdist is not None else max(1, (nzd[-1] + 1) if nzd else 1, len(dl) if len(nzd) == 1 else 1)
            ll = (ll + [0] * 288)[:hlit]
            dl = (dl + [0] * 32)[:hdist]
            plan = bk.plan if bk.plan is not None else rle_plan(ll + dl)
            if bk.plan is not None:
                got, ub16 = plan_lengths(plan, hlit + hdist)
                if ub16:
                    header_verdict = "ub"
                else:
                    got += [0] * (hlit + hdist - len(got))
                    ll, dl = got[:hlit], got[hlit:]
            if bk.cl_lens is not None:
                cll = list(bk.cl_lens)
            else:
                f = [0] * 19
                for s, _ in plan:
                    f[s] += 1
                cll = limited_lengths(f, 7)
            need = max([k + 1 for k, s in enumerate(CL_ORDER) if cll[s]] + [4])
            hclen = bk.hclen if bk.hclen is not None else need
            cll = [cll[s] if CL_ORDER.index(s) < hclen else 0 for s in range(19)]
            B.add([hlit - 257, hdist - 1, hclen - 4], [5, 5, 4])
            B.add([cll[CL_ORDER[k]] for k in range(hclen)], [3] * hclen)
            clc = canonical(cll)
            mn, mx = q5_range(cll)
            if header_verdict == "ok" and kraft(cll) > 32768:
                header_verdict = "ub"
            vals, nb = [], []
            for s, k in plan:
                c, n = _code_of(s, clc, cll)
                if header_verdict == "ok" and not (cll[s] and mn <= cll[s] <= mx):
                    header_verdict = "fail"                    # a code-length symbol the reference cannot decode
                xb = {16: 2, 17: 3, 18: 7}.get(s, 0)
                xv = {16: k - 3, 17: k - 3, 18: k - 11}.get(s, 0)
                vals.append(c | (xv << n))
                nb.append(n + xb)
            B.add(vals, nb)
            if header_verdict == "ok":
                if kraft(ll) > 32768:
                    header_verdict = "ub"
                elif any(x >= hdist for x in dl):
                    header_verdict = "fail"                    # rule Q3 (inflate.c:599-602)
                elif kraft(dl) > 32768:
                    header_verdict = "ub"
            spec_valid &= hlit <= 286 and hdist <= 30 and bk.plan is None and header_verdict == "ok"
            spec_valid &= kraft(ll) == 32768 or (sum(1 for x in ll if x) == 1 and max(ll) == 1)
            spec_valid &= kraft(dl) == 32768 or max(dl) <= 1
        # symbols
        lc = canonical(ll)
        dc = canonical(dl)                                  # (fixed: 5-bit codes equal to the symbol)
        llen = np.array(ll + [0] * (288 - len(ll)), np.int64)
        dlen = np.array(dl + [0] * (32 - len(dl)), np.int64)
        lcode = np.array([rev(c, x) for c, x in zip(lc + [0] * (288 - len(lc)), llen)], np.uint64)
        dcode = np.array([rev(c, x) for c, x in zip(dc + [0] * (32 - len(dc)), dlen)], np.uint64)
        # the canonical hole of an incomplete litlen code: the first code of the longest length past the assigned ones
        K = max(int(x) for x in llen) if llen.any() else 1
        hole_code = rev((sum(1 << (K - int(x)) for x in llen if x)) & ((1 << K) - 1), K)
        s = t.sym.copy()
        is_hole = s == HOLE
        s[is_hole] = 0
        c = np.where(is_hole, np.uint64(hole_code), lcode[s])
        n = np.where(is_hole, K, llen[s])
        lxb = np.where((s >= 257) & ~is_hole, _LXB[np.clip(s - 257, 0, 31)], 0)
        hasd = (t.dsym >= 0) & (s >= 257) & ~is_hole       # (286/287 with distance bits behind: how a decoder that took them
                                                            # for lengths would go on)
        ds = np.clip(t.dsym, 0, 31)
        dn = np.where(hasd, dlen[ds], 0)
        dxb = np.where(hasd, _DXB[ds], 0)
        val = c | (t.lx.astype(np.uint64) << n.astype(np.uint64))
        val |= np.where(hasd, dcode[ds], 0).astype(np.uint64) << (n + lxb).astype(np.uint64)
        val |= np.where(hasd, t.dx, 0).astype(np.uint64) << (n + lxb + dn).astype(np.uint64)
        offs = B.add(val, n + lxb + dn + dxb)
        offsets.append(offs)
        lmn, lmx = q5_range(ll)
        dmn, dmx = q5_range(dl) if bk.btype == 2 else (5, 5)
        plans.append(("huff", hdr_at, bk.final, header_verdict, t, offs, (llen, lmn, lmx), (dlen, dmn, dmx), bk.eob, B.pos))
        spec_valid &= header_verdict == "ok" and bk.eob
    end_bits = B.pos
    if not blocks or not blocks[-1].final:
        spec_valid = False
    return Stream(B.pack(tail), blocks, offsets, plans, bool(spec_valid), end_bits)


# ------------------------------------------------------------------------------------- what the reference does ----
def _expand(out, t, upto):
    """LZ77 expansion of the first `upto` tokens of t onto bytearray `out`."""
    sym = t.sym[:upto].tolist()
    ln = token_out_len(Tokens(t.sym[:upto], t.lx[:upto], t.dsym[:upto], t.dx[:upto])).tolist()
    ds = t.dsym[:upto].tolist()
    dx = t.dx[:upto].tolist()
    i = 0
    while i < upto:
        if sym[i] < 256:
            j = i
            while j < upto and sym[j] < 256:
                j += 1
            out += bytes(sym[i:j])
            i = j
            continue
        if sym[i] != 256:
            L, D = ln[i], DIST_BASE[ds[i]] + dx[i]
            if D >= L:
                out += out[len(out) - D: len(out) - D + L]
            else:
                pat = out[len(out) - D:]
                out += (pat * (L // D + 1))[:L]
        i += 1


def expect(s, cap=None, in_size=None):
    """(verdict, bytes) of the reference on s.data[:in_size] with output capacity cap."""
    n = len(s.data) if in_size is None else in_size
    cap = (1 << 40) if cap is None else cap
    if cap < n or n < 5:
        return "fail", b""                                   # inflate.c:826 / :836
    out = bytearray()
    for p in s.plans:
        kind, hdr_at, final = p[0], p[1], p[2]
        if hdr_at >= 8 * n:
            return "ub", b""                                 # the reference would read the next header past the input
        if kind == "btype3":
            if final:
                return "good", bytes(out)
            continue
        if kind == "stored":
            _, _, _, ln, nl, at, data = p
            if ln != (~nl & 0xFFFF):
                return "fail", b""                           # inflate.c:949
            if at + ln > n or ln > len(data):
                return "ub", b""
            if len(out) + ln > cap:
                return "ub", b""
            out += data[:ln]
            if final:
                return "good", bytes(out)
            continue
        _, _, _, hv, t, offs, (llen, lmn, lmx), (dlen, dmn, dmx), eob, blk_end = p
        if hv != "ok":
            return hv, b""
        if not eob:  # the decoder goes on past the written tokens: rule Q2 ends it there, or it reads what follows
            t = cat(t, _tok([HOLE if lmn > lmx or not llen.any() else -3]))
            offs = np.concatenate([offs, [blk_end]])
        q2 = offs > 8 * (n - 1)                              # rule Q2: ceil(bits / 8) >= size before a litlen symbol
        sym = t.sym
        sl = np.where(sym < 0, 0, llen[np.clip(sym, 0, 287)])
        bad_l = (sym == HOLE) | ((sym >= 0) & ((sl == 0) | (sl < lmn) | (sl > lmx)))
        ub_l = ~bad_l & (sym > 285)
        ism = ~bad_l & (sym >= 257) & (sym <= 285)
        dsy = np.clip(t.dsym, 0, 31)
        dl = dlen[dsy]
        bad_d = ism & ((t.dsym < 0) | (dl == 0) | (dl < dmn) | (dl > dmx) | (t.dsym > 29))
        olen = token_out_len(t)
        pos = len(out) + np.concatenate([[0], np.cumsum(olen)[:-1]]).astype(np.int64)
        dist = np.where(ism & ~bad_d, _DBASE[np.clip(t.dsym, 0, 29)] + t.dx, 0)
        bad_dist = ism & ~bad_d & (dist > pos)
        over = ((sym >= 0) & (sym < 256) & (pos >= cap)) | (ism & ~bad_d & ~bad_dist & (pos + olen > cap))
        ev = [(np.argmax(q2) if q2.any() else 1 << 62, 0, "q2"),
              (np.argmax(bad_l) if bad_l.any() else 1 << 62, 1, "fail"),
              (np.argmax(ub_l) if ub_l.any() else 1 << 62, 1, "ub"),
              (np.argmax(bad_d) if bad_d.any() else 1 << 62, 1, "fail"),
              (np.argmax(bad_dist) if bad_dist.any() else 1 << 62, 1, "fail"),
              (np.argmax(over) if over.any() else 1 << 62, 1, "ub")]
        first = min(ev)
        if first[0] < (1 << 62):
            _expand(out, t, int(first[0]))
            if first[2] == "q2":
                return "good", bytes(out)
            return first[2], b""
        if not eob:
            return "unknown", b""                            # whatever the bits after the last token decode to
        _expand(out, t, len(t))
        if final:
            return "good", bytes(out)
    return "ub", b""                                         # no final block and nothing behind the last one


# ---------------------------------------------------------------------------------------------------- helpers ----
def pad_to(cur_bits, target_bits, filler=(0x30, 0x90)):
    """Literals (fixed code: `filler[0]` is 8 bits, `filler[1]` is 9 bits) that take a fixed block from bit `cur_bits` to
    exactly `target_bits` (or the first reachable offset just after it)."""
    need = max(0, target_bits - cur_bits)
    while need % 8 and need < 9 * (need % 8):
        need += 1                                        # too close for an exact hit: the first offset after it
    nine = need % 8
    return bytes([filler[0]]) * ((need - 9 * nine) // 8) + bytes([filler[1]]) * nine


# -------------------------------------------------------------------------------------------------- catalogue ----
# Stream families shared by the emulator suite (small) and the GPU suite (large). Every case is a dict:
#   name, stream, cap, path ("walk": the warp-per-stream decoder and its rounds, "fx": one fixed block, "bsplit": many
#   blocks, long enough for the block-split path), want = (verdict, bytes) of the reference.
def filler(n_out, rng, start_pos=0, max_dist=32768, lit_share=0.5, alphabet=None):
    """Tokens that produce about n_out bytes: runs of literals and matches that reach back at most max_dist (and never
    before the output start: positions count from start_pos)."""
    k = max(1, n_out // 6)
    is_lit = rng.random(k) < lit_share
    ln = np.where(is_lit, 1, rng.integers(3, 40, k))
    ln[: max(0, 64 - start_pos)] = 1
    is_lit |= ln == 1
    pos = start_pos + np.concatenate([[0], np.cumsum(ln)[:-1]])
    alpha = np.arange(1, 256) if alphabet is None else np.asarray(alphabet)
    lit = alpha[rng.integers(0, len(alpha), k)]
    d = np.minimum(rng.integers(1, max_dist + 1, k), np.maximum(pos, 1))
    sym = np.where(is_lit, lit, 0)
    m = matches(np.where(is_lit, 3, ln), np.where(is_lit, 1, d))
    return Tokens(np.where(is_lit, sym, m.sym), np.where(is_lit, 0, m.lx), np.where(is_lit, -1, m.dsym),
                  np.where(is_lit, 0, m.dx))


def _case(name, blocks, path, cap=None, tail=b"", in_size=None):
    s = write(blocks, tail)
    data = s.data if in_size is None else s.data[:in_size]
    c = cap if cap is not None else max(s.max_out, len(data)) + 4096
    return dict(name=name, stream=s, data=data, cap=c, path=path, want=s.expect(c, len(data)))


def _q5_lit_lens(first_len):
    """symbol 0 first with `first_len` bits; 1-127 at 8, 128-285 at 9 bits: for first_len 10 it is the unique longest,
    so the reference (whose maximum then stays 9) cannot decode it; for 9 a later 9 raises the maximum to 9."""
    return [first_len] + [8] * 127 + [9] * 158


def fam_a(big, rng):
    out_n = 400_000 if big else 60_000
    no0 = np.arange(1, 256)
    cases = []
    body = filler(out_n, rng, alphabet=no0)
    k = int(len(body) * 0.8)
    used = cat(Tokens(*(getattr(body, f)[:k] for f in ("sym", "lx", "dsym", "dx"))), lits(b"\0"),
               Tokens(*(getattr(body, f)[k:] for f in ("sym", "lx", "dsym", "dx"))))
    dl = [5] * 30
    for fl, tok, nm in ((10, body, "A1 lit unique longest unused"), (10, used, "A2 lit unique longest used deep"),
                        (9, used, "A first length equals a later maximum")):
        cases.append(_case(nm, [dynamic(tok, final=True, lit_lens=_q5_lit_lens(fl), dist_lens=dl)], "walk"))
    # distance alphabet: symbol 0 (distance 1) first and uniquely longest
    dq = [6] + [5] * 29
    nod1 = filler(out_n, rng)
    nod1.dx[nod1.dsym == 0] = 0
    nod1.dsym[nod1.dsym == 0] = 1                      # distance 2 instead of 1
    cases.append(_case("A dist unique longest unused", [dynamic(nod1, final=True, dist_lens=dq)], "walk"))
    kd = int(len(nod1) * 0.8)
    withd1 = cat(Tokens(*(getattr(nod1, f)[:kd] for f in ("sym", "lx", "dsym", "dx"))), lits(b"x"), match(5, 1),
                 Tokens(*(getattr(nod1, f)[kd:] for f in ("sym", "lx", "dsym", "dx"))))
    cases.append(_case("A dist unique longest used deep", [dynamic(withd1, final=True, dist_lens=dq)], "walk"))
    # code-length alphabet: symbol 0 first and uniquely longest (5 bits; 1-15 at 4 bits)
    cl = [5] + [4] * 15 + [0, 0, 0]
    ll = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 6    # 286 symbols, no zero length: symbol 0 of the CL code unused
    tok = filler(out_n // 4, rng)
    p_full = [(x, 1) for x in ll + [5] * 30]
    cases.append(_case("A CL unique longest unused", [dynamic(tok, final=True, hlit=286, hdist=30, cl_lens=cl, plan=p_full)], "walk"))
    p_zero = [(x, 1) for x in ll[:-1] + [0] + [5] * 30]
    cases.append(_case("A CL unique longest used", [dynamic(tok, final=True, hlit=286, hdist=30, cl_lens=cl, plan=p_zero)], "walk"))
    return cases


def _perm_lengths(freqs, want_long):
    """Lengths of a complete <= 15-bit code whose LONGEST codes go to the symbols in want_long (in that order)."""
    ln = limited_lengths(freqs, 15)
    order = sorted((s for s in range(len(ln)) if ln[s]), key=lambda s: -ln[s])
    lens_sorted = [ln[s] for s in order]
    rest = [s for s in order if s not in want_long]
    out = [0] * len(ln)
    for s, x in zip(list(want_long) + rest, lens_sorted):
        out[s] = x
    return out


def fam_b(big, rng):
    out_n = 400_000 if big else 80_000
    f = np.ones(286, np.int64)
    f[:24] = 1 << np.arange(40, 16, -1)                   # steep frequencies: the code reaches 15 bits
    tok = filler(out_n, rng)
    ll = _perm_lengths(f, [284, 285, 257, 258])
    fd = 1 << np.arange(30, 0, -1).astype(np.int64)
    dl = _perm_lengths(fd, [29, 28])
    assert max(ll) == 15 and max(dl) == 15 and ll[284] == 15 and dl[29] == 15
    cases = [_case("B 15-bit codes on frequent length symbols", [dynamic(tok, final=True, lit_lens=ll, dist_lens=dl)], "walk")]
    # 48-bit symbols: 284+31 (258) at distance 29+8191 (32768), once the output is past 32 KiB
    pre = filler(40_000, rng, max_dist=300)
    n48 = 3000 if big else 600
    t48 = cat(*([match(258, 32768, lsym=284, lx=31)] * 4))
    t48 = Tokens(*(np.tile(getattr(t48, f), n48 // 4) for f in ("sym", "lx", "dsym", "dx")))
    mix = cat(pre, t48, lits(b"tail"), t48)
    cases.append(_case("B 48-bit symbol stretch", [dynamic(mix, final=True, lit_lens=ll, dist_lens=dl)], "walk"))
    return cases


def fam_c(big, rng):
    out_n = 300_000 if big else 60_000
    tok = filler(out_n, rng, alphabet=np.arange(0, 200))
    ll = [8] * 200 + [0] * 56 + [8] + [9] * 29     # Kraft < 1: literals 200-255 have no code
    cases = [_case("C incomplete, hole never hit", [dynamic(tok, final=True, lit_lens=ll)], "walk")]
    k = int(len(tok) * 0.85)
    holed = cat(Tokens(*(getattr(tok, f)[:k] for f in ("sym", "lx", "dsym", "dx"))), hole(), lits(b"after"))
    cases.append(_case("C incomplete, hole hit deep", [dynamic(holed, final=True, lit_lens=ll)], "walk"))
    lit_only = lits(rng.integers(0, 256, out_n // 4, dtype=np.uint8).tobytes())
    cases.append(_case("C HDIST=1 length 0, literals only", [dynamic(lit_only, final=True, dist_lens=[0], hdist=1)], "walk"))
    one = cat(lits(b"abcdefgh" * 8), matches(np.full(out_n // 40, 20), np.full(out_n // 40, 7)))
    cases.append(_case("C HDIST=6 one 1-bit code", [dynamic(one, final=True, dist_lens=[0, 0, 0, 0, 0, 1], hdist=6)], "walk"))
    cases.append(_case("C HDIST=2 one 1-bit code at 0", [dynamic(cat(lits(b"zz"), matches([10] * 50, [1] * 50)), final=True, dist_lens=[1, 0], hdist=2)], "walk"))
    cases.append(_case("C HDIST=1 1-bit code (Q3)", [dynamic(cat(lits(b"zz"), match(10, 1)), final=True, dist_lens=[1], hdist=1)], "walk"))
    return cases


def fam_d(big, rng):
    out_n = 300_000 if big else 60_000
    tok = filler(out_n, rng)
    ll = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8    # 286/287 carry lengths (the fixed code's)
    dl = [5] * 32
    cases = [_case("D 286/287 and 30/31 coded, unused", [dynamic(tok, final=True, lit_lens=ll, dist_lens=dl, hlit=288, hdist=32)], "walk")]
    k = int(len(tok) * 0.8)
    head = Tokens(*(getattr(tok, f)[:k] for f in ("sym", "lx", "dsym", "dx")))
    for nm, bad in (("D distance 30 used", raw(257, 0, 30, 0)), ("D distance 31 used", raw(280, 3, 31, 0)),
                    ("D litlen 286 used", raw(286, 0, 0)), ("D litlen 287 used", raw(287, 0, 3))):
        cases.append(_case(nm, [dynamic(cat(head, bad, lits(b"after")), final=True, lit_lens=ll, dist_lens=dl, hlit=288, hdist=32)], "walk"))
    fx_n = 200_000 if big else 90_000
    ftok = filler(fx_n, rng)
    kf = int(len(ftok) * 0.9)
    fhead = Tokens(*(getattr(ftok, f)[:kf] for f in ("sym", "lx", "dsym", "dx")))
    cases.append(_case("D fixed block, clean", [fixed(ftok, final=True)], "fx"))
    for nm, bad in (("D fixed distance 30", raw(258, 0, 30)), ("D fixed distance 31", raw(258, 0, 31)),
                    ("D fixed litlen 286", raw(286, 0, 0)), ("D fixed litlen 287", raw(287, 0, 3))):
        cases.append(_case(nm, [fixed(cat(fhead, bad, lits(b"after" * 50)), final=True)], "fx"))
    return cases


def fam_e(big, rng):
    tok = filler(30_000, rng)
    cases = []
    z = [(18, 138), (18, 120)]                    # 258 zero lengths (HLIT 257 + HDIST 1) from a 4-entry CL code
    pre = fixed(filler(5000, rng))
    cases.append(_case("E HCLEN 4, empty tables, Q2 ends it", [pre, dynamic(_tok([]), final=True, eob=False, hlit=257, hdist=1, hclen=4,
                                                                           cl_lens=[0] * 18 + [1], plan=z)], "walk"))
    cases.append(_case("E HCLEN 4, empty tables, symbol follows", [pre, dynamic(_tok([]), final=True, eob=False, hlit=257, hdist=1, hclen=4,
                                                                               cl_lens=[0] * 18 + [1], plan=z)], "walk", tail=b"\xff" * 4))
    cases.append(_case("E HCLEN 19", [dynamic(tok, final=True, hclen=19)], "walk"))
    lit_only = lits(rng.integers(0, 256, 20000, dtype=np.uint8).tobytes())
    cases.append(_case("E HLIT 257", [dynamic(lit_only, final=True, hlit=257, dist_lens=[0], hdist=1)], "walk"))
    cases.append(_case("E HLIT 288 HDIST 32", [dynamic(tok, final=True, hlit=288, hdist=32)], "walk"))
    # repeat codes across the boundary and past the end: 257 literal/EOB lengths of 9 (+ 256 at 9), 30 distances of 5
    ll = [9] * 257 + [0] * 29
    p = [(9, 1), (16, 6)] * 36 + [(9, 1), (16, 4)]        # 257 nines: 36*7 + 5
    assert plan_lengths(p, 257)[0] == [9] * 257
    lits_only = lits(rng.integers(0, 256, 10000, dtype=np.uint8).tobytes())
    p_cross = [(9, 1), (16, 6)] * 36 + [(9, 1), (16, 3), (16, 3)]   # the last 16 runs two lengths into the distance code
    cases.append(_case("E 16 across the litlen/dist boundary", [dynamic(lits_only, final=True, hlit=257, hdist=30, plan=p_cross + [(18, 28)])], "walk"))
    p_past = p + [(18, 40)]                                    # 18 writes past the end of HLIT + HDIST
    cases.append(_case("E 18 past the end", [dynamic(lits_only, final=True, hlit=257, hdist=30, plan=p_past)], "walk"))
    p_past16 = p + [(5, 1), (16, 6), (16, 6), (16, 6), (16, 6), (16, 6)]  # 1 + 30 > 30: the last 16 runs one past the end
    cases.append(_case("E 16 past the end", [dynamic(lits_only, final=True, hlit=257, hdist=30, plan=p_past16)], "walk"))
    cases.append(_case("E 16 first", [dynamic(lits_only, final=True, hlit=257, hdist=2, plan=[(16, 3)] + p)], "walk"))
    over = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
    over[5] = 7                                            # one code shorter: over-subscribed
    cases.append(_case("E over-subscribed litlen", [dynamic(lits_only, final=True, lit_lens=over, hlit=288)], "walk"))
    cases.append(_case("E over-subscribed distance", [dynamic(tok, final=True, dist_lens=[1, 1, 1] + [5] * 27)], "walk"))
    cases.append(_case("E over-subscribed CL code", [dynamic(tok, final=True, cl_lens=[2] * 19)], "walk"))
    return cases


def _tiny_blocks(n_out, rng, every):
    """Many small blocks: dynamic blocks of ~`every` output bytes with BTYPE-3 blocks, EOB-only dynamic and fixed
    blocks, LEN-0 stored blocks and stored payloads of 500-700 bytes (which straddle the 512-byte input halves)."""
    blocks, pos, k = [], 0, 0
    while pos < n_out:
        t = filler(every, rng, start_pos=pos)
        blocks.append(dynamic(t))
        pos += int(token_out_len(t).sum())
        r = k % 7
        if r == 1:
            blocks.append(btype3())
        elif r == 2:
            blocks.append(dynamic(_tok([]), lit_lens=[0] * 256 + [1]))
        elif r == 3:
            blocks.append(fixed(_tok([])))
        elif r == 4:
            blocks.append(stored(b""))
        elif r == 5 and k % 21 == 5:  # (a chunk with a stored block of > 256 bytes is decoded again, not expanded from tokens)
            d = rng.integers(0, 256, int(rng.integers(500, 700)), dtype=np.uint8).tobytes()
            blocks.append(stored(d))
            pos += len(d)
        k += 1
    blocks.append(dynamic(filler(every, rng, start_pos=pos), final=True))
    return blocks


def _out_len(blocks):
    return sum(int(token_out_len(b.tokens).sum()) if b.tokens is not None else len(b.data) if b.btype == 0 else 0
               for b in blocks)


def _odd_block(kind, pos, rng):
    """A dynamic block with an odd table (or an odd symbol) whose symbols are valid at output position `pos`."""
    if kind == "Q5 unused" or kind == "Q5 used":
        t = filler(3000, rng, start_pos=pos, alphabet=np.arange(1, 256))
        if kind == "Q5 used":
            t = cat(t, lits(b"\0"), filler(300, rng, start_pos=pos, alphabet=np.arange(1, 256)))
        return dynamic(t, lit_lens=_q5_lit_lens(10), dist_lens=[5] * 30)
    if kind == "hole":
        t = filler(3000, rng, start_pos=pos, alphabet=np.arange(0, 200))
        return dynamic(cat(t, hole()), lit_lens=[8] * 200 + [0] * 56 + [8] + [9] * 29)
    full = dict(lit_lens=fixed_litlen_lengths(), dist_lens=[5] * 32, hlit=288, hdist=32)
    if kind == "286/287 coded, unused":
        return dynamic(filler(3000, rng, start_pos=pos), **full)
    if kind == "distance 30":
        return dynamic(cat(filler(3000, rng, start_pos=pos), raw(257, 0, 30, 0)), **full)
    if kind == "litlen 286":
        return dynamic(cat(filler(3000, rng, start_pos=pos), raw(286, 0, 0)), **full)
    if kind == "over-subscribed litlen":
        over = fixed_litlen_lengths()
        over[5] = 7
        return dynamic(filler(3000, rng, start_pos=pos), lit_lens=over, dist_lens=[5] * 30, hlit=288)
    if kind == "Q3":
        return dynamic(cat(lits(b"zz"), match(10, 1)), dist_lens=[1], hdist=1)
    assert kind == "16 across the boundary"
    p_cross = [(9, 1), (16, 6)] * 36 + [(9, 1), (16, 3), (16, 3)]
    return dynamic(lits(rng.integers(0, 256, 2000, dtype=np.uint8).tobytes()), hlit=257, hdist=30, plan=p_cross + [(18, 28)])


ODD_KINDS = ("Q5 unused", "Q5 used", "hole", "286/287 coded, unused", "distance 30", "litlen 286", "over-subscribed litlen",
             "Q3", "16 across the boundary")


def fam_f(big, rng):
    n = 1_300_000 if big else 80_000
    blocks = _tiny_blocks(n, rng, 700 if big else 400)
    cases = [_case("F tiny blocks", blocks, "bsplit"),
             _case("F tiny blocks, data after the final block", blocks, "bsplit", tail=b"\x5a" * 300)]
    # the same stream with one odd block 60 % of the way in: a block-split chunk well after the first decodes through it
    # (the header search proposes only valid, complete tables, so the chunk that reaches it started before it)
    n_odd = 400_000 if big else 50_000
    base = _tiny_blocks(n_odd, rng, 700 if big else 400)
    at = int(len(base) * 0.6)
    for kind in ODD_KINDS:
        odd = _odd_block(kind, _out_len(base[:at]), rng)
        cases.append(_case("F odd block: " + kind, base[:at] + [odd] + base[at:], "bsplit"))
    return cases


def _trains(pos):
    """Run-length trains of period 1, 2 and 4 and lengths 47, 48 and 258, each starting at every output offset mod 16
    (the stream's output at `pos` when the tokens begin); a few distinct bytes before each train are its pattern."""
    parts = []
    for d in (1, 2, 4):
        for L in (47, 48, 258):
            for off in range(16):
                k = 4 + (off - pos - 4) % 16            # literals so that the match starts at an offset = off (mod 16)
                parts += [lits(bytes((7 * i + d + L) & 255 for i in range(k))), match(L, d)]
                pos += k + L
    return cat(*parts)


def fam_g(big, rng):
    cases = []
    n_lead = 24000 if big else 12000
    lead = fixed(lits(rng.integers(0, 256, n_lead, dtype=np.uint8).tobytes()))
    parts = []
    parts.append(cat(*[match(L, d) for d in [3] + list(range(5, 32)) for L in (3, 7, 31, 100, 258)]))
    parts.append(cat(*[match(L, 32) for L in range(33, 259)]))
    parts.append(cat(*[cat(match(L, L), match(L, L - 1)) for L in range(4, 259, 3)]))
    # dense short matches whose source ends -2..+2 bytes around the start of one of the preceding 32 tokens' outputs
    ln = rng.integers(3, 9, 4000)
    back = rng.integers(1, 32, 4000)
    dens = []
    for i in range(4000):
        j = max(0, i - back[i])
        span = int(ln[j:i].sum()) if i > j else 0
        dist = max(1, span + int(ln[i]) + int(rng.integers(-2, 3)))
        dens.append((int(ln[i]), dist))
    parts.append(matches([a for a, _ in dens], [b for _, b in dens]))
    rest = cat(*parts)

    def seq(pos, *pieces):
        """Tokens of `pieces` placed one after the other from output position pos ("T" = trains + the rest, an int =
        that much filler)."""
        out = []
        for p in pieces:
            t = cat(_trains(pos), rest) if p == "T" else filler(p, rng, start_pos=pos)
            out.append(t)
            pos += int(token_out_len(t).sum())
        return cat(*out), pos

    # the trains deep inside long blocks, so that lane-parallel rounds (10.5 KiB of compressed data each) expand them
    nf = 60_000 if big else 25_000
    deep1, pos = seq(n_lead, nf, "T", nf, "T")
    deep2, pos = seq(pos, nf, "T", nf, "T")
    last, _ = seq(pos, "T")
    blocks = [lead, dynamic(deep1), fixed(deep2), dynamic(last, final=True)]
    cases.append(_case("G expansion trains and overlaps", blocks, "walk"))
    one, _ = seq(64, "T", "T")
    cases.append(_case("G expansion trains, one fixed block", [fixed(cat(lits(b"q" * 64), one), final=True)], "fx"))
    # dist = pos (good) / pos + 1 (fails) past the first round: a literal-heavy prefix puts the compressed offset past
    # 10.5 KiB (the round length; fixed code: 8-9 bits per literal) while the output is still < 32 KiB
    n_pre = 16000 if big else 12000
    pre = lits(rng.integers(144, 256, n_pre, dtype=np.uint8).tobytes())   # 9-bit literals
    cases.append(_case("G dist = pos", [fixed(cat(pre, match(200, n_pre), lits(b"end" * 400)), final=True)], "fx"))
    cases.append(_case("G dist = pos + 1", [fixed(cat(pre, match(200, n_pre + 1), lits(b"end" * 400)), final=True)], "fx"))
    cases.append(_case("G dist = pos, dynamic", [dynamic(cat(pre, lits(b"x"), match(200, n_pre + 1), lits(b"end" * 400)), final=True)], "walk"))
    cases.append(_case("G dist = pos + 1, dynamic", [dynamic(cat(pre, match(200, n_pre + 1), lits(b"end" * 400)), final=True)], "walk"))
    return cases


def fam_h(big, rng):
    """Domain boundaries: long streams of far matches (up to 32768) and whole stretches copied from the previous 32 KiB,
    so that fixed-path groups, block-split chunks and pieces start inside matches and copy the previous domain's
    markers."""
    n = 1_200_000 if big else 160_000
    pre = filler(40_000, rng, max_dist=1000)
    far = matches(np.full(n // 258, 258), rng.choice([32768, 32767, 32000, 24577, 16385], n // 258))
    mixed = filler(n, rng, start_pos=40_000, max_dist=32768, lit_share=0.05)
    cases = [_case("H far copies, one fixed block", [fixed(cat(pre, far), final=True)], "fx"),
             _case("H far mixed, one fixed block", [fixed(cat(pre, mixed), final=True)], "fx")]
    blocks, pos = [dynamic(pre)], 40_000
    while pos < n:
        t = matches(np.full(200, 258), rng.choice([32768, 30000, 25000], 200)) if len(blocks) % 3 else filler(30_000, rng, start_pos=pos, lit_share=0.1)
        blocks.append(dynamic(t))
        pos += int(token_out_len(t).sum())
    blocks.append(dynamic(filler(3000, rng, start_pos=pos), final=True))
    cases.append(_case("H far copies, many blocks", blocks, "bsplit"))
    return cases


def fam_i(big, rng):
    cases = []
    base = filler(30_000 if big else 12_000, rng)
    for last_nm, last in (("literal", lits(b"A")), ("match", match(20, 300)), ("48-bit", match(258, 32768, lsym=284, lx=31))):
        pre = cat(lits(rng.integers(0, 256, 33000, dtype=np.uint8).tobytes()), base) if last_nm == "48-bit" else base
        s0 = write([fixed(pre, final=True, eob=False)])
        for delta in range(16):
            # the last symbol starts `delta` bits before the last whole byte's end ... past it (rule Q2 drops it when it
            # starts inside the last byte)
            target = (s0.end_bits // 8 + 12) * 8 + delta
            pad = pad_to(s0.end_bits, target)
            s = write([fixed(cat(pre, lits(pad), last), final=True, eob=False)])
            cut = len(s.data)
            t = int(s.offsets[-1][-1])
            if t % 8:   # cut the input inside the last symbol's first byte: rule Q2 drops it (nothing is read past the end)
                cut = (t + 7) // 8
            cases.append(dict(name="I Q2 %s +%d" % (last_nm, delta), stream=s, data=s.data[:cut], cap=cut + 300000, path="walk",
                              want=s.expect(cut + 300000, cut)))
    big_fixed = write([fixed(filler(150_000 if big else 60_000, rng), final=True)])
    n_out = len(big_fixed.output)
    for nm, cap in (("exact", n_out), ("exact-1", n_out - 1)):
        cases.append(dict(name="I capacity %s (fixed)" % nm, stream=big_fixed, data=big_fixed.data, cap=cap, path="fx",
                          want=big_fixed.expect(cap)))
    many = write(_tiny_blocks(1_100_000 if big else 100_000, rng, 600))
    m_out = len(many.output)
    for nm, cap in (("exact", m_out), ("exact-1", m_out - 1)):
        cases.append(dict(name="I capacity %s (blocks)" % nm, stream=many, data=many.data, cap=cap, path="bsplit",
                          want=many.expect(cap)))
    cases.append(dict(name="I cap < in_size", stream=big_fixed, data=big_fixed.data, cap=len(big_fixed.data) - 1, path="fx",
                      want=big_fixed.expect(len(big_fixed.data) - 1)))
    return cases


FAMILIES = dict(A=fam_a, B=fam_b, C=fam_c, D=fam_d, E=fam_e, F=fam_f, G=fam_g, H=fam_h, I=fam_i)


def catalogue(big, families="ABCDEFGHI", seed=1):
    out = []
    for f in families:
        out += FAMILIES[f](big, np.random.default_rng(seed + ord(f)))
    return out
