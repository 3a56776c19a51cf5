"""A coefficient-level progressive (SOF2) JPEG encoder for the tests (T.81 Annex G, the procedures of libjpeg's jcphuff.c).

``encode_progressive`` takes the same component list and quantised coefficients as ``jpeg_synth.encode_from_coefs``
(whose output is then the file's *baseline twin*: same frame, same coefficients), any scan script, any sampling the
library accepts (h1v2 included) and any restart interval.  Every scan gets its own Huffman tables, defined in front of it
(fixed-length codes over the symbols the scan uses), as progressive encoders redefine them between scans.
"""
import numpy as np

import jpeg_synth as js

# libjpeg's jpeg_simple_progression for three components / for one (component, Ss, Se, Ah, Al)
SCRIPT_YCC = [((0, 1, 2), 0, 0, 0, 1), ((0,), 1, 5, 0, 2), ((2,), 1, 63, 0, 1), ((1,), 1, 63, 0, 1), ((0,), 6, 63, 0, 2),
              ((0,), 1, 63, 2, 1), ((0, 1, 2), 0, 0, 1, 0), ((2,), 1, 63, 1, 0), ((1,), 1, 63, 1, 0), ((0,), 1, 63, 1, 0)]
SCRIPT_GRAY = [((0,), 0, 0, 0, 1), ((0,), 1, 5, 0, 2), ((0,), 6, 63, 0, 2), ((0,), 1, 63, 2, 1), ((0,), 0, 0, 1, 0),
               ((0,), 1, 63, 1, 0)]


class _Writer:
    """Scan tokens first (symbols are only coded once the scan's tables are known), bytes at the end."""

    def __init__(self):
        self.tok = []            # ("s", table_key, symbol) | ("b", value, nbits) | ("rst", n)

    def sym(self, key, s):
        self.tok.append(("s", key, s))

    def bits(self, v, n):
        if n:
            self.tok.append(("b", v & ((1 << n) - 1), n))


def _fixed_table(symbols):
    """counts / symbols of a fixed-length code over `symbols` (the all-ones code stays unused)."""
    syms = sorted(set(symbols))
    ln = 1
    while (1 << ln) - 1 < len(syms):
        ln += 1
    counts = [0] * 16
    counts[ln - 1] = len(syms)
    return counts, syms


def encode_progressive(width, height, comps, coefs, script, restart_interval=0, qts=None):
    """comps: [(h, v, qt_id, dc_id, ac_id)]; coefs: as for jpeg_synth.encode_from_coefs (MCU-padded grids, zig-zag,
    DC absolute); script: [(component indices, Ss, Se, Ah, Al)].  Returns the JPEG bytes."""
    dqt = js.std_tables()[1]
    qts = qts if qts is not None else dqt
    hs, vs = comps[0][0], comps[0][1]
    mw, mh = (width + 7) // 8, (height + 7) // 8
    nmx, nmy = (mw + hs - 1) // hs, (mh + vs - 1) // vs
    out = bytearray(b"\xFF\xD8")
    for tid in sorted(set(c[2] for c in comps)):
        out += b"\xFF\xDB" + (2 + 65).to_bytes(2, "big") + bytes([tid]) + bytes(int(q) for q in qts[tid])
    out += b"\xFF\xC2" + (8 + 3 * len(comps)).to_bytes(2, "big") + b"\x08" + height.to_bytes(2, "big") + width.to_bytes(2, "big")
    out += bytes([len(comps)])
    for i, c in enumerate(comps):
        out += bytes([i + 1, (c[0] << 4) | c[1], c[2]])
    if restart_interval:
        out += b"\xFF\xDD\x00\x04" + restart_interval.to_bytes(2, "big")
    for cids, ss, se, ah, al in script:
        w = _Writer()
        if len(cids) > 1:                               # interleaved (DC only): MCU order over the padded grid
            blocks = []
            for my in range(nmy):
                for mx in range(nmx):
                    mcu = []
                    for j in cids:
                        h, v = comps[j][0], comps[j][1]
                        for y in range(v):
                            for x in range(h):
                                mcu.append((j, my * v + y, mx * h + x))
                    blocks.append(mcu)
        else:
            j = cids[0]
            h, v = comps[j][0], comps[j][1]
            bw = ((width * h + hs - 1) // hs + 7) // 8
            bh = ((height * v + vs - 1) // vs + 7) // 8
            blocks = [[(j, by, bx)] for by in range(bh) for bx in range(bw)]
        _encode_scan(w, comps, coefs, cids, blocks, ss, se, ah, al, restart_interval)
        # tables of this scan
        used = {}
        for t in w.tok:
            if t[0] == "s":
                used.setdefault(t[1], []).append(t[2])
        maps = {}
        for (cls, tid), syms in sorted(used.items()):
            counts, sy = _fixed_table(syms)
            out += b"\xFF\xC4" + (2 + 17 + len(sy)).to_bytes(2, "big") + bytes([(cls << 4) | tid]) + bytes(counts) + bytes(sy)
            maps[(cls, tid)] = js._code_map(counts, sy)
        out += b"\xFF\xDA" + (6 + 2 * len(cids)).to_bytes(2, "big") + bytes([len(cids)])
        for j in cids:
            out += bytes([j + 1, (comps[j][3] << 4) | comps[j][4]])
        out += bytes([ss, se, (ah << 4) | al])
        bits = js._Bits()
        for t in w.tok:
            if t[0] == "s":
                bits.put(*maps[t[1]][t[2]])
            elif t[0] == "b":
                bits.put(t[1], t[2])
            else:
                bits.flush()
                bits.out += bytes([0xFF, 0xD0 + (t[1] & 7)])
        bits.flush()
        out += bits.out
    out += b"\xFF\xD9"
    return bytes(out)


def _encode_scan(w, comps, coefs, cids, blocks, ss, se, ah, al, ri):
    pred = {j: 0 for j in cids}
    state = {"eobrun": 0, "be": []}
    ackey = (1, comps[cids[0]][4])

    def emit_eobrun():
        n = state["eobrun"]
        if n:
            nb = n.bit_length() - 1
            w.sym(ackey, nb << 4)
            w.bits(n, nb)
            state["eobrun"] = 0
            for b in state["be"]:
                w.bits(b, 1)
            state["be"] = []

    nrst = 0
    for bi, mcu in enumerate(blocks):
        if ri and bi and bi % ri == 0:
            emit_eobrun()
            w.tok.append(("rst", nrst))
            nrst += 1
            pred = {j: 0 for j in cids}
        for j, by, bx in mcu:
            zz = [int(x) for x in coefs[j][by][bx]]
            if ss == 0:
                if ah == 0:
                    v = zz[0] >> al
                    s, b = js._mag(v - pred[j])
                    pred[j] = v
                    w.sym((0, comps[j][3]), s)
                    w.bits(b, s)
                else:
                    w.bits((zz[0] >> al) & 1, 1)
                continue
            if ah == 0:
                r = 0
                for k in range(ss, se + 1):
                    x = zz[k]
                    t = abs(x) >> al
                    if t == 0:
                        r += 1
                        continue
                    emit_eobrun()
                    while r > 15:
                        w.sym(ackey, 0xF0)
                        r -= 16
                    v = t if x > 0 else -t
                    s, b = js._mag(v)
                    w.sym(ackey, (r << 4) | s)
                    w.bits(b, s)
                    r = 0
                if r:
                    state["eobrun"] += 1
                    if state["eobrun"] == 0x7FFF:
                        emit_eobrun()
                continue
            absv = [abs(zz[k]) >> al for k in range(64)]
            eob = max([k for k in range(ss, se + 1) if absv[k] == 1], default=-1)
            r, br = 0, []
            for k in range(ss, se + 1):
                t = absv[k]
                if t == 0:
                    r += 1
                    continue
                while r > 15 and k <= eob:
                    emit_eobrun()
                    w.sym(ackey, 0xF0)
                    r -= 16
                    for b in br:
                        w.bits(b, 1)
                    br = []
                if t > 1:
                    br.append(t & 1)
                    continue
                emit_eobrun()
                w.sym(ackey, (r << 4) | 1)
                w.bits(1 if zz[k] > 0 else 0, 1)
                for b in br:
                    w.bits(b, 1)
                br = []
                r = 0
            if r > 0 or br:
                state["eobrun"] += 1
                state["be"] += br
                if state["eobrun"] == 0x7FFF or len(state["be"]) > 937:
                    emit_eobrun()
    emit_eobrun()


def pil_twins(arr, quality=90, subsampling=2, restart_blocks=0, gray=False):
    """Pillow's progressive file and its baseline twin (libjpeg quantises both the same way)."""
    import io
    from PIL import Image
    im = Image.fromarray(arr)
    if gray:
        im = im.convert("L")
    outs = []
    for prog in (True, False):
        kw = dict(quality=quality, progressive=prog)
        if not gray:
            kw["subsampling"] = subsampling
        if restart_blocks:
            kw["restart_marker_blocks"] = restart_blocks
        buf = io.BytesIO()
        im.save(buf, "JPEG", **kw)
        outs.append(buf.getvalue())
    return outs[0], outs[1]


def prog_twins(width, height, comps, coefs, script, restart_interval=0):
    """(progressive file, baseline twin without restart markers) of the test encoder."""
    return (encode_progressive(width, height, comps, coefs, script, restart_interval),
            js.encode_from_coefs(width, height, comps, coefs))


def within_grids(width, height, comps):
    """Per unit of the MCU-interleaved order: True if the unit lies inside its component's block grid (the units a
    non-interleaved scan codes; the others are MCU padding, which no output pixel depends on)."""
    hs, vs = comps[0][0], comps[0][1]
    mw, mh = (width + 7) // 8, (height + 7) // 8
    nmx, nmy = (mw + hs - 1) // hs, (mh + vs - 1) // vs
    m = []
    for my in range(nmy):
        for mx in range(nmx):
            for j, c in enumerate(comps):
                h, v = c[0], c[1]
                bw = ((width * h + hs - 1) // hs + 7) // 8
                bh = ((height * v + vs - 1) // vs + 7) // 8
                for y in range(v):
                    for x in range(h):
                        m.append(mx * h + x < bw and my * v + y < bh)
    return np.array(m, dtype=bool)
