"""The device PCD ingest -- LZF streams, ASCII record tiles and the record gather (csrc/pcd_ingest.cuh, host side
pcd_decode_files / pointcloud2_clouds in hafgpu.cu) -- at every shape and malformed input its kernels branch on.

References: LZF streams are written as explicit tokens (``lit``, ``ref``, ``raw`` bytes for malformed tails) and decoded by
``lzf_reference``, a plain decoder of the token grammar; it is pinned against the C++ reader (csrc/host/pcd_io.hpp through
``haf_cli --dump-pcd``) and against haf_grasping_b200/pcd.py on valid and corrupt streams.  ASCII and binary clouds come
from pcd.py, which the C++ reader must match on every catalogue file.

The kernels' control flow is restated in ``lzf_walk`` (input ring refills, ring slots, lane rounds, the rejection checks),
``ascii_walk`` (thread chunks, tiles, the tile -> file map, scan rounds), ``gather_walk_pcd`` and ``pc2_walk`` (load
alignments, segments, the grid-stride loop), so that the CPU test ``test_cases_cover_every_branch`` can show that the
catalogues reach every listed branch and that each catalogue entry reaches one no other entry does.  The GPU cases compare
every cloud byte for byte, single and batched, and the launches of each call with the kinds it holds.
"""
import struct
import subprocess

import numpy as np
import pytest

from conftest import FEATURES, RANGE

IN_RING, OUT_RING, REFILL, LOOKAHEAD = 8192, 16384, 4096, 512     # lzf_decompress_kernel
CHUNK, TILE, SCAN_ROUND = 16, 256 * 16, 1024                     # ASCII: bytes per thread, bytes per tile, tiles per scan round
GATHER_GRID_MAX = 148 * 16                                       # launch_gather: CTAs of 256 threads at most
BLANKS = b" \t\r"                                                # is_blank


# ---- LZF: tokens, assembler, reference decoder --------------------------------------------------------------------------
def lit(data):
    return ("lit", bytes(data))


def ref(length, dist):
    return ("ref", length, dist)


def raw(data):
    return ("raw", bytes(data))


def encode(tok):
    """the bytes of one token (liblzf: ctrl < 32 literal run of ctrl + 1 bytes; else length (ctrl >> 5, 7: + next byte) + 2,
    distance ((ctrl & 31) << 8 | next byte) + 1)"""
    if tok[0] == "raw":
        return tok[1]
    if tok[0] == "lit":
        assert 1 <= len(tok[1]) <= 32
        return bytes([len(tok[1]) - 1]) + tok[1]
    _, length, dist = tok
    assert 3 <= length <= 264 and 1 <= dist <= 8192
    d, l2 = dist - 1, length - 2
    if l2 < 7:
        return bytes([(l2 << 5) | (d >> 8), d & 0xFF])
    return bytes([0xE0 | (d >> 8), l2 - 7, d & 0xFF])


def assemble(tokens):
    return b"".join(encode(t) for t in tokens)


def lzf_reference(stream, out_len):
    """(decoded bytes or None, verdict): a plain decoder of the token grammar, one check per way a stream can be wrong"""
    out = bytearray()
    ip, n = 0, len(stream)
    while ip < n:
        ctrl = stream[ip]
        ip += 1
        if ctrl < 32:
            run = stream[ip:ip + ctrl + 1]
            if len(out) + ctrl + 1 > out_len:
                return None, "literal past out_len"
            if len(run) < ctrl + 1:
                return None, "literal past the input"
            out += run
            ip += ctrl + 1
            continue
        length = ctrl >> 5
        if length == 7:
            if ip >= n:
                return None, "no length byte"
            length += stream[ip]
            ip += 1
        if ip >= n:
            return None, "no distance byte"
        dist = ((ctrl & 31) << 8 | stream[ip]) + 1
        ip += 1
        length += 2
        if dist > len(out):
            return None, "distance before the output"
        if len(out) + length > out_len:
            return None, "reference past out_len"
        for _ in range(length):
            out.append(out[-dist])
    if len(out) != out_len:
        return None, "short output"
    return bytes(out), "ok"


class LzfBuilder:
    """a stream token by token, with ip / op tracked so tokens can be put at chosen input positions"""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.tokens = []
        self.ip = self.op = 0

    def add(self, tok):
        if tok[0] == "ref" and callable(tok[2]):
            tok = ref(tok[1], tok[2](self.op))
        self.tokens.append(tok)
        self.ip += len(encode(tok))
        self.op += 0 if tok[0] == "raw" else len(tok[1]) if tok[0] == "lit" else tok[1]
        return self

    def lit(self, n):
        return self.add(lit(self.rng.integers(0, 256, n, dtype=np.uint8).tobytes()))

    def ref(self, length, dist):
        return self.add(ref(length, dist))

    @staticmethod
    def _fill_steps(gap):
        """literal tokens (input bytes each) that fill exactly `gap` input bytes"""
        assert gap == 0 or gap >= 2, gap
        steps = []
        while gap:
            step = 33 if gap >= 35 or gap == 33 else 17 if gap == 34 else gap
            steps.append(step)
            gap -= step
        return steps

    def fill_to(self, ip):
        for step in self._fill_steps(ip - self.ip):
            self.lit(step - 1)
        return self

    def end_at(self, in_len):
        """literals, then one last token, so that the stream is in_len bytes and its output a multiple of 12 bytes"""
        for kind, size, ib in [("lit", m, m + 1) for m in range(1, 33)] + [("ref", m, 2 if m <= 8 else 3) for m in range(3, 265)]:
            gap = in_len - ib - self.ip
            if gap < 0 or gap == 1:
                continue
            steps = self._fill_steps(gap)
            if (self.op + sum(s - 1 for s in steps) + size) % 12 == 0:
                self.fill_to(in_len - ib)
                return self.lit(size) if kind == "lit" else self.ref(size, 1)
        raise AssertionError(in_len)

    def pad12(self):
        return self.lit(-self.op % 12) if self.op % 12 else self

    def stream(self):
        return assemble(self.tokens)


# ---- the kernel's control flow, restated (lzf_decompress_kernel) --------------------------------------------------------
def _edge(pos):
    """'before_refill' / 'after_wrap' ...: where an input byte sits against the 4 KB refills and the 8 KB input ring"""
    if pos % REFILL == REFILL - 1:
        return "before_" + ("wrap" if (pos + 1) % IN_RING == 0 else "refill")
    if pos and pos % REFILL == 0:
        return "after_" + ("wrap" if pos % IN_RING == 0 else "refill")
    return None


def lzf_walk(stream, out_len):
    """(branch items reached, verdict) of one stream"""
    hits = {"in_len_%d" % len(stream)} | ({"in_len_over_64k"} if len(stream) > 65536 else set())
    n = len(stream)
    ip = op = loaded = 0

    def at(pos, role):
        e = _edge(pos)
        if e:
            hits.add("%s_%s" % (role, e))

    while ip < n:
        while loaded < n and loaded < ip + LOOKAHEAD:
            loaded += min(REFILL, n - loaded)
        # every byte a token may read is in the ring and not yet overwritten by a later refill
        assert loaded - IN_RING <= ip and min(n, ip + 35) <= loaded
        ctrl = stream[ip]
        at(ip, "ctrl")
        if ctrl < 32:
            m = ctrl + 1
            if op + m > out_len:
                hits.add("reject_token_after_complete_output" if op == out_len else "reject_literal_past_out_len")
                return hits, "literal past out_len"
            if ip + 1 + m > n:
                hits.add("reject_literal_past_input")
                if ip + 1 < n:
                    hits.add("reject_literal_run_cut_short")
                return hits, "literal past the input"
            hits.add("literal_%d" % m)
            if (ip + 1) // IN_RING != (ip + m) // IN_RING:
                hits.add("literal_bytes_wrap_input_ring")
            if m == 32 and ip + 1 + m == n:
                hits.add("literal_32_ends_at_in_len")
            ip += 1 + m
            op += m
            continue
        length, q = ctrl >> 5, ip + 1
        if length == 7:
            if q >= n:
                hits.add("reject_no_length_byte")
                return hits, "no length byte"
            at(q, "len")
            length += stream[q]
            q += 1
        if q >= n:
            hits.add("reject_no_distance_byte")
            return hits, "no distance byte"
        at(q, "dist")
        dist = ((ctrl & 31) << 8 | stream[q]) + 1
        q += 1
        length += 2
        if dist > op:
            hits.add("reject_distance_op_plus_1" if dist == op + 1 else "reject_distance_before_output")
            return hits, "distance before the output"
        if op + length > out_len:
            hits.add("reject_token_after_complete_output" if op == out_len else
                     "reject_reference_overruns_by_1" if op + length == out_len + 1 else "reject_reference_past_out_len")
            return hits, "reference past out_len"
        hits.add("reference_%d" % length if length <= 9 or length == 264 else "reference_long")
        hits.add("lane_rounds_%d" % -(-length // 32))
        if dist in (1, 31, 32, 33):
            hits.add("distance_%d" % dist)
        if dist < length and length % dist:
            hits.add("distance_below_length_not_dividing")
        if dist == op:
            hits.add("distance_equals_op")
        if dist == 8192 and op > 2 * OUT_RING:
            hits.add("distance_8192_op_over_32768")
        elif dist == 8192 and op > OUT_RING:
            hits.add("distance_8192_op_over_16384")
        if (op - dist) % OUT_RING + min(length, dist) > OUT_RING:
            hits.add("reference_source_wraps_output_ring")
        ip = q
        op += length
    if op != out_len:
        hits.add("reject_stream_ends_at_out_len_minus_1" if op == out_len - 1 else "reject_short_output")
        return hits, "short output"
    return hits, "ok"


LZF_ITEMS = (["literal_1", "literal_31", "literal_32"] + ["reference_%d" % k for k in range(3, 10)] + ["reference_264", "lane_rounds_9"]
             + ["distance_1", "distance_31", "distance_32", "distance_33", "distance_below_length_not_dividing",
                "distance_8192_op_over_16384", "distance_8192_op_over_32768", "distance_equals_op", "reference_source_wraps_output_ring",
                "literal_bytes_wrap_input_ring", "literal_32_ends_at_in_len", "in_len_over_64k"]
             + ["%s_%s_%s" % (r, s, k) for r in ("ctrl", "len", "dist") for s in ("before", "after") for k in ("refill", "wrap")]
             + ["in_len_%d" % n for n in (0, 1, 511, 512, 513, 4095, 4096, 4097, 8191, 8192, 8193)])
LZF_REJECTS = ["reject_literal_past_input", "reject_literal_run_cut_short", "reject_literal_past_out_len", "reject_no_length_byte", "reject_no_distance_byte",
               "reject_distance_op_plus_1", "reject_reference_overruns_by_1", "reject_stream_ends_at_out_len_minus_1",
               "reject_token_after_complete_output"]


# ---- LZF catalogue ----------------------------------------------------------------------------------------------------
def _tokens_case():
    """every token shape: literal runs of 1, 31, 32; references of 3 .. 9 and 264 bytes (9 lane rounds); distances 1, 31,
    32, 33, equal to op, below the length and not dividing it"""
    B = LzfBuilder(1)
    B.lit(1).ref(3, 1).lit(31).ref(4, 31).lit(32).ref(5, 32).ref(6, 33).ref(7, lambda op: op).ref(8, 2).ref(9, 5)
    B.ref(264, 7).ref(264, 1).ref(100, 3).ref(40, lambda op: op).lit(2)
    return B.pad12()


def _ring_edges_case():
    """control, length and distance bytes at the last byte before and the first byte after 4 KB refills and 8 KB ring wraps;
    references at distance 8192 once the 16 KB output ring has wrapped (op > 16384, > 32768); a literal run across a ring wrap;
    more than 64 KB of input"""
    B = LzfBuilder(2)
    B.lit(32)
    plan = [(1, "ctrl", -1), (2, "ctrl", -1), (3, "ctrl", 0), (4, "ctrl", 0), (5, "len", -1), (6, "len", -1), (7, "len", 0),
            (8, "len", 0), (9, "dist", -1), (10, "dist", -1), (11, "dist", 0), (12, "dist", 0)]
    for k, role, side in plan:
        pos = REFILL * k + side
        long_ref = role == "len" or (role == "dist" and k % 2 == 0) or (role == "ctrl" and k in (2, 3))
        ctrl_at = pos - {"ctrl": 0, "len": 1, "dist": 2 if long_ref else 1}[role]
        B.fill_to(ctrl_at - 40)
        B.ref(200, 8192 if B.op >= 8192 else B.op).ref(6, 4000 if B.op >= 4000 else 1)     # output ring traffic between the edges
        B.fill_to(ctrl_at)
        if role == "ctrl" and k in (1, 4):
            B.lit(32 if k == 1 else 7)
        else:
            length = 9 + 19 * k if long_ref else 3 + k % 6
            B.ref(length, 8192 if B.op > 8192 else max(1, B.op - k))
    B.ref(100, lambda op: op % OUT_RING + 10)                            # source bytes 16374 .. 16383, then 0 .. of the output ring
    B.fill_to(7 * IN_RING - 6).lit(32)                                   # literal bytes across the ring wrap at 57344
    B.ref(264, 8192)
    return B.end_at(70001)


def _length_case(in_len):
    B = LzfBuilder(in_len)
    B.lit(20).ref(30, 20)
    if in_len > 600:
        B.fill_to(in_len // 2).ref(50, 17)
    return B.end_at(in_len)


def _literal_at_end_case():
    B = LzfBuilder(9)
    B.lit(24).ref(70, 24).lit(5)
    B.lit(-(B.op + 32) % 12 or 12)
    return B.lit(32)


def lzf_valid_cases():
    """name -> (stream, out_len); every output is a whole number of 12-byte points, so the cloud covers every decoded byte"""
    cases = {"tokens": _tokens_case(), "ring_edges": _ring_edges_case(), "literal_32_at_end": _literal_at_end_case()}
    for n in (511, 512, 513, 4095, 4096, 4097, 8191, 8192, 8193):
        cases["in_len_%d" % n] = _length_case(n)
    out = {}
    for name, B in cases.items():
        assert B.op % 12 == 0, name
        out[name] = (B.stream(), B.op)
    return out


def lzf_bad_cases():
    """name -> (stream, out_len): one case per rejection lzf_decompress_kernel checks"""
    def prefix(seed=3, op=60):
        return LzfBuilder(seed).lit(20).ref(op - 20, 20)
    cases = {}
    cases["empty_stream"] = ([], 12)                                                      # in_len 0
    cases["lone_literal_control"] = ([raw([0])], 12)                                      # in_len 1: a literal past the end of the input
    B = prefix()
    cases["literal_past_input"] = (B.tokens + [raw([5, 1, 2])], 72)
    cases["literal_past_out_len"] = (prefix().lit(4).tokens, 63)
    cases["long_reference_without_length_byte"] = (prefix().tokens + [raw([0xE0])], 120)
    cases["reference_without_distance_byte"] = (prefix().tokens + [raw([0x40])], 120)
    cases["distance_op_plus_1"] = (prefix().ref(3, lambda op: op + 1).tokens, 72)
    cases["reference_overruns_by_1"] = (prefix().ref(13, 7).tokens, 72)
    cases["stream_ends_at_out_len_minus_1"] = (prefix().ref(11, 7).tokens, 72)
    cases["literal_after_complete_output"] = (prefix().lit(12).lit(1).tokens, 72)
    return {k: (assemble(t), n) for k, (t, n) in cases.items()}


def lzf_pcd(stream, out_len):
    """a binary_compressed PCD file around one stream: x / y / z float32, out_len // 12 points"""
    n = out_len // 12
    return pcd_header("binary_compressed", n) + struct.pack("<II", len(stream), out_len) + stream


def blob_xyz(blob):
    n = len(blob) // 12
    return np.ascontiguousarray(np.frombuffer(blob, np.float32, count=3 * n).reshape(3, n).T)


# ---- PCD files --------------------------------------------------------------------------------------------------------
XYZ = (("x", "F", 4, 1), ("y", "F", 4, 1), ("z", "F", 4, 1))


def pcd_header(kind, n, fields=XYZ, comment=""):
    return ("# .PCD v0.7%s\nVERSION 0.7\nFIELDS %s\nSIZE %s\nTYPE %s\nCOUNT %s\nWIDTH %d\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS %d\nDATA %s\n"
            % (comment, " ".join(f[0] for f in fields), " ".join(str(f[2]) for f in fields), " ".join(f[1] for f in fields),
               " ".join(str(f[3]) for f in fields), n, n, kind)).encode()


def data_section(f):
    return f[f.index(b"\n", f.index(b"\nDATA ") + 1) + 1:]


def header_points(f):
    return int(f.split(b"\nPOINTS ")[1].split(b"\n")[0])


class AsciiBody:
    """the DATA section of an ASCII file, with records placed at chosen byte offsets (gaps are lines of blanks)"""

    def __init__(self, seed, ntok=3):
        self.rng = np.random.default_rng(seed)
        self.b = bytearray()
        self.ntok = ntok
        self.records = 0

    def text(self, sep=b" "):
        return sep.join(b"%.9g" % v for v in self.rng.normal(size=self.ntok).astype(np.float32))

    def rec(self, text=None, eol=b"\n"):
        self.b += (self.text() if text is None else text) + eol
        self.records += 1
        return self

    def pad_to(self, pos):
        gap = pos - len(self.b)
        assert gap >= 0 and (not self.b or self.b[-1:] == b"\n"), gap
        if gap:
            self.b += b" " * (gap - 1) + b"\n"
        return self

    def records_to(self, pos):
        """records up to 40 bytes before pos, then blanks up to pos"""
        while len(self.b) + 40 < pos:
            self.rec()
        return self.pad_to(pos)

    def rec_at(self, pos, text=None, eol=b"\n"):
        return self.records_to(pos).rec(text, eol)


def ascii_file(body, points=None, fields=XYZ):
    return pcd_header("ascii", body.records if points is None else points, fields) + bytes(body.b)


def _chunk_positions():
    """leading blank lines, then a record start at each of the 16 bytes of a thread's chunk, tab-separated records"""
    A = AsciiBody(20)
    A.b += b"\n \t\r\n\n"
    for k in range(CHUNK):
        A.pad_to(-(-len(A.b) // CHUNK) * CHUNK + k).rec(A.text(b"\t" if k % 2 else b" "))
    return ascii_file(A)


def _tile_edges():
    """record starts at tile bytes 4095, 4096 and 4097; a record and a line of blanks across tile boundaries; CR LF with the
    CR as a tile's last byte; a data section of exactly 7 tiles"""
    A = AsciiBody(21)
    A.rec_at(TILE - 1)
    A.rec_at(2 * TILE)
    A.rec_at(3 * TILE + 1)
    A.rec_at(4 * TILE - 10)                          # ~30 bytes: across the boundary
    A.records_to(5 * TILE - 20).pad_to(5 * TILE + 20)   # blanks across the boundary
    t = A.text()
    A.rec_at(6 * TILE - 1 - len(t), t, b"\r\n")
    A.records_to(7 * TILE)
    return ascii_file(A)


def _length_plus_1_no_newline():
    A = AsciiBody(22)
    t = A.text()
    A.records_to(2 * TILE + 1 - len(t)).rec(t, b"")
    return ascii_file(A)


def _length_minus_1():
    A = AsciiBody(23)
    return ascii_file(A.records_to(3 * TILE - 1))


def _surplus_inside_tile():
    """POINTS ends inside a tile, CR LF lines, 9 surplus records after it in the same tile"""
    A = AsciiBody(24)
    for _ in range(250):
        A.rec(eol=b"\r\n")
    return ascii_file(A, points=A.records - 9)


def _vt_ff():
    """vertical tab and form feed are token characters: they neither split fields nor make a line blank"""
    A = AsciiBody(25)
    A.rec().rec(b"1.5\x0b 2 3").rec(b"1\x0b2 3 4").rec(b"\x0c1 2 3").rec(b"4 5 6\x0c").rec(b"  \x0b7 8 9").rec(b"7\x0c8 9 10 11")
    return ascii_file(A)


COUNTED = (("normal", "F", 4, 3), ("z", "F", 4, 1), ("rgb", "U", 4, 2), ("y", "F", 4, 1), ("x", "F", 4, 1))


def _count_permuted():
    """a COUNT 3 and a COUNT 2 field ahead of z, y, x: x / y / z are tokens 7, 6, 3"""
    A = AsciiBody(26, ntok=8)
    for i in range(300):
        toks = A.text().split(b" ")
        toks[4] = b"%d" % (i * 7919)
        toks[5] = b"%d" % (4294967295 - i)
        A.rec(b" ".join(toks))
    return ascii_file(A, fields=COUNTED)


def _short_record_last_tile():
    A = AsciiBody(27)
    A.records_to(2 * TILE + 100).rec(b"0.5 0.25").records_to(2 * TILE + 300)
    return ascii_file(A)


def _ff_only_line():
    A = AsciiBody(28)
    return ascii_file(A.records_to(500).rec(b"\x0c").records_to(900), points=A.records - 1)


def ascii_valid_cases():
    return {"chunk_positions": _chunk_positions(), "tile_edges": _tile_edges(), "len_plus_1_no_newline": _length_plus_1_no_newline(),
            "len_minus_1": _length_minus_1(), "surplus_inside_tile": _surplus_inside_tile(), "vt_ff": _vt_ff(),
            "count_permuted": _count_permuted()}


def ascii_bad_cases():
    return {"short_record_last_tile": _short_record_last_tile(), "ff_only_line": _ff_only_line()}


def scan_round_batch():
    """many small ASCII files whose first tiles land at 1023, 1024 and 2048, files across the scan rounds' edges, a POINTS 0
    ASCII file and binary / binary_compressed files in between"""
    files, tile = [], 0
    k = 0
    while tile < 2050:
        ntiles = 2 if tile in (600, 1500) else 1030 if tile == 2049 else 1     # the last file runs across tile 3072
        A = AsciiBody(1000 + k)
        if ntiles > 1:
            A.records_to((ntiles - 1) * TILE + 50)
        else:
            for _ in range(1 + k % 4):
                A.rec()
        files.append(ascii_file(A))
        tile += ntiles
        k += 1
        if k == 700:
            files.append(ascii_file(AsciiBody(0), points=0))
        if k % 500 == 0:
            xyz = np.random.default_rng(k).normal(size=(5, 3)).astype(np.float32)
            files.append(pcd_header("binary", 5) + xyz.tobytes())
            files.append(lzf_pcd(*_literal_stream(np.ascontiguousarray(xyz.T).tobytes())))
    return files


def _literal_stream(blob):
    return assemble([lit(blob[i:i + 32]) for i in range(0, len(blob), 32)]), len(blob)


# ---- the ASCII passes, restated (ascii_count / scan / parse kernels, pcd_decode_files) ----------------------------------
def lines_of(data):
    """(begin, end, is_record) of every line; a record is a line holding a byte other than blank, tab and CR"""
    out, s = [], 0
    while s < len(data):
        e = data.find(b"\n", s)
        e = len(data) if e < 0 else e
        out.append((s, e, any(c not in BLANKS for c in data[s:e])))
        s = e + 1
    return out


def ascii_tok(f):
    """token numbers of x, y, z (COUNT-aware), as the host sends them in AsciiFile.tok"""
    hdr = f[:f.index(b"\nDATA ")].decode().split("\n")
    h = {ln.split()[0]: ln.split()[1:] for ln in hdr if ln and not ln.startswith("#")}
    counts = [int(c) for c in h["COUNT"]]
    return [sum(counts[:h["FIELDS"].index(a)]) for a in "xyz"]


def ascii_walk(files):
    """branch items reached by the ASCII files of one batch (files of other kinds take no tiles)"""
    hits, tile = set(), 0
    asc = [f for f in files if b"\nDATA ascii\n" in f]
    for f in asc:
        data, npts, tok = data_section(f), header_points(f), ascii_tok(f)
        if npts == 0:
            if len(files) > 1:
                hits.add("points_0_file_in_batch")
            continue
        n_tiles = -(-len(data) // TILE)
        tb, tile = tile, tile + n_tiles
        if tb in (1023, 1024, 2048):
            hits.add("first_tile_%d" % tb)
        if tb // SCAN_ROUND != (tile - 1) // SCAN_ROUND:
            hits.add("file_across_scan_rounds")
        lines = lines_of(data)
        records = [(s, e) for s, e, r in lines if r]
        for r, (s, e) in enumerate(records[:npts + 1]):
            hits.add("start_chunk_byte_%d" % (s % CHUNK))
            if s % TILE == TILE - 1:
                hits.add("start_tile_byte_4095")
            if s % TILE in (0, 1) and s > TILE:
                hits.add("start_tile_byte_%d" % (TILE + s % TILE))
            if s // TILE != max(s, e - 1) // TILE:
                hits.add("record_across_tiles")
            ntok = len([t for t in data[s:e].replace(b"\t", b" ").replace(b"\r", b" ").split(b" ") if t])
            if r < npts and ntok <= max(tok):
                hits.add("short_record" + ("_in_last_tile" if s // TILE == n_tiles - 1 and n_tiles > 1 else ""))
            if r < npts and (b"\x0b" in data[s:e] or b"\x0c" in data[s:e]):
                hits.add("vt_ff_record" if ntok > max(tok) else "vt_ff_only_line")
        if len(records) > npts and records[npts][0] // TILE == records[npts - 1][0] // TILE:
            hits.add("points_end_inside_tile_with_surplus")
        for s, e, r in lines:
            if not r and e > s and s // TILE != (e - 1) // TILE:
                hits.add("blank_line_across_tiles")
            if e > s and data[e - 1:e] == b"\r" and (e - 1) % TILE == TILE - 1 and e < len(data):
                hits.add("crlf_cr_last_tile_byte")
        if lines and not lines[0][2]:
            hits.add("leading_blank_lines")
        if data[-1:] != b"\n":
            hits.add("no_final_newline")
        if len(data) > TILE and (len(data) + 1) % TILE in (0, 1, 2):
            hits.add("data_len_k4096%s" % {0: "_minus_1", 1: "", 2: "_plus_1"}[(len(data) + 1) % TILE])
        if tok != [0, 1, 2] and max(tok) > 2 and not tok[0] < tok[1] < tok[2]:
            hits.add("count_over_1_fields_ahead_of_permuted_xyz")
    return hits


ASCII_ITEMS = (["start_chunk_byte_%d" % k for k in range(CHUNK)]
               + ["start_tile_byte_4095", "start_tile_byte_4096", "start_tile_byte_4097", "record_across_tiles", "blank_line_across_tiles",
                  "crlf_cr_last_tile_byte", "data_len_k4096", "data_len_k4096_plus_1", "data_len_k4096_minus_1", "leading_blank_lines",
                  "no_final_newline", "points_end_inside_tile_with_surplus", "vt_ff_record", "count_over_1_fields_ahead_of_permuted_xyz",
                  "first_tile_1023", "first_tile_1024", "first_tile_2048", "file_across_scan_rounds", "points_0_file_in_batch"])
ASCII_REJECTS = ["short_record_in_last_tile", "vt_ff_only_line"]


# ---- the gather, restated (gather_segments_kernel, launch_gather) -------------------------------------------------------
def gather_threads(n_points):
    return min(-(-n_points // 256), GATHER_GRID_MAX) * 256


def binary_fields(rec_bytes):
    """a record layout of 12, 13 or 17 bytes with x / y / z float32 and (offset of x, y, z)"""
    return {12: (XYZ, (0, 4, 8)),
            13: ((("label", "U", 1, 1), ("x", "F", 4, 1), ("y", "F", 4, 1), ("z", "F", 4, 1)), (1, 5, 9)),
            17: ((("x", "F", 4, 1), ("label", "U", 1, 1), ("rgb", "U", 4, 1), ("z", "F", 4, 1), ("y", "F", 4, 1)), (0, 13, 9))}[rec_bytes]


def binary_file(xyz, rec_bytes, seed, comment=""):
    n = len(xyz)
    fields, offs = binary_fields(rec_bytes)
    recs = np.random.default_rng(seed).integers(0, 256, (n, rec_bytes), dtype=np.uint8)
    for k, o in enumerate(offs):
        recs[:, o:o + 4] = xyz[:, k].copy().view(np.uint8).reshape(n, 4)
    return pcd_header("binary", n, fields, comment) + recs.tobytes()


def gather_walk_pcd(files):
    """alignments of x / y / z loads of binary records (the batch's bytes start 256-aligned on the device), grid-stride"""
    hits, at, total = set(), 0, 0
    for f in files:
        total += header_points(f)
        if b"\nDATA binary\n" in f:
            n = header_points(f)
            d = at + len(f) - len(data_section(f))
            if n:
                step = len(data_section(f)) // n
                for a, o in enumerate(binary_fields(step)[1]):
                    for m in {(d + o + i * step) % 4 for i in range(min(n, 4))}:
                        hits.add("record_%d_%s_align_%d" % (step, "xyz"[a], m))
        at += len(f)
    if total > gather_threads(total):
        hits.add("grid_stride_binary_pcd")
    return hits


GATHER_ITEMS = (["record_%d_%s_align_%d" % (s, a, m) for s in (12, 13, 17) for a in "xyz" for m in range(4)]
                + ["grid_stride_binary_pcd", "grid_stride_pointcloud2", "pointcloud2_1000_clouds_empty_and_one_point"])


def pc2_batch(n_clouds, seed):
    """PointCloud2 clouds of assorted layouts, empty and one-point clouds interleaved: (data, byte offsets, layouts, want)"""
    rng = np.random.default_rng(seed)
    layouts = [(16, 0, 4, 8), (13, 1, 5, 9), (17, 9, 1, 13), (12, 8, 4, 0), (32, 4, 12, 20)]
    sizes = [(0, 1, 3, 0, 1, 40, 0, 2)[c % 8] for c in range(n_clouds)]
    bufs, lays, want = [], [], []
    for c, n in enumerate(sizes):
        step, ox, oy, oz = layouts[c % 5]
        xyz = rng.normal(size=(n, 3)).astype(np.float32)
        b = rng.integers(0, 256, (n, step), dtype=np.uint8)
        for k, o in enumerate((ox, oy, oz)):
            b[:, o:o + 4] = xyz[:, k].copy().view(np.uint8).reshape(n, 4)
        bufs.append(b.reshape(-1))
        lays.append(layouts[c % 5])
        want.append(xyz)
    return np.concatenate(bufs), np.cumsum([0] + [len(b) for b in bufs]), lays, want


def pc2_walk(offs, lays):
    sizes = [(offs[c + 1] - offs[c]) // lays[c][0] for c in range(len(lays))]
    hits = set()
    if len(sizes) >= 1000 and any(sizes[c] == 0 and c and sizes[c - 1] and c + 1 < len(sizes) and sizes[c + 1] for c in range(len(sizes))) \
            and 1 in sizes:
        hits.add("pointcloud2_1000_clouds_empty_and_one_point")
    if sum(sizes) > gather_threads(sum(sizes)):
        hits.add("grid_stride_pointcloud2")
    return hits


BIG_POINTS = 700_000


def alignment_batch():
    """12-, 13- and 17-byte records, the 12-byte ones with their data at all four offsets mod 4"""
    rng = np.random.default_rng(40)
    files, at = [], 0
    for k, step in enumerate((12, 12, 12, 12, 13, 17)):
        xyz = rng.normal(size=(37 + k, 3)).astype(np.float32)
        f = [binary_file(xyz, step, k, comment=" " * c) for c in range(4)]
        f = [g for g in f if (at + len(g) - len(data_section(g))) % 4 == k % 4][0]    # data of the k-th file at offset k mod 4
        files.append(f)
        at += len(f)
    return files


def big_binary_batch():
    rng = np.random.default_rng(41)
    return [binary_file(rng.normal(size=(400_000, 3)).astype(np.float32), 12, 1),
            binary_file(rng.normal(size=(BIG_POINTS - 400_000, 3)).astype(np.float32), 17, 2)]


# ---- CPU: references, restatements, coverage ----------------------------------------------------------------------------
def _fnv1a(b):
    a = np.frombuffer(b, np.uint8)
    h = 1469598103934665603
    for x in a.tolist():
        h = ((h ^ x) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


@pytest.fixture(scope="module")
def cli():
    from haf_grasping_b200 import build
    return build.build_cli()


def cpp_read(cli, tmp_path, name, raw_bytes):
    """(points, fnv1a of the xyz bytes) or the error text of the C++ reader"""
    f = tmp_path / (name + ".pcd")
    f.write_bytes(raw_bytes)
    r = subprocess.run([cli, "--pcd", str(f), "--dump-pcd"], capture_output=True, text=True)
    if r.returncode:
        return r.stderr
    n, h = r.stdout.split()
    return int(n), int(h)


def test_python_lzf_rejects_truncated_literal():
    from haf_grasping_b200 import pcd
    for stream, out_len in ((bytes([5, 1, 2]), 6), (bytes([3, 1, 2, 3, 4]), 2), (bytes([0xE0]), 9), (bytes([0x20]), 3)):
        with pytest.raises(ValueError, match="corrupt LZF stream"):
            pcd.lzf_decompress(stream, out_len)


def test_host_readers_split_on_blank_tab_cr_only(cli, tmp_path):
    """vertical tab and form feed are token characters in both host readers, as on the device"""
    from haf_grasping_b200 import pcd
    body = b"1.5\x0b 2 3\n1\x0b2 3 4\n\x0c1 2 3\n4 5 6\x0c\n7\t8\r9\n"
    f = pcd_header("ascii", 5) + body
    want = np.array([[1.5, 2, 3], [1, 3, 4], [0, 2, 3], [4, 5, 6], [7, 8, 9]], np.float32)
    assert pcd.read_pcd_bytes(f).tobytes() == want.tobytes()
    assert cpp_read(cli, tmp_path, "vtff", f) == (5, _fnv1a(want.tobytes()))
    bad = pcd_header("ascii", 2) + b"1 2 3\n\x0c\n4 5 6\n"       # a line of one form feed is a record, and a short one
    with pytest.raises(ValueError, match="short ASCII record"):
        pcd.read_pcd_bytes(bad)
    assert "short ASCII record" in cpp_read(cli, tmp_path, "ffline", bad)


def test_lzf_reference_pinned_to_both_host_readers(cli, tmp_path):
    from haf_grasping_b200 import pcd
    for name, (stream, out_len) in {**lzf_valid_cases(), **lzf_bad_cases()}.items():
        blob, verdict = lzf_reference(stream, out_len)
        walk_hits, walk_verdict = lzf_walk(stream, out_len)
        assert walk_verdict == verdict, name
        f = lzf_pcd(stream, out_len)
        cpp = cpp_read(cli, tmp_path, name, f)
        if verdict == "ok":
            assert pcd.lzf_decompress(stream, out_len) == blob, name
            assert pcd.read_pcd_bytes(f).tobytes() == blob_xyz(blob).tobytes() and len(blob) % 12 == 0, name
            assert cpp == (out_len // 12, _fnv1a(blob_xyz(blob).tobytes())), name
        else:
            with pytest.raises(ValueError, match="corrupt LZF stream"):
                pcd.lzf_decompress(stream, out_len)
            assert "corrupt LZF stream" in cpp, (name, cpp)


def test_lzf_assembler_round_trips():
    """the builder's tokens are what the reference decoder reads back, token for token"""
    B = _tokens_case()
    blob, verdict = lzf_reference(B.stream(), B.op)
    assert verdict == "ok" and len(blob) == B.op
    out = bytearray()
    for t in B.tokens:
        if t[0] == "lit":
            out += t[1]
        else:
            for _ in range(t[1]):
                out.append(out[-t[2]])
    assert bytes(out) == blob


def test_ascii_catalogue_host_readers_agree(cli, tmp_path):
    from haf_grasping_b200 import pcd
    for name, f in ascii_valid_cases().items():
        want = pcd.read_pcd_bytes(f)
        assert len(want) == header_points(f) > 0, name
        assert cpp_read(cli, tmp_path, name, f) == (len(want), _fnv1a(want.tobytes())), name
    for name, f in ascii_bad_cases().items():
        with pytest.raises(ValueError, match="short ASCII record"):
            pcd.read_pcd_bytes(f)
        assert "short ASCII record" in cpp_read(cli, tmp_path, name, f), name
    for name, f in (("aligned", alignment_batch()[0]), ("rec17", alignment_batch()[-1])):
        want = pcd.read_pcd_bytes(f)
        assert cpp_read(cli, tmp_path, name, f) == (len(want), _fnv1a(want.tobytes())), name


def _unique_items(per_case, items):
    """each case must reach a listed item no other case reaches"""
    for name, h in per_case.items():
        others = set().union(*[g for k, g in per_case.items() if k != name])
        assert (h - others) & set(items), name


def test_cases_cover_every_branch():
    valid = {k: lzf_walk(*v)[0] for k, v in lzf_valid_cases().items()}
    bad = {k: lzf_walk(*v)[0] for k, v in lzf_bad_cases().items()}
    reached = set().union(*valid.values(), *bad.values())
    assert not set(LZF_ITEMS) - reached, sorted(set(LZF_ITEMS) - reached)
    assert not set(LZF_REJECTS) - set().union(*bad.values()), sorted(set(LZF_REJECTS) - set().union(*bad.values()))
    _unique_items(valid, LZF_ITEMS)
    _unique_items(bad, LZF_ITEMS + LZF_REJECTS)

    asc = {k: ascii_walk([f]) for k, f in ascii_valid_cases().items()}
    asc["scan_round_batch"] = ascii_walk(scan_round_batch())
    reached = set().union(*asc.values())
    assert not set(ASCII_ITEMS) - reached, sorted(set(ASCII_ITEMS) - reached)
    _unique_items(asc, ASCII_ITEMS)
    bad = {k: ascii_walk([f]) for k, f in ascii_bad_cases().items()}
    assert not set(ASCII_REJECTS) - set().union(*bad.values()), bad
    _unique_items(bad, ASCII_REJECTS)

    g = {"alignment": gather_walk_pcd(alignment_batch()), "big_binary": gather_walk_pcd(big_binary_batch()),
         "pc2_batch": pc2_walk(*pc2_batch(1200, 50)[1:3]),
         "pc2_big": pc2_walk(np.array([0, BIG_POINTS * 16]), [(16, 0, 4, 8)])}
    reached = set().union(*g.values())
    assert not set(GATHER_ITEMS) - reached, sorted(set(GATHER_ITEMS) - reached)
    _unique_items(g, GATHER_ITEMS)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu(hg, tmp_models):
    g = hg.GraspSearch(FEATURES, RANGE, tmp_models(256))
    yield g
    g.close()


def launches(files):
    """kernels one decode call runs: ASCII count / scan / parse, LZF, gather -- each kind present, files of POINTS 0 aside"""
    kinds = {f.split(b"\nDATA ")[1].split(b"\n")[0] for f in files if header_points(f)}
    return 3 * (b"ascii" in kinds) + (b"binary_compressed" in kinds) + bool(kinds & {b"binary", b"binary_compressed"})


def decode_checked(gpu, files, want):
    l0 = gpu.launch_count()
    got = gpu.pcd_decode_batch_to_host(files)
    assert gpu.launch_count() - l0 == launches(files)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape and g.tobytes() == w.tobytes(), i


@pytest.mark.gpu
def test_lzf_catalogue(gpu, hg):
    valid = lzf_valid_cases()
    files, want = [], []
    for name, (stream, out_len) in valid.items():
        f = lzf_pcd(stream, out_len)
        w = blob_xyz(lzf_reference(stream, out_len)[0])
        assert gpu.pcd_decode_to_host(f).tobytes() == w.tobytes(), name
        files.append(f)
        want.append(w)
    decode_checked(gpu, files, want)
    decode_checked(gpu, files[::-1], want[::-1])
    for j, (name, (stream, out_len)) in enumerate(lzf_bad_cases().items()):
        f = lzf_pcd(stream, out_len)
        with pytest.raises(hg.HafError) as e:
            gpu.pcd_decode(f)
        assert e.value.code == -2 and "corrupt LZF stream" in str(e.value), (name, str(e.value))
        k = j % (len(files) + 1)
        with pytest.raises(hg.HafError) as e:
            gpu.pcd_decode_batch(files[:k] + [f] + files[k:])
        assert e.value.code == -2 and ("PCD file %d: corrupt LZF stream" % k) in str(e.value), (name, str(e.value))
    decode_checked(gpu, files, want)                     # the context decodes the next good batch


@pytest.mark.gpu
def test_ascii_catalogue(gpu, hg):
    from haf_grasping_b200 import pcd
    cases = ascii_valid_cases()
    files = list(cases.values())
    want = [pcd.read_pcd_bytes(f) for f in files]
    for name, f, w in zip(cases, files, want):
        l0 = gpu.launch_count()
        assert gpu.pcd_decode_to_host(f).tobytes() == w.tobytes(), name
        assert gpu.launch_count() - l0 == 3
    empty = ascii_file(AsciiBody(0), points=0)
    decode_checked(gpu, [empty] + files[:3] + [empty] + files[3:], [want[0][:0]] + want[:3] + [want[0][:0]] + want[3:])
    for j, (name, f) in enumerate(ascii_bad_cases().items()):
        with pytest.raises(hg.HafError) as e:
            gpu.pcd_decode(f)
        assert e.value.code == -2 and "short ASCII record" in str(e.value), (name, str(e.value))
        k = 2 + j
        with pytest.raises(hg.HafError) as e:
            gpu.pcd_decode_batch(files[:k] + [f] + files[k:])
        assert ("PCD file %d: short ASCII record" % k) in str(e.value), (name, str(e.value))


@pytest.mark.gpu
def test_ascii_scan_rounds_batch(gpu):
    from haf_grasping_b200 import pcd
    files = scan_round_batch()
    want = [pcd.read_pcd_bytes(f) if header_points(f) else np.zeros((0, 3), np.float32) for f in files]
    decode_checked(gpu, files, want)


@pytest.mark.gpu
def test_binary_record_alignments(gpu):
    from haf_grasping_b200 import pcd
    files = alignment_batch()
    want = [pcd.read_pcd_bytes(f) for f in files]
    decode_checked(gpu, files, want)
    for f, w in zip(files, want):
        assert gpu.pcd_decode_to_host(f).tobytes() == w.tobytes()
    # beside ASCII and LZF files, whose sections shift every later binary section
    lz = lzf_valid_cases()["tokens"]
    mixed = [files[0], ascii_valid_cases()["vt_ff"], files[4], lzf_pcd(*lz), files[5], files[1]]
    decode_checked(gpu, mixed, [pcd.read_pcd_bytes(f) for f in mixed])


@pytest.mark.gpu
def test_gather_grid_stride(gpu):
    import torch
    from haf_grasping_b200 import pcd
    files = big_binary_batch()
    want = [pcd.read_pcd_bytes(f) for f in files]
    assert sum(len(w) for w in want) == BIG_POINTS > gather_threads(BIG_POINTS)
    decode_checked(gpu, files, want)
    xyz = np.concatenate(want)
    buf = np.random.default_rng(42).integers(0, 256, (BIG_POINTS, 16), dtype=np.uint8)
    for k, o in enumerate((0, 4, 8)):
        buf[:, o:o + 4] = xyz[:, k].copy().view(np.uint8).reshape(BIG_POINTS, 4)
    data = buf.reshape(-1)
    for src in (data, torch.from_numpy(data).cuda()):
        l0 = gpu.launch_count()
        _, po = gpu.pointcloud2_batch_to_xyz(src, [0, len(data)], [(16, 0, 4, 8)])
        assert gpu.launch_count() - l0 == 1 and list(po) == [0, BIG_POINTS]
        assert gpu.debug_pcd_xyz(BIG_POINTS).tobytes() == xyz.tobytes()


@pytest.mark.gpu
def test_pointcloud2_many_clouds(gpu):
    import torch
    data, offs, lays, want = pc2_batch(1200, 50)
    for src in (data, torch.from_numpy(data).cuda()):
        l0 = gpu.launch_count()
        _, po = gpu.pointcloud2_batch_to_xyz(src, offs, lays)
        assert gpu.launch_count() - l0 == 1
        assert list(po) == list(np.cumsum([0] + [len(w) for w in want]))
        got = gpu.debug_pcd_xyz(int(po[-1]))
        for c, w in enumerate(want):
            assert got[po[c]:po[c + 1]].tobytes() == w.tobytes(), c
