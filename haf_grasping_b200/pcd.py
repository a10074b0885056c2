"""Host-side PCD v0.7 ingest (ASCII, binary, binary_compressed) -- the data format the reference
client feeds the action server (reference src/calc_grasppoints_action_client.cpp:137-157,
pcl::io::loadPCDFile).  ROS/PCL-free; returns float32 [n, 3] xyz.

PCL semantics reproduced:
  * ASCII: exactly POINTS records are consumed, extra lines are ignored (pcd4/pcd5 declare 200 points
    but carry 208 lines); tokens are parsed straight to float32 (strtof), not via double.
  * binary_compressed: uint32 compressed size, uint32 uncompressed size, LZF stream, fields stored
    struct-of-arrays (all x, then all y, then all z).
"""
from __future__ import annotations

import ctypes
import ctypes.util
import struct

import numpy as np

_libc = ctypes.CDLL(ctypes.util.find_library("c") or "libc.so.6")
_libc.strtof.restype = ctypes.c_float
_libc.strtof.argtypes = [ctypes.c_char_p, ctypes.c_void_p]


def _strtof(tok: bytes) -> float:
    return _libc.strtof(tok, None)


def ascii_tokens(line: bytes) -> list:
    """the tokens of one line of an ASCII DATA section: fields are separated by runs of blank, tab and CR only (PCL's
    boost::split on "\\t\\r "); vertical tab and form feed are token characters, as on the device (csrc/pcd_ingest.cuh)"""
    return [t for t in line.replace(b"\t", b" ").replace(b"\r", b" ").split(b" ") if t]


def ascii_token_value(tok: bytes) -> float:
    """a FLOAT32 token: strtof of its longest numeric prefix.  strtof would skip a leading vertical tab or form feed; those
    are token characters here, so such a token has no numeric prefix and reads 0, as on the device."""
    return 0.0 if tok[:1] in (b"\v", b"\f") else _strtof(tok)


def lzf_decompress(src: bytes, out_len: int) -> bytes:
    """liblzf stream decoder (the codec PCL embeds for DATA binary_compressed).  Rejects, with ValueError("corrupt LZF
    stream ..."), exactly the streams the C++ reader (csrc/host/pcd_io.hpp) and the device kernel reject: a token cut off
    by the end of the input, a reference before the start of the output, a token past out_len, a stream short of out_len."""
    out = bytearray(out_len)
    ip, op, n = 0, 0, len(src)
    while ip < n:
        ctrl = src[ip]
        ip += 1
        if ctrl < 32:  # literal run of ctrl+1 bytes
            ln = ctrl + 1
            if op + ln > out_len or ip + ln > n:
                raise ValueError("corrupt LZF stream: literal run past the end of the input or the output")
            out[op:op + ln] = src[ip:ip + ln]
            ip += ln
            op += ln
        else:  # back reference
            ln = ctrl >> 5
            if ln == 7:
                if ip >= n:
                    raise ValueError("corrupt LZF stream: no length byte")
                ln += src[ip]
                ip += 1
            if ip >= n:
                raise ValueError("corrupt LZF stream: no distance byte")
            ref = op - ((ctrl & 0x1F) << 8) - src[ip] - 1
            ip += 1
            ln += 2
            if ref < 0 or op + ln > out_len:
                raise ValueError("corrupt LZF stream: reference before the start or past the end of the output")
            if ref + ln <= op:
                out[op:op + ln] = out[ref:ref + ln]
            else:  # overlapping copy, byte by byte
                for k in range(ln):
                    out[op + k] = out[ref + k]
            op += ln
    if op != out_len:
        raise ValueError(f"corrupt LZF stream: decoded to {op} bytes, expected {out_len}")
    return bytes(out)


def read_pcd(path: str) -> np.ndarray:
    with open(path, "rb") as fh:
        return read_pcd_bytes(fh.read(), path)


def header_points(raw) -> int:
    """the point count a PCD header declares: POINTS, else WIDTH * HEIGHT (HEIGHT defaults to 1).  raw: bytes-like; only the
    header is read."""
    mv = memoryview(raw).cast("B")
    n = 4096
    while True:
        head = bytes(mv[:n])
        hdr = {}
        lines = head.split(b"\n")
        complete = lines if n >= len(mv) else lines[:-1]
        for ln in complete:
            toks = ln.split()
            if not toks or toks[0].startswith(b"#"):
                continue
            hdr[toks[0]] = toks[1:]
            if toks[0] == b"DATA":
                break
        if b"DATA" in hdr or n >= len(mv):
            break
        n *= 4
    if b"POINTS" in hdr:
        return int(hdr[b"POINTS"][0])
    return int(hdr.get(b"WIDTH", [b"0"])[0]) * int(hdr.get(b"HEIGHT", [b"1"])[0])


def read_pcd_bytes(raw: bytes, path: str = "<bytes>") -> np.ndarray:
    pos = 0
    hdr = {}
    data_kind = None
    while True:
        nl = raw.index(b"\n", pos)
        line = raw[pos:nl].decode("ascii", "replace").strip()
        pos = nl + 1
        if not line or line.startswith("#"):
            continue
        key, _, rest = line.partition(" ")
        hdr[key.upper()] = rest.split()
        if key.upper() == "DATA":
            data_kind = rest.strip().lower()
            break
    fields = [f.lower() for f in hdr["FIELDS"]]
    sizes = [int(s) for s in hdr["SIZE"]]
    types = hdr["TYPE"]
    counts = [int(c) for c in hdr.get("COUNT", ["1"] * len(fields))]
    npts = int(hdr["POINTS"][0]) if "POINTS" in hdr else int(hdr["WIDTH"][0]) * int(hdr["HEIGHT"][0])
    for ax in "xyz":
        if ax not in fields:
            raise ValueError(f"PCD {path}: no field '{ax}'")
    if data_kind == "ascii":
        # column offsets of x,y,z in a record (COUNT > 1 fields occupy several tokens)
        tok_off = np.concatenate([[0], np.cumsum(counts)])
        cols = [int(tok_off[fields.index(ax)]) for ax in "xyz"]
        out = np.empty((npts, 3), np.float32)
        idx = 0
        for ln in raw[pos:].split(b"\n"):
            if idx >= npts:
                break
            toks = ascii_tokens(ln)
            if not toks:
                continue
            if len(toks) <= max(cols):
                raise ValueError(f"PCD {path}: short ASCII record")
            for k, c in enumerate(cols):
                t = toks[c]
                out[idx, k] = np.float32("nan") if t.lower() == b"nan" else ascii_token_value(t)
            idx += 1
        if idx != npts:
            raise ValueError(f"PCD {path}: {idx} records, header says {npts}")
        return out
    np_types = {("F", 4): "<f4", ("F", 8): "<f8", ("U", 1): "u1", ("U", 2): "<u2", ("U", 4): "<u4",
                ("I", 1): "i1", ("I", 2): "<i2", ("I", 4): "<i4"}
    if data_kind == "binary":
        dt = np.dtype([(f, np_types[(t, s)], (c,)) for f, t, s, c in zip(fields, types, sizes, counts)])
        rec = np.frombuffer(raw, dtype=dt, count=npts, offset=pos)
        return np.stack([rec[ax][:, 0].astype(np.float32) for ax in "xyz"], axis=1)
    if data_kind == "binary_compressed":
        comp, uncomp = struct.unpack_from("<II", raw, pos)
        if pos + 8 + comp > len(raw):
            raise ValueError(f"PCD {path}: compressed PCD truncated")
        blob = lzf_decompress(raw[pos + 8:pos + 8 + comp], uncomp)
        out = np.empty((npts, 3), np.float32)
        off = 0
        offs = {}
        for f, t, s, c in zip(fields, types, sizes, counts):
            offs[f] = (off, np_types[(t, s)], c)
            off += npts * s * c
        for k, ax in enumerate("xyz"):
            o, dt, c = offs[ax]
            out[:, k] = np.frombuffer(blob, dtype=dt, count=npts * c, offset=o)[::c].astype(np.float32)
        return out
    raise ValueError(f"PCD {path}: unsupported DATA {data_kind}")
