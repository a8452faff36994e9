"""FLAC container plumbing kept on the host: metadata blocks and VORBIS_COMMENT tags.

Frames (all codec arithmetic) are produced/consumed by the CUDA engine; this
module only writes/reads the byte-level metadata the reference obtains from
libFLAC's stream header (docs/sonos-pyflac.txt:2200-2212) and from mutagen
(reference converter.py:263-390).  No mutagen dependency: VORBIS_COMMENT is a
little-endian length-prefixed list (RFC 9639 section 8.6).
"""
from __future__ import annotations

import struct
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

VENDOR = "flac-raster-b200 0.1 (sm_100a CUDA FLAC engine)"

BLOCK_STREAMINFO = 0
BLOCK_PADDING = 1
BLOCK_APPLICATION = 2
BLOCK_VORBIS_COMMENT = 4

# APPLICATION block of this engine: the stream's seek index (include/flacraster_b200.h, frb_encode_index).  Other decoders
# skip APPLICATION blocks they do not know (libFLAC's default metadata filter, RFC 9639 section 8.4).
SEEK_INDEX_ID = b"frbI"


@dataclass
class StreamInfo:
    min_blocksize: int
    max_blocksize: int
    min_framesize: int
    max_framesize: int
    sample_rate: int
    channels: int
    bits_per_sample: int
    total_samples: int
    md5: bytes = b"\0" * 16

    def pack(self) -> bytes:
        v = ((self.sample_rate & 0xFFFFF) << 44) | ((self.channels - 1) << 41) | \
            ((self.bits_per_sample - 1) << 36) | (self.total_samples & 0xFFFFFFFFF)
        return (struct.pack(">HH", self.min_blocksize, self.max_blocksize)
                + self.min_framesize.to_bytes(3, "big") + self.max_framesize.to_bytes(3, "big")
                + v.to_bytes(8, "big") + self.md5)

    @classmethod
    def unpack(cls, b: bytes) -> "StreamInfo":
        if len(b) < 34:
            raise ValueError("STREAMINFO too short")
        mn, mx = struct.unpack(">HH", b[:4])
        v = int.from_bytes(b[10:18], "big")
        return cls(mn, mx, int.from_bytes(b[4:7], "big"), int.from_bytes(b[7:10], "big"),
                   v >> 44, ((v >> 41) & 7) + 1, ((v >> 36) & 31) + 1, v & 0xFFFFFFFFF, bytes(b[18:34]))


@dataclass
class FlacHeader:
    streaminfo: StreamInfo
    tags: Dict[str, List[str]] = field(default_factory=dict)
    vendor: str = ""
    first_frame_offset: int = 0
    applications: Dict[bytes, bytes] = field(default_factory=dict)     # APPLICATION blocks: 4-byte id -> data


def pack_seek_index(channels: int, blocksize: int, frame_bytes, sub_bitoff) -> bytes:
    """Body of the "frbI" APPLICATION block: little-endian u32 arrays as the GPU decoder takes them.
    Layout: u8 version (1), u8 channels, u16 0, u32 blocksize, u32 n_frames, u32 frame_bytes[n_frames],
    u32 sub_bitoff[n_frames * channels] (left out for single-channel streams: a subframe starts right behind the frame header)."""
    import numpy as np
    fb = np.ascontiguousarray(frame_bytes, dtype="<u4")
    out = [struct.pack("<BBHII", 1, channels, 0, blocksize, fb.size), fb.tobytes()]
    if channels > 1:
        sb = np.ascontiguousarray(sub_bitoff, dtype="<u4")
        if sb.size != fb.size * channels:
            raise ValueError("seek index: subframe table does not match the frame count")
        out.append(sb.tobytes())
    return b"".join(out)


def unpack_seek_index(data: bytes, channels: int, blocksize: int, n_frames: int):
    """-> (frame_bytes u32[n_frames], sub_bitoff u32[n_frames*channels] or None), or None when the block does not describe
    this stream (wrong version, geometry or length): the caller then decodes without an index."""
    import numpy as np
    if len(data) < 12:
        return None
    ver, ch, _, bs, nf = struct.unpack_from("<BBHII", data, 0)
    if ver != 1 or ch != channels or bs != blocksize or nf != n_frames:
        return None
    need = 12 + 4 * nf + (4 * nf * ch if ch > 1 else 0)
    if len(data) != need:
        return None
    fb = np.frombuffer(data, dtype="<u4", count=nf, offset=12)
    sb = np.frombuffer(data, dtype="<u4", count=nf * ch, offset=12 + 4 * nf) if ch > 1 else None
    return fb, sb


def _block(block_type: int, body: bytes, last: bool) -> bytes:
    return bytes([(0x80 if last else 0) | block_type]) + len(body).to_bytes(3, "big") + body


def pack_vorbis_comment(tags: Dict[str, str] | List[Tuple[str, str]], vendor: str = VENDOR) -> bytes:
    items = list(tags.items()) if isinstance(tags, dict) else list(tags)
    v = vendor.encode("utf-8")
    out = [struct.pack("<I", len(v)), v, struct.pack("<I", len(items))]
    for k, val in items:
        e = f"{k}={val}".encode("utf-8")
        out += [struct.pack("<I", len(e)), e]
    return b"".join(out)


def unpack_vorbis_comment(body: bytes) -> Tuple[str, Dict[str, List[str]]]:
    pos = 0
    (vl,) = struct.unpack_from("<I", body, pos); pos += 4
    vendor = body[pos:pos + vl].decode("utf-8", "replace"); pos += vl
    (n,) = struct.unpack_from("<I", body, pos); pos += 4
    tags: Dict[str, List[str]] = {}
    for _ in range(n):
        (el,) = struct.unpack_from("<I", body, pos); pos += 4
        e = body[pos:pos + el].decode("utf-8", "replace"); pos += el
        if "=" in e:
            k, val = e.split("=", 1)
            tags.setdefault(k.upper(), []).append(val)
    return vendor, tags


def build_header(si: StreamInfo, tags: Optional[Dict[str, str]] = None, vendor: str = VENDOR,
                 padding: int = 0, seek_index: Optional[bytes] = None) -> bytes:
    """'fLaC' + STREAMINFO + VORBIS_COMMENT [+ APPLICATION "frbI" (pack_seek_index)] [+ PADDING]."""
    vc = pack_vorbis_comment(tags or {}, vendor)
    out = b"fLaC" + _block(BLOCK_STREAMINFO, si.pack(), False) + _block(BLOCK_VORBIS_COMMENT, vc, padding <= 0 and seek_index is None)
    if seek_index is not None:
        if len(seek_index) + 4 >= 1 << 24:
            seek_index = None                     # a metadata block holds < 16 MiB: very long streams go without an index
            out = b"fLaC" + _block(BLOCK_STREAMINFO, si.pack(), False) + _block(BLOCK_VORBIS_COMMENT, vc, padding <= 0)
        else:
            out += _block(BLOCK_APPLICATION, SEEK_INDEX_ID + seek_index, padding <= 0)
    if padding > 0:
        out += _block(BLOCK_PADDING, b"\0" * padding, True)
    return out


def parse_header(data: bytes | memoryview) -> FlacHeader:
    """Walk the metadata chain; returns STREAMINFO, tags and the first frame offset."""
    if len(data) < 8 or bytes(data[:4]) != b"fLaC":
        raise ValueError("not a FLAC stream (missing fLaC marker)")
    pos, last, si, tags, vendor, apps = 4, False, None, {}, "", {}
    while not last:
        if pos + 4 > len(data):
            raise ValueError("truncated metadata")
        h = data[pos]
        last = bool(h & 0x80)
        btype = h & 0x7F
        blen = int.from_bytes(bytes(data[pos + 1:pos + 4]), "big")
        pos += 4
        if pos + blen > len(data):
            raise ValueError("truncated metadata block")
        body = bytes(data[pos:pos + blen])
        if btype == BLOCK_STREAMINFO:
            si = StreamInfo.unpack(body)
        elif btype == BLOCK_VORBIS_COMMENT:
            vendor, tags = unpack_vorbis_comment(body)
        elif btype == BLOCK_APPLICATION and blen >= 4:
            apps[body[:4]] = body[4:]
        elif btype == 127:
            raise ValueError("invalid metadata block type")
        pos += blen
    if si is None:
        raise ValueError("missing STREAMINFO")
    return FlacHeader(si, tags, vendor, pos, apps)


def read_header(read, first: int = 1 << 16) -> FlacHeader:
    """parse_header for a stream that is read piece by piece: read(start, n) returns up to n bytes from `start` (a local
    file or HTTP range requests).  A first piece of `first` bytes; a block that reaches beyond it is read in one more piece
    together with the header of the block behind it.  The body of a PADDING block at the end of the chain is not read."""
    buf = bytearray(read(0, first))
    if len(buf) < 8 or bytes(buf[:4]) != b"fLaC":
        raise ValueError("not a FLAC stream (missing fLaC marker)")

    def have(end: int) -> bool:
        if end > len(buf):
            buf.extend(read(len(buf), end - len(buf)))
        return end <= len(buf)

    pos, last, si, tags, vendor, apps = 4, False, None, {}, "", {}
    while not last:
        if not have(pos + 4):
            raise ValueError("truncated metadata")
        h = buf[pos]
        last = bool(h & 0x80)
        btype = h & 0x7F
        blen = int.from_bytes(bytes(buf[pos + 1:pos + 4]), "big")
        pos += 4
        if btype == 127:
            raise ValueError("invalid metadata block type")
        if btype in (BLOCK_STREAMINFO, BLOCK_VORBIS_COMMENT, BLOCK_APPLICATION) or not last:
            if not have(pos + blen + (0 if last else 4)) and not have(pos + blen):
                raise ValueError("truncated metadata block")
            body = bytes(buf[pos:pos + blen])
            if btype == BLOCK_STREAMINFO:
                si = StreamInfo.unpack(body)
            elif btype == BLOCK_VORBIS_COMMENT:
                vendor, tags = unpack_vorbis_comment(body)
            elif blen >= 4:
                apps[body[:4]] = body[4:]
        pos += blen
    if si is None:
        raise ValueError("missing STREAMINFO")
    return FlacHeader(si, tags, vendor, pos, apps)
