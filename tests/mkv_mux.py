"""Test infrastructure: a small Matroska writer (EBML, RFC 8794 / RFC 9559) that wraps the Annex-B streams of
synth.generate() in a Matroska file, with knobs for the variants the Matroska front end has to read.

Every IDR NAL unit becomes one frame.  The first parameter sets go into the avcC of the track's CodecPrivate; those
that come later (a stream whose parameter sets change), or all of them with in_band, stay in band at the start of
the frame that follows them.  So the NAL units come out in the order of the Annex-B stream."""
from __future__ import annotations

import random
import struct

from mp4_mux import nal_units

UNKNOWN8 = b"\x01\xff\xff\xff\xff\xff\xff\xff"


def vint(n: int, width: int = 0) -> bytes:
    """An EBML size of `width` bytes (0: the shortest that holds n without being all ones)."""
    w = width or next(w for w in range(1, 9) if n < (1 << (7 * w)) - 1)
    return (n | 1 << (7 * w)).to_bytes(w, "big")


def el(eid: int, *parts: bytes, size_width: int = 0) -> bytes:
    body = b"".join(parts)
    return eid.to_bytes((eid.bit_length() + 7) // 8, "big") + vint(len(body), size_width) + body


def uint(eid: int, v: int) -> bytes:
    return el(eid, v.to_bytes(max(1, (v.bit_length() + 7) // 8), "big"))


def avcc(sps: list[bytes], pps: list[bytes], length_size: int) -> bytes:
    first = sps[0] if sps else bytes(4)
    out = bytes([1, first[1] if sps else 66, first[2] if sps else 0, first[3] if sps else 30,
                 0xFC | (length_size - 1), 0xE0 | len(sps)])
    out += b"".join(struct.pack(">H", len(s)) + s for s in sps)
    return out + bytes([len(pps)]) + b"".join(struct.pack(">H", len(p)) + p for p in pps)


def signed_vint(d: int) -> bytes:
    """A signed EBML lace size difference."""
    w = next(w for w in range(1, 9) if abs(d) < (1 << (7 * w - 1)) - 1)
    return vint(d + (1 << (7 * w - 1)) - 1, w)


def lace(frames: list[bytes], kind: str) -> tuple[int, bytes]:
    """(lacing bits of the flags byte, lace header + frames)."""
    if len(frames) == 1 and kind == "none":
        return 0, frames[0]
    head = bytes([len(frames) - 1])
    if kind == "xiph":
        for f in frames[:-1]:
            head += b"\xff" * (len(f) // 255) + bytes([len(f) % 255])
        return 0x02, head + b"".join(frames)
    if kind == "ebml":
        if len(frames) > 1:
            head += vint(len(frames[0]))
        for a, b in zip(frames, frames[1:-1]):
            head += signed_vint(len(b) - len(a))
        return 0x06, head + b"".join(frames)
    if kind == "fixed":
        assert len({len(f) for f in frames}) == 1
        return 0x04, head + b"".join(frames)
    raise ValueError(kind)


def mux(stream: bytes, *, length_size: int = 4, segment_unknown: bool = False, cluster_unknown: bool = False,
        block_group: bool = False, lacing: str = "none", per_block: int = 1, per_cluster: int = 2,
        audio_first: bool = False, seek_cues_void: bool = False, in_band: bool = False,
        damaged_frame: tuple[int, list[bytes]] | None = None, codec_id: bytes = b"V_MPEG4/ISO/AVC",
        codec_private: bool = True, content_encodings: bool = False, doctype: bytes = b"matroska",
        video_track: bool = True, seed: int = 1) -> bytes:
    """Matroska file holding the NAL units of the Annex-B `stream`.

    length_size       1, 2 or 4 byte NAL length fields (lengthSizeMinusOne + 1)
    segment_unknown   Segment of unknown size (8-byte all-ones size)
    cluster_unknown   Clusters of unknown size (1-byte 0xFF size)
    block_group       Blocks inside BlockGroups (with a BlockDuration) instead of SimpleBlocks
    lacing            "none", "xiph", "ebml" or "fixed" (fixed pads the frames of a block to one size with filler
                      NAL units); per_block frames go into one block
    per_cluster       blocks per Cluster
    audio_first       an audio track (A_AAC, number 1) in front of the video track, its blocks interleaved
    seek_cues_void    a SeekHead and a Void element before Info, and Cues at the end
    in_band           every parameter set in band; CodecPrivate holds empty lists
    damaged_frame     (k, NAL units): after frame k, one more frame holding these NAL units whose last length field
                      runs past the end of the frame
    codec_id, codec_private, content_encodings, doctype, video_track: for the refusal cases
    """
    rng = random.Random(seed)
    lfmt = {1: ">B", 2: ">H", 4: ">I"}[length_size]
    frames, pending, first_ps = [], [], None
    for nal in nal_units(stream):
        t = nal[0] & 31
        if t in (7, 8):
            pending.append(nal)
            continue
        assert t == 5, f"unexpected NAL type {t}"
        if first_ps is None and not in_band:
            first_ps, pending = pending, []
        frames.append(pending + [nal])
        pending = []
    if damaged_frame is not None:
        frames.insert(damaged_frame[0] + 1, damaged_frame[1])
    datas = [b"".join(struct.pack(lfmt, len(n)) + n for n in f) for f in frames]
    if damaged_frame is not None:
        k, last = damaged_frame[0] + 1, damaged_frame[1][-1]
        cut = len(datas[k]) - len(last) - length_size
        datas[k] = datas[k][:cut] + struct.pack(lfmt, min(len(last) + 7, (1 << (8 * length_size)) - 1)) + last
    first_ps = first_ps or []
    priv = avcc([n for n in first_ps if n[0] & 31 == 7], [n for n in first_ps if n[0] & 31 == 8], length_size)

    vnum = 2 if audio_first else 1
    groups = [datas[i:i + per_block] for i in range(0, len(datas), per_block)]
    if lacing == "fixed":
        padded = []
        for g in groups:
            target = max(len(d) for d in g) + length_size + 2
            padded.append([d + struct.pack(lfmt, target - len(d) - length_size) + b"\x0c" + b"\xff" * (target - len(d) - length_size - 2) + b"\x80"
                           for d in g])
        groups = padded

    def block(track: int, payload_frames: list[bytes], tc: int) -> bytes:
        bits, body = lace(payload_frames, lacing if track == vnum else "none")
        head = vint(track) + struct.pack(">h", tc)
        if block_group:
            return el(0xA0, el(0xA1, head, bytes([bits]), body), uint(0x9B, 1))
        return el(0xA3, head, bytes([0x80 | bits]), body)

    clusters = []
    for ci in range(0, len(groups), per_cluster):
        parts = [uint(0xE7, ci * 40)]
        for j, g in enumerate(groups[ci:ci + per_cluster]):
            if audio_first:
                parts.append(el(0xA3, vint(1), struct.pack(">h", j), b"\x80", bytes(rng.randrange(256) for _ in range(90))))
            parts.append(block(vnum, g, j))
        body = b"".join(parts)
        clusters.append(b"\x1f\x43\xb6\x75" + (b"\xff" if cluster_unknown else vint(len(body))) + body)

    entries = []
    if audio_first:
        entries.append(el(0xAE, uint(0xD7, 1), uint(0x73C5, 11), uint(0x83, 2), el(0x86, b"A_AAC"),
                          el(0xE1, el(0xB5, struct.pack(">f", 48000.0)), uint(0x9F, 2))))
    if video_track:
        v = [uint(0xD7, vnum), uint(0x73C5, 12), uint(0x83, 1), el(0x86, codec_id)]
        if codec_private:
            v.append(el(0x63A2, priv))
        if content_encodings:
            v.append(el(0x6D80, el(0x6240, uint(0x5031, 0), el(0x5034, uint(0x4254, 3)))))
        v.append(el(0xE0, uint(0xB0, 16), uint(0xBA, 16)))
        entries.append(el(0xAE, *v))
    tracks = el(0x1654AE6B, *entries)
    info = el(0x1549A966, uint(0x2AD7B1, 1000000), el(0x4D80, b"mkv_mux"), el(0x5741, b"mkv_mux"))
    seg = []
    if seek_cues_void:
        seg.append(el(0x114D9B74, el(0x4DBB, el(0x53AB, b"\x15\x49\xa9\x66"), uint(0x53AC, 0))))
        seg.append(el(0xEC, bytes(23)))
    seg += [info, tracks] + clusters
    if seek_cues_void:
        seg.append(el(0x1C53BB6B, el(0xBB, uint(0xB3, 0), el(0xB7, uint(0xF7, vnum), uint(0xF1, 0)))))
    body = b"".join(seg)
    segment = b"\x18\x53\x80\x67" + (UNKNOWN8 if segment_unknown else vint(len(body), 8)) + body
    header = el(0x1A45DFA3, uint(0x4286, 1), uint(0x42F7, 1), uint(0x42F2, 4), uint(0x42F3, 8), el(0x4282, doctype),
                uint(0x4287, 4), uint(0x4285, 2))
    return header + segment


def es_twin(stream: bytes) -> bytes:
    """The Annex-B stream as the Matroska front end sizes it (see mp4_mux.es_twin): a frame holding one IDR NAL unit
    behind a 4-byte length field is as large as that picture's Annex-B distance."""
    assert stream.endswith(bytes(64))
    return stream[:-60]
