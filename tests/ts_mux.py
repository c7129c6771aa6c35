"""Test infrastructure: a small MPEG-2 transport stream writer (ISO/IEC 13818-1) that carries an Annex-B stream as the
PES payloads of one H.264 PID, with knobs for the variants and the damage the TS front end has to handle.

The PES payloads of the video PID, concatenated, are exactly the Annex-B stream given to mux(): that stream is the
twin mvf_open_ts() must agree with.  mux() also reports which bytes of it each video packet carried, so a test can
work out which NAL units a damaged packet touches."""
from __future__ import annotations

import random
import struct
from dataclasses import dataclass

from helpers import split_nals

VIDEO_PID, AUDIO_PID, NULL_PID = 0x100, 0x101, 0x1FFF


def crc32_mpeg(data: bytes) -> int:
    c = 0xFFFFFFFF
    for b in data:
        c ^= b << 24
        for _ in range(8):
            c = ((c << 1) ^ 0x04C11DB7) & 0xFFFFFFFF if c & 0x80000000 else (c << 1) & 0xFFFFFFFF
    return c


def section(table_id: int, ext: int, body: bytes, version: int = 0) -> bytes:
    """A long-form PSI section with its CRC_32."""
    head = struct.pack(">BHHBBB", table_id, 0xB000 | (len(body) + 9), ext, 0xC1 | version << 1, 0, 0)
    data = head + body
    return data + struct.pack(">I", crc32_mpeg(data))


def pat(programs: list[tuple[int, int]]) -> bytes:
    """programs: (program_number, PMT PID); program 0 is the network PID."""
    return section(0x00, 1, b"".join(struct.pack(">HH", n, 0xE000 | pid) for n, pid in programs))


def pmt(program: int, streams: list[tuple[int, int]], program_info: bytes = b"") -> bytes:
    """streams: (stream_type, elementary PID)."""
    body = struct.pack(">HH", 0xE000 | (streams[0][1] if streams else 0x1FFF), 0xF000 | len(program_info)) + program_info
    body += b"".join(struct.pack(">BHH", st, 0xE000 | pid, 0xF000) for st, pid in streams)
    return section(0x02, program, body)


@dataclass
class Packet:
    pid: int
    payload: bytes = b""
    pusi: bool = False
    es: tuple[int, int] | None = None   # video: the range of the Annex-B stream this packet carries
    tei: bool = False
    scrambled: int = 0
    cc: int = 0


def packetize(pid: int, data: bytes, pusi_first: bool = True, es_base: int | None = None, es_skip: int = 0,
              stuff_every: int = 0, rng: random.Random | None = None) -> list[Packet]:
    """One PES packet or PSI run cut into packets; the last one is filled up with adaptation-field stuffing.
    stuff_every k > 0: every k-th packet also carries a shorter payload behind a stuffed adaptation field."""
    out, i, k = [], 0, 0
    while i < len(data) or not out:
        room = 184
        if stuff_every and rng is not None and i and k % stuff_every == stuff_every - 1:     # never inside a PES header
            room = rng.randrange(1, 150)
        n = min(room, len(data) - i)
        es = None
        if es_base is not None:
            lo, hi = max(i, es_skip), max(i + n, es_skip)
            es = (es_base + lo - es_skip, es_base + hi - es_skip)
        out.append(Packet(pid, data[i:i + n], pusi_first and i == 0, es=es))
        i += n
        k += 1
    return out


def psi_packets(pid: int, sections: list[bytes]) -> list[Packet]:
    """Sections written back to back on one PID: a packet in which a section starts has payload_unit_start_indicator
    and a pointer_field to the first such section (the tail of the one before may come first); stuffing 0xFF at the
    end."""
    stream = b"".join(sections)
    starts = []
    o = 0
    for s in sections:
        starts.append(o)
        o += len(s)
    out, i = [], 0
    while i < len(stream):
        first = next((s for s in starts if i <= s < i + 183), None)
        if first is not None:
            ptr = first - i
            body = bytes([ptr]) + stream[i:i + 183]
            i += 183
        else:
            body = stream[i:i + 184]
            i += 184
        out.append(Packet(pid, body + b"\xff" * (184 - len(body)), first is not None))
    return out


def access_units(es: bytes) -> list[int]:
    """Offsets at which access units start: 0, and the start code of every NAL unit that follows a slice."""
    offs, pos, prev_slice = [0], 0, False
    for nal in split_nals(es):
        if pos and prev_slice:
            offs.append(pos)
        prev_slice = nal[4] & 31 in (1, 5)
        pos += len(nal)
    return offs


def with_aud_sei(es: bytes, seed: int = 1) -> bytes:
    """The stream with an access unit delimiter and an SEI NAL unit in front of every access unit."""
    rng = random.Random(seed)
    au, out, pos = set(access_units(es)), b"", 0
    nals = split_nals(es)
    for nal in nals:
        if pos in au:
            out += b"\x00\x00\x00\x01\x09\xf0"
            out += b"\x00\x00\x00\x01\x06\x05\x10" + bytes(rng.randrange(1, 256) for _ in range(16)) + b"\x80"
        out += nal
        pos += len(nal)
    return out + es[pos:]


def mux(es: bytes, *, packet_size: int = 188, psi_every: int = 0, programs: str = "video", psi_span: bool = False,
        audio: bool = False, bounded: bool = True, pes_per_au: int = 1, stuffing: int = 0, null_packets: bool = False,
        drop: tuple[int, ...] = (), tei: tuple[int, ...] = (), dup: tuple[int, ...] = (), cut: tuple[int, ...] = (),
        scrambled: bool = False, video_type: int = 0x1B, seed: int = 1, info: dict | None = None) -> bytes:
    """Transport stream carrying the Annex-B stream `es` on PID 0x100 (stream_type `video_type`).

    packet_size   188, 192 (M2TS: 4-byte TP_extra_header in front) or 204 (16 parity bytes behind)
    psi_every     k > 0: PAT and PMT again every k packets (else once, at the start)
    programs      "video": one program; "audio_first": program 1 holds only audio, program 2 the video;
                  "two_video": program 1 video, program 2 an HEVC stream (stream_type 0x24) on another PID;
                  "audio_only": no video at all (the video PID still carries the stream)
    psi_span      a PMT long enough (program_info descriptors) to span packets, written twice back to back so
                  that the second copy starts behind a pointer_field
    audio         audio PES packets (PID 0x101) interleaved with the video packets
    bounded       PES_packet_length set (where it fits 16 bits); else 0, unbounded
    pes_per_au    each access unit split over this many PES packets, at arbitrary bytes
    stuffing      k > 0: every k-th video packet carries a short payload behind adaptation-field stuffing
    null_packets  null packets (PID 0x1FFF) in between
    drop / tei / dup / cut
                  indices among the video packets: dropped (a continuity gap), sent with transport_error_indicator,
                  sent twice, or -- for cut -- the last packet of the PES holding it dropped with the continuity
                  counters renumbered, so only the PES length shows the loss
    scrambled     transport_scrambling_control 2 on the video packets
    info          if given, receives "lost": the Annex-B ranges the damage removed, in stream order
    """
    rng = random.Random(seed)
    # PES packets of the video stream
    au = access_units(es) + [len(es)]
    video: list[Packet] = []
    for a, b in zip(au, au[1:]):
        cuts = sorted({a, b} | {rng.randrange(a + 1, b) for _ in range(pes_per_au - 1) if b - a > 1})
        for c0, c1 in zip(cuts, cuts[1:]):
            payload = es[c0:c1]
            hdr_data = bytes([0x21, 0, 1, 0, 1])            # a PTS
            plen = 3 + len(hdr_data) + len(payload)
            pes = struct.pack(">3sBHBBB", b"\x00\x00\x01", 0xE0, plen if bounded and plen < 65536 else 0, 0x80, 0x80,
                              len(hdr_data)) + hdr_data + payload
            video += packetize(VIDEO_PID, pes, es_base=c0, es_skip=9 + len(hdr_data), stuff_every=stuffing, rng=rng)
    for p in video:
        p.scrambled = 2 if scrambled else 0
    # damage
    cut_set = set()
    for i in cut:
        j = i
        while j + 1 < len(video) and not video[j + 1].pusi:
            j += 1
        assert bounded and not video[j].pusi, "cut needs a bounded PES packet of two or more packets"
        cut_set.add(j)
    lost = [video[i].es for i in sorted(set(drop) | cut_set | set(tei))]
    if info is not None:
        info["lost"] = sorted(lost)
    for i in tei:
        video[i].tei = True
    seq = []
    for i, p in enumerate(video):
        if i in drop or i in cut_set:
            seq.append(("gap" if i in drop else "cut", p))
            continue
        seq.append(("", p))
        if i in dup:
            seq.append(("dup", p))
    cc, vid_out = 0, []
    for kind, p in seq:
        if kind == "dup":
            vid_out.append(Packet(**{**p.__dict__}))
            continue
        if kind == "gap":
            cc = (cc + 1) & 15
            continue
        if kind == "cut":
            continue
        p.cc = cc
        cc = (cc + 1) & 15
        vid_out.append(p)

    # PSI
    if programs == "video":
        prog_list, pmts = [(1, 0x1000)], [(0x1000, pmt(1, [(video_type, VIDEO_PID)] + ([(0x0F, AUDIO_PID)] if audio else [])))]
    elif programs == "audio_first":
        prog_list = [(0, 0x0010), (1, 0x1000), (2, 0x1001)]
        pmts = [(0x1000, pmt(1, [(0x0F, AUDIO_PID)])), (0x1001, pmt(2, [(video_type, VIDEO_PID)]))]
    elif programs == "two_video":
        prog_list = [(1, 0x1000), (2, 0x1001)]
        pmts = [(0x1000, pmt(1, [(video_type, VIDEO_PID), (0x0F, AUDIO_PID)])), (0x1001, pmt(2, [(0x24, 0x200)]))]
    elif programs == "audio_only":
        prog_list, pmts = [(1, 0x1000)], [(0x1000, pmt(1, [(0x0F, AUDIO_PID)]))]
    else:
        raise ValueError(programs)
    if psi_span:
        descriptors = b"".join(bytes([0x80 + k % 16, 60]) + bytes(rng.randrange(256) for _ in range(60)) for k in range(4))
        pmts = [(pid, pmt(int.from_bytes(s[3:5], "big"), streams_of(s), descriptors)) for pid, s in pmts]

    def psi() -> list[Packet]:
        out = psi_packets(0, [pat(prog_list)])
        for pid, s in pmts:
            out += psi_packets(pid, [s, s] if psi_span else [s])
        return out

    # interleave: PSI first, then the video packets with audio / null packets / PSI repetitions in between
    seq2 = psi()
    n_since = len(seq2)
    for i, p in enumerate(vid_out):
        seq2.append(p)
        n_since += 1
        if audio and i % 5 == 2:
            apes = struct.pack(">3sBHBBB", b"\x00\x00\x01", 0xC0, 3 + 150, 0x80, 0, 0) + bytes(rng.randrange(256) for _ in range(150))
            seq2 += packetize(AUDIO_PID, apes)
        if null_packets and i % 4 == 1:
            seq2.append(Packet(NULL_PID, bytes(rng.randrange(256) for _ in range(184))))
        if psi_every and n_since >= psi_every:
            seq2 += psi()
            n_since = 0

    ccs: dict[int, int] = {}
    out = bytearray()
    for p in seq2:
        if p.pid != VIDEO_PID:
            p.cc = ccs.get(p.pid, 0)
            ccs[p.pid] = (p.cc + 1) & 15
        out += encode(p, packet_size, rng)
    return bytes(out)


def streams_of(pmt_section: bytes) -> list[tuple[int, int]]:
    pil = int.from_bytes(pmt_section[10:12], "big") & 0xFFF
    p, end, out = 12 + pil, len(pmt_section) - 4, []
    while p + 5 <= end:
        out.append((pmt_section[p], int.from_bytes(pmt_section[p + 1:p + 3], "big") & 0x1FFF))
        p += 5 + (int.from_bytes(pmt_section[p + 3:p + 5], "big") & 0xFFF)
    return out


def encode(p: Packet, packet_size: int, rng: random.Random) -> bytes:
    n = len(p.payload)
    assert n <= 184
    if n < 184:
        af_len = 183 - n
        af = b"" if af_len == 0 else bytes([0x00]) + b"\xff" * (af_len - 1)
        body = bytes([af_len]) + af + p.payload
        afc = 3 if n else 2
    else:
        body, afc = p.payload, 1
    head = struct.pack(">BHB", 0x47, (0x8000 if p.tei else 0) | (0x4000 if p.pusi else 0) | p.pid,
                       p.scrambled << 6 | afc << 4 | p.cc)
    pkt = head + body
    if p.tei:
        pkt = pkt[:4] + bytes(b ^ 0x5A for b in pkt[4:])
    assert len(pkt) == 188
    if packet_size == 192:
        return struct.pack(">I", rng.randrange(1 << 30)) + pkt
    if packet_size == 204:
        return pkt + bytes(rng.randrange(256) for _ in range(16))
    return pkt


def annexb_nals(es: bytes) -> list[tuple[int, int]]:
    """(first zero of the 3-byte start code, NAL header offset) of every NAL unit, found as mvf_open_annexb finds
    them."""
    out, q = [], 2
    while True:
        q = es.find(b"\x01", q)
        if q < 0 or q >= len(es) - 1:
            return out
        if es[q - 1] == 0 and es[q - 2] == 0:
            out.append((q - 2, q + 1))
        q += 1


def surviving(es: bytes, lost: list[tuple[int, int]]) -> bytes:
    """The Annex-B stream without the NAL units a damaged stretch [a, b) touches, as mvf_open_ts drops them: the NAL
    unit in progress when the bytes went missing, and every NAL unit whose start code is not wholly behind them."""
    nals = annexb_nals(es)
    dropped = set()
    for a, b in lost:
        cur = [i for i, (_, h) in enumerate(nals) if h < a]
        if cur:
            dropped.add(cur[-1])
        dropped |= {i for i, (z, h) in enumerate(nals) if h >= a and z < b}
    bounds = [z for z, _ in nals] + [len(es)]
    return b"".join(es[bounds[i]:bounds[i + 1]] for i in range(len(nals)) if i not in dropped)
