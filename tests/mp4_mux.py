"""Test infrastructure: a small ISO BMFF (MP4) writer that wraps the Annex-B streams of synth.generate() in an MP4
file, with knobs for the container variants the MP4 front end has to read.

Every IDR NAL unit becomes one sync sample.  The parameter sets in front of it either go into the avcC box of a
sample description -- a new description whenever they change, so a stream whose parameter sets change gets several
descriptions, selected through stsc -- or (avc3) stay in band at the start of the sample."""
from __future__ import annotations

import random
import struct

from helpers import split_nals


def box(kind: bytes, *parts: bytes) -> bytes:
    body = b"".join(parts)
    return struct.pack(">I4s", 8 + len(body), kind) + body


def full_box(kind: bytes, version: int, flags: int, *parts: bytes) -> bytes:
    return box(kind, struct.pack(">I", version << 24 | flags), *parts)


def nal_units(stream: bytes) -> list[bytes]:
    """The NAL units of an Annex-B stream from synth.generate(), without start codes."""
    return [n[4:] for n in split_nals(stream)]


def avcc(sps: list[bytes], pps: list[bytes], length_size: int, high_tail: bool) -> bytes:
    """AVCDecoderConfigurationRecord (ISO/IEC 14496-15 5.3.3.1)."""
    first = sps[0] if sps else bytes(4)
    out = bytes([1, first[1] if sps else 66, first[2] if sps else 0, first[3] if sps else 30,
                 0xFC | (length_size - 1), 0xE0 | len(sps)])
    out += b"".join(struct.pack(">H", len(s)) + s for s in sps)
    out += bytes([len(pps)]) + b"".join(struct.pack(">H", len(p)) + p for p in pps)
    if high_tail:       # chroma_format 4:2:0, 8-bit luma and chroma, no SPS extensions
        out += bytes([0xFC | 1, 0xF8, 0xF8, 0])
    return box(b"avcC", out)


def visual_entry(kind: bytes, width: int, height: int, *children: bytes) -> bytes:
    return box(kind, bytes(6), struct.pack(">H", 1), bytes(16), struct.pack(">HH", width, height),
               struct.pack(">II", 0x480000, 0x480000), bytes(4), struct.pack(">H", 1), bytes(32),
               struct.pack(">Hh", 0x18, -1), *children)


def sample_table(entries: list[bytes], sizes: list[int], chunks: list[tuple[int, int, int]], sync: list[int] | None,
                 co64: bool, constant_size: bool) -> bytes:
    """stbl; chunks: (file offset, samples, 1-based description index) in order."""
    runs = []
    for i, (_, n, d) in enumerate(chunks):
        if not runs or runs[-1][1:] != (n, d):
            runs.append((i + 1, n, d))
    parts = [full_box(b"stsd", 0, 0, struct.pack(">I", len(entries)), *entries),
             full_box(b"stts", 0, 0, struct.pack(">III", 1, len(sizes), 1))]
    if sync is not None:
        parts.append(full_box(b"stss", 0, 0, struct.pack(">I", len(sync)), *(struct.pack(">I", s) for s in sync)))
    parts.append(full_box(b"stsc", 0, 0, struct.pack(">I", len(runs)), *(struct.pack(">III", *r) for r in runs)))
    if constant_size:
        assert len(set(sizes)) == 1
        parts.append(full_box(b"stsz", 0, 0, struct.pack(">II", sizes[0], len(sizes))))
    else:
        parts.append(full_box(b"stsz", 0, 0, struct.pack(">II", 0, len(sizes)), *(struct.pack(">I", s) for s in sizes)))
    if co64:
        parts.append(full_box(b"co64", 0, 0, struct.pack(">I", len(chunks)), *(struct.pack(">Q", c[0]) for c in chunks)))
    else:
        parts.append(full_box(b"stco", 0, 0, struct.pack(">I", len(chunks)), *(struct.pack(">I", c[0]) for c in chunks)))
    return box(b"stbl", *parts)


def track(track_id: int, handler: bytes, media_header: bytes, stbl: bytes, width: int = 0, height: int = 0) -> bytes:
    tkhd = full_box(b"tkhd", 0, 3, struct.pack(">IIIII", 0, 0, track_id, 0, 0), bytes(8), struct.pack(">hhhH", 0, 0, 0, 0),
                    struct.pack(">9I", 0x10000, 0, 0, 0, 0x10000, 0, 0, 0, 0x40000000), struct.pack(">II", width << 16, height << 16))
    mdhd = full_box(b"mdhd", 0, 0, struct.pack(">IIIIHH", 0, 0, 25, 0, 0x55C4, 0))
    hdlr = full_box(b"hdlr", 0, 0, struct.pack(">I4s", 0, handler), bytes(12), b"handler\x00")
    dinf = box(b"dinf", full_box(b"dref", 0, 0, struct.pack(">I", 1), full_box(b"url ", 0, 1)))
    return box(b"trak", tkhd, box(b"mdia", mdhd, hdlr, box(b"minf", media_header, dinf, stbl)))


def mux(stream: bytes, *, length_size: int = 4, co64: bool = False, chunk_pattern=(1,), moov_first: bool = True,
        largesize_mdat: bool = False, audio_first: bool = False, junk_samples: int = 0, aud_sei: bool = False,
        avc3: bool = False, high_tail: bool = True, constant_size: bool = False, chunk_gaps: bool = False,
        damaged_sample: tuple[int, list[bytes]] | None = None, brand: bytes | None = b"isom", seed: int = 1) -> bytes:
    """MP4 file holding the NAL units of the Annex-B `stream`.

    length_size       1, 2 or 4 byte NAL length fields (lengthSizeMinusOne + 1)
    co64              64-bit chunk offsets instead of stco
    chunk_pattern     samples per chunk, cycled (a chunk also ends where the sample description changes)
    moov_first        moov before mdat (else after it)
    largesize_mdat    mdat with a 64-bit largesize header
    audio_first       an audio track (mp4a) in front of the video track, its samples in mdat too
    junk_samples      non-sync samples after every IDR sample, each with well-formed type-1 NAL units of random bytes
    aud_sei           an access unit delimiter and an SEI NAL unit in front of the IDR NAL inside each sample
    avc3              parameter sets in band (sample entry avc3, empty avcC lists) instead of in avcC
    high_tail         the High-profile fields after the PPS list of avcC
    constant_size     filler NAL units (type 12) bring every sample to one size; stsz then holds a single size
    chunk_gaps        random bytes between the chunks in mdat
    damaged_sample    (k, NAL units): after the k-th video sample, one more sample holding these NAL units whose
                      last length field runs past the end of the sample
    brand             major brand of the ftyp box; None: no ftyp box
    """
    rng = random.Random(seed)
    lfmt = {1: ">B", 2: ">H", 4: ">I"}[length_size]

    def prefixed(nal: bytes) -> bytes:
        assert len(nal) < 1 << (8 * length_size), "NAL unit too long for the length field"
        return struct.pack(lfmt, len(nal)) + nal

    # samples: [NAL units], sync, description index (1-based); descriptions: (sps list, pps list)
    samples, descs, pending = [], [], []
    width = height = 0          # informative only in a visual sample entry; the decoder takes the SPS
    for nal in nal_units(stream):
        t = nal[0] & 31
        if t in (7, 8):
            pending.append(nal)
            continue
        assert t == 5, f"unexpected NAL type {t}"
        body = []
        if aud_sei:
            body += [b"\x09\xf0", b"\x06\x05\x10" + bytes(rng.randrange(256) for _ in range(16)) + b"\x80"]
        if avc3:
            body += pending
            if not descs:
                descs.append(([], []))
        elif pending:
            descs.append(([n for n in pending if n[0] & 31 == 7], [n for n in pending if n[0] & 31 == 8]))
        pending = []
        samples.append((body + [nal], True, len(descs)))
        for _ in range(junk_samples):
            junk = [bytes([0x41]) + bytes(rng.randrange(1, 256) for _ in range(rng.randrange(4, 120)))
                    for _ in range(rng.randrange(1, 4))]
            samples.append((junk, False, len(descs)))
    if damaged_sample is not None:
        k, nals = damaged_sample
        samples.insert(k + 1, (nals, False, samples[k][2]))
    datas = [b"".join(prefixed(n) for n in nals) for nals, _, _ in samples]
    if damaged_sample is not None:
        k = damaged_sample[0] + 1
        last = damaged_sample[1][-1]
        cut = len(datas[k]) - len(last) - length_size
        datas[k] = datas[k][:cut] + struct.pack(lfmt, min(len(last) + 7, (1 << (8 * length_size)) - 1)) + last
    if constant_size:
        target = max(len(d) for d in datas) + length_size + 2
        datas = [d + prefixed(b"\x0c" + b"\xff" * (target - len(d) - length_size - 2) + b"\x80") for d in datas]

    # mdat payload: audio chunk, then the video chunks in order (with optional gaps)
    audio = bytes(rng.randrange(256) for _ in range(300)) if audio_first else b""
    payload, rel_chunks = bytearray(audio), []
    i, p = 0, 0
    while i < len(samples):
        n = chunk_pattern[p % len(chunk_pattern)]
        p += 1
        d = samples[i][2]
        group = [j for j in range(i, min(i + n, len(samples))) if samples[j][2] == d]
        if chunk_gaps:
            payload += bytes(rng.randrange(256) for _ in range(rng.randrange(1, 9)))
        rel_chunks.append((len(payload), len(group), d))
        for j in group:
            payload += datas[j]
        i += len(group)

    entries = [visual_entry(b"avc3" if avc3 else b"avc1", width, height, avcc(s, q, length_size, high_tail)) for s, q in descs]
    sync = [j + 1 for j, s in enumerate(samples) if s[1]]

    def build_moov(mdat_body_start: int) -> bytes:
        chunks = [(mdat_body_start + off, n, d) for off, n, d in rel_chunks]
        video = track(2 if audio_first else 1, b"vide", full_box(b"vmhd", 0, 1, bytes(8)),
                      sample_table(entries, [len(x) for x in datas], chunks, None if len(sync) == len(samples) else sync,
                                   co64, constant_size), width, height)
        traks = [video]
        if audio_first:
            mp4a = box(b"mp4a", bytes(6), struct.pack(">H", 1), bytes(8), struct.pack(">HHHHI", 2, 16, 0, 0, 44100 << 16))
            achunks = [(mdat_body_start, 3, 1)]
            traks.insert(0, track(1, b"soun", full_box(b"smhd", 0, 0, bytes(4)),
                                  sample_table([mp4a], [100, 100, 100], achunks, None, co64, False)))
        mvhd = full_box(b"mvhd", 0, 0, struct.pack(">IIII", 0, 0, 1000, 0), struct.pack(">IH", 0x10000, 0x100), bytes(10),
                        struct.pack(">9I", 0x10000, 0, 0, 0, 0x10000, 0, 0, 0, 0x40000000), bytes(24),
                        struct.pack(">I", len(traks) + 1))
        return box(b"moov", mvhd, *traks)

    ftyp = box(b"ftyp", brand, struct.pack(">I", 512), b"isomiso2avc1mp41") if brand else b""
    mdat_hdr = 16 if largesize_mdat else 8

    def mdat() -> bytes:
        if largesize_mdat:
            return struct.pack(">I4sQ", 1, b"mdat", 16 + len(payload)) + bytes(payload)
        return box(b"mdat", bytes(payload))

    if moov_first:
        size = len(build_moov(0))
        moov = build_moov(len(ftyp) + size + mdat_hdr)
        assert len(moov) == size
        return ftyp + moov + mdat()
    return ftyp + mdat() + build_moov(len(ftyp) + mdat_hdr)


def es_twin(stream: bytes) -> bytes:
    """The Annex-B stream as the MP4 front end sizes it: synth.generate() ends a stream in 64 zero bytes, which
    mvf_select_idr() counts into the last picture; 4 of them stand in for the length field the MP4 sample of that
    picture carries instead, so that both forms give every picture the same size."""
    assert stream.endswith(bytes(64))
    return stream[:-60]
