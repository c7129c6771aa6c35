"""Robustness of the MP4 front end: damaged MP4 files (box sizes, entry counts, chunk offsets, NAL length fields,
truncation at box boundaries, random bytes in moov) under AddressSanitizer + UBSan must end in a return code, never
in a crash or an out-of-bounds access."""
import re
import shutil
import subprocess
from pathlib import Path

import pytest

from mp4_mux import mux

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def fuzzer(tmp_path_factory):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    exe = tmp_path_factory.mktemp("fuzz_mp4") / "fuzz_mp4"
    r = subprocess.run(["gcc", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                        f"-I{ROOT / 'include'}", f"-I{ROOT / 'minivideo_b200' / 'csrc'}", "-o", str(exe),
                        str(ROOT / "tests" / "fuzz_mp4.c"), str(ROOT / "minivideo_b200" / "csrc" / "h264_front.c"),
                        "-lm", "-lpthread"], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("sanitizer build not available: " + r.stderr[-300:])
    return exe


@pytest.mark.parametrize("cfg,knobs", [
    (dict(width_mbs=6, height_mbs=4, profile_idc=66, seed=41), dict(length_size=4, chunk_pattern=(2, 1, 3))),
    (dict(width_mbs=5, height_mbs=5, profile_idc=100, transform8x8=1, scaling_lists=1, seed=42),
     dict(length_size=2, co64=True, moov_first=False, junk_samples=1, chunk_pattern=(3,))),
    ("multi", dict(length_size=4, largesize_mdat=True, chunk_pattern=(1, 2))),
], ids=["baseline_stco", "high_co64_moov_last", "three_descriptions"])
def test_mp4_front_end_survives_damaged_files_under_sanitizers(fuzzer, tmp_path, cfg, knobs):
    from helpers import paramset_change_stream
    from minivideo_b200 import synth
    stream = paramset_change_stream()[0] if cfg == "multi" else synth.generate(5, **cfg)[0]
    (tmp_path / "s.mp4").write_bytes(mux(stream, **knobs))
    r = subprocess.run([str(fuzzer), str(tmp_path / "s.mp4"), "3000", str(knobs["length_size"])],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-500:], r.stderr[-3000:])
    m = re.search(r"rounds=3000 opened=(\d+) parsed=(\d+) failure=(\d+) unsupported=(\d+)", r.stdout)
    assert m, r.stdout
    opened, parsed, failure, _ = map(int, m.groups())
    assert opened > 100 and parsed > 100 and failure > 100, r.stdout      # every outcome was reached
