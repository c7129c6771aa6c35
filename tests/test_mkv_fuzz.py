"""Robustness of the Matroska front end: damaged files (vint widths and sizes, element IDs, lace counts and sizes,
CodecPrivate, truncation at element boundaries, random bytes) under AddressSanitizer + UBSan must end in a return
code, never in a crash or an out-of-bounds access."""
import re
import shutil
import subprocess
from pathlib import Path

import pytest

from mkv_mux import mux

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def fuzzer(tmp_path_factory):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    exe = tmp_path_factory.mktemp("fuzz_mkv") / "fuzz_mkv"
    r = subprocess.run(["gcc", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                        f"-I{ROOT / 'include'}", f"-I{ROOT / 'minivideo_b200' / 'csrc'}", "-o", str(exe),
                        str(ROOT / "tests" / "fuzz_mkv.c"), str(ROOT / "minivideo_b200" / "csrc" / "h264_front.c"),
                        "-lm", "-lpthread"], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("sanitizer build not available: " + r.stderr[-300:])
    return exe


@pytest.mark.parametrize("cfg,knobs", [
    (dict(width_mbs=6, height_mbs=4, profile_idc=66, seed=41), dict(lacing="xiph", per_block=2, audio_first=True)),
    (dict(width_mbs=5, height_mbs=5, profile_idc=100, transform8x8=1, scaling_lists=1, seed=42),
     dict(length_size=2, lacing="ebml", per_block=3, block_group=True, seek_cues_void=True)),
    ("multi", dict(segment_unknown=True, cluster_unknown=True, lacing="fixed", per_block=2)),
], ids=["baseline_xiph", "high_ebml_groups", "three_generations_unknown_sizes"])
def test_mkv_front_end_survives_damaged_files_under_sanitizers(fuzzer, tmp_path, cfg, knobs):
    from helpers import paramset_change_stream
    from minivideo_b200 import synth
    stream = paramset_change_stream()[0] if cfg == "multi" else synth.generate(5, **cfg)[0]
    (tmp_path / "s.mkv").write_bytes(mux(stream, **knobs))
    r = subprocess.run([str(fuzzer), str(tmp_path / "s.mkv"), "3000"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-500:], r.stderr[-3000:])
    m = re.search(r"rounds=3000 opened=(\d+) parsed=(\d+) failure=(\d+) unsupported=(\d+)", r.stdout)
    assert m, r.stdout
    opened, parsed, failure, _ = map(int, m.groups())
    assert opened > 100 and parsed > 100 and failure > 100, r.stdout      # every outcome was reached
