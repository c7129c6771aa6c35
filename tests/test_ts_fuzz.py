"""Robustness of the transport stream front end: damaged streams (continuity counters, transport_error_indicator,
pointer_field, section and PES header lengths, adaptation-field lengths, truncation, random bytes) under
AddressSanitizer + UBSan must end in a return code, never in a crash or an out-of-bounds access."""
import re
import shutil
import subprocess
from pathlib import Path

import pytest

from ts_mux import mux, with_aud_sei

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def fuzzer(tmp_path_factory):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    exe = tmp_path_factory.mktemp("fuzz_ts") / "fuzz_ts"
    r = subprocess.run(["gcc", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                        f"-I{ROOT / 'include'}", f"-I{ROOT / 'minivideo_b200' / 'csrc'}", "-o", str(exe),
                        str(ROOT / "tests" / "fuzz_ts.c"), str(ROOT / "minivideo_b200" / "csrc" / "h264_front.c"),
                        "-lm", "-lpthread"], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("sanitizer build not available: " + r.stderr[-300:])
    return exe


@pytest.mark.parametrize("cfg,knobs", [
    (dict(width_mbs=6, height_mbs=4, profile_idc=66, seed=41), dict(packet_size=188, psi_every=15, audio=True)),
    (dict(width_mbs=5, height_mbs=5, profile_idc=100, transform8x8=1, scaling_lists=1, seed=42),
     dict(packet_size=192, pes_per_au=3, stuffing=2, psi_span=True, psi_every=30)),
    ("multi", dict(packet_size=204, bounded=False, null_packets=True, psi_every=20)),
], ids=["baseline_188", "high_m2ts", "three_generations_204"])
def test_ts_front_end_survives_damaged_streams_under_sanitizers(fuzzer, tmp_path, cfg, knobs):
    from helpers import paramset_change_stream
    from minivideo_b200 import synth
    stream = paramset_change_stream()[0] if cfg == "multi" else with_aud_sei(synth.generate(5, **cfg)[0])
    (tmp_path / "s.ts").write_bytes(mux(stream, **knobs))
    r = subprocess.run([str(fuzzer), str(tmp_path / "s.ts"), "3000", str(knobs["packet_size"])],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-500:], r.stderr[-3000:])
    m = re.search(r"rounds=3000 opened=(\d+) parsed=(\d+) failure=(\d+) unsupported=(\d+)", r.stdout)
    assert m, r.stdout
    opened, parsed, failure, _ = map(int, m.groups())
    assert opened > 100 and parsed > 100 and failure > 100, r.stdout      # every outcome was reached
