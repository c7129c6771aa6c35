"""Build every native library of this repository in-tree.

    python -m minivideo_b200.build [--force]

libmvgpu.so   : CUDA kernels + C ABI (nvcc, sm_100a only)      -> minivideo_b200/
libmvfront.so : host front end (Annex-B/CAVLC parser -> SoA)   -> minivideo_b200/
libmvsynth.so : synthetic intra-only stream generator           -> minivideo_b200/
oracle/librecon_oracle.so, oracle/_ref/* : test infrastructure (see oracle/Makefile)

The .so files are git-ignored but travel to the GPU box with the snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "minivideo_b200"
CSRC = PKG / "csrc"
INC = ROOT / "include"
REFERENCE = Path(os.environ.get("MVG_REFERENCE", "/root/reference"))

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--shared", "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _reference_has(rel: str) -> bool:
    """Whether the reference tree holds `rel`; a tree this user may not read counts as absent."""
    p = REFERENCE / rel
    try:
        return p.exists() and os.access(p, os.R_OK)
    except OSError:
        return False


def _stale(target: Path, sources: list[Path]) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(s.exists() and s.stat().st_mtime > t for s in sources)


def _run(cmd: list[str], log: Path | None = None) -> None:
    res = subprocess.run(cmd, capture_output=True, text=True)
    if log is not None:
        log.write_text(res.stdout + res.stderr)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("build failed: " + " ".join(cmd))


def build_synth(force: bool = False) -> Path:
    out = PKG / "libmvsynth.so"
    src = [CSRC / "h264_synth.c", INC / "mvsynth.h", CSRC / "h264_cavlc_tables.h"]
    if force or _stale(out, src):
        _run(["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-Wextra", f"-I{INC}", f"-I{CSRC}",
              "-o", str(out), str(src[0]), "-lm"])
    return out


def build_front(force: bool = False) -> Path | None:
    out = PKG / "libmvfront.so"
    src = [CSRC / "h264_front.c", INC / "mvfront.h", INC / "mvgpu.h", CSRC / "h264_cavlc_tables.h"]
    if not src[0].exists():
        return None
    if force or _stale(out, src):
        _run(["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-Wextra", f"-I{INC}", f"-I{CSRC}",
              "-o", str(out), str(src[0]), "-lm", "-lpthread"])
    return out


def build_gpu(force: bool = False) -> Path:
    out = PKG / "libmvgpu.so"
    cu = sorted(CSRC.glob("*.cu"))
    deps = cu + sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.h")) + [INC / "mvgpu.h"]
    if force or _stale(out, deps):
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        extra = ["-DMVG_K2_PROFILE"] if os.environ.get("MVG_K2_PROFILE") else []     # dev: in-kernel cycle accounting
        extra += ["-D" + d for d in os.environ.get("MVG_EXTRA_DEFINES", "").split()]     # dev: experiments
        _run([nvcc, *NVCC_FLAGS, *extra, f"-I{INC}", f"-I{CSRC}", "-o", str(out), *map(str, cu)],
             log=PKG / "libmvgpu.build.log")
    return out


def build_thumbnailer(force: bool = False) -> Path:
    """mv_thumbnailer: the CLI over libmvfront.so + libmvgpu.so (mini_thumbnailer-compatible arguments), and
    libminivideo_b200.so: the reference's public entry points (minivideo.h) backed by the same core."""
    out = PKG / "mv_thumbnailer"
    core = [CSRC / "mv_thumbcore.c", CSRC / "mv_png.c", CSRC / "mv_thumbcore.h", CSRC / "mv_png.h", INC / "mvfront.h",
            INC / "mvgpu.h", PKG / "libmvfront.so", PKG / "libmvgpu.so"]
    libs = [f"-L{PKG}", "-Wl,-rpath,$ORIGIN", "-lmvfront", "-lmvgpu", "-lstdc++", "-lm", "-lpthread", "-ldl", "-lrt"]
    if force or _stale(out, core + [CSRC / "mv_thumbnailer.c"]):
        _run(["gcc", "-O2", "-Wall", "-Wextra", f"-I{INC}", f"-I{CSRC}", "-o", str(out), str(CSRC / "mv_thumbnailer.c"),
              str(core[0]), str(core[1]), *libs])
    shim = PKG / "libminivideo_b200.so"
    if force or _stale(shim, core + [CSRC / "minivideo_shim.c"]):
        _run(["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-Wextra", f"-I{INC}", f"-I{CSRC}", "-o", str(shim),
              str(CSRC / "minivideo_shim.c"), str(core[0]), str(core[1]), *libs])
    return out


def build_oracle(force: bool = False) -> Path:
    out = ROOT / "oracle" / "librecon_oracle.so"
    src = [ROOT / "oracle" / "recon_oracle.c", ROOT / "oracle" / "recon_oracle.h", ROOT / "oracle" / "Makefile"]
    if force or _stale(out, src):
        _run(["make", "-C", str(ROOT / "oracle"), "oracle"] + (["-B"] if force else []))
    return out


def build_reference(force: bool = False) -> Path | None:
    """Compile the unmodified reference (only where its tree is mounted)."""
    out = ROOT / "oracle" / "_ref" / "ref_decode"
    if not _reference_has("minivideo/src"):
        return out if out.exists() else None
    if force or _stale(out, [ROOT / "oracle" / "ref_driver.c", ROOT / "oracle" / "ref_png.c", ROOT / "oracle" / "Makefile"]):
        _run(["make", "-C", str(ROOT / "oracle"), "ref", f"REF={REFERENCE}", "-j8"])
    return out


def build_shim_cli(force: bool = False) -> Path | None:
    """The reference's own mini_thumbnailer main.cpp linked against libminivideo_b200.so (only where the
    reference tree is mounted; the binary lives in oracle/_ref and travels to the GPU box)."""
    out = ROOT / "oracle" / "_ref" / "mini_thumbnailer_b200"
    if not _reference_has("mini_thumbnailer/src/main.cpp"):
        return out if out.exists() else None
    if force or _stale(out, [PKG / "libminivideo_b200.so", ROOT / "oracle" / "Makefile"]):
        _run(["make", "-C", str(ROOT / "oracle"), "shimcli", f"REF={REFERENCE}"])
    return out


def build_all(force: bool = False) -> dict:
    out = {
        "synth": build_synth(force),
        "front": build_front(force),
        "oracle": build_oracle(force),
        "reference": build_reference(force),
        "gpu": build_gpu(force),
        "thumbnailer": build_thumbnailer(force),
    }
    out["shim_cli"] = build_shim_cli(force)
    return out


if __name__ == "__main__":
    for name, path in build_all("--force" in sys.argv).items():
        print(f"{name:10s} {path}")
