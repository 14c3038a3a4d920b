"""Checkers for the power-spectrum mode (fx_engine.h FX_SPECTRUM_POWER), for tests/ and tools/parity_report.py only.

The mode is defined by one substitution: each forward transform hands its consumers (|X[k]|, 0) in place of
(Re X[k], Im X[k]), |X| = (float) sqrt ((double) Re^2 + (double) Im^2).  The checkers under oracle/ stay as they are; this
module compiles each of them once more with exactly that substitution applied to its single forward-transform entry point
of the real-time path, into a per-user cache directory outside the tree:
  port       oracle/fx_oracle.c, the substitution at the end of frequency_data (FFTAnalyser::getFrequencyData)
  reference  oracle/ref_driver.cpp over oracle/juce_shim/JuceHeader.h with the substitution at the end of the shim's
             FFT::performRealOnlyForwardTransform for forward plans -- the reference's own classes, unmodified, then
             receive |X|.  Only where the reference sources exist (REF_SRC, as oracle/Makefile); otherwise None.
The legacy entry point of these builds is not used (the legacy analyser already uses true magnitudes).
Both builds export the fxo_* API of oracle/fx_oracle_api.h, so tests/oracle_util.py's Oracle drives them as it drives the
parity-mode checkers."""
from __future__ import annotations

import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_util as ou

REF_SRC = os.environ.get("REF_SRC", "/root/reference/Source")

_PORT_ANCHOR = """    fft_real_forward (&t->fwd, buf2n, t->scratch);
}
"""
_PORT_SUBST = """    fft_real_forward (&t->fwd, buf2n, t->scratch);
    {
        int k;
        for (k = 0; k < t->n; ++k) {
            const double re = buf2n[2 * k], im = buf2n[2 * k + 1];
            buf2n[2 * k] = (float) sqrt (re * re + im * im);
            buf2n[2 * k + 1] = 0.0f;
        }
    }
}
"""
_SHIM_ANCHOR = """        perform (scratch.data(), reinterpret_cast<Complex*> (d));
    }
"""
_SHIM_SUBST = """        perform (scratch.data(), reinterpret_cast<Complex*> (d));
        if (! inverse)
            for (int i = 0; i < 2 * size; i += 2)
            {
                d[i] = (float) sqrt ((double) d[i] * d[i] + (double) d[i + 1] * d[i + 1]);
                d[i + 1] = 0.0f;
            }
    }
"""


def _substituted(path: str, anchor: str, subst: str) -> str:
    src = open(path).read()
    if src.count(anchor) != 1:
        raise RuntimeError(f"{path}: the forward-transform entry point this module substitutes was not found exactly once")
    return src.replace(anchor, subst)


def _cache_dir(tag: str) -> str:
    d = os.path.join(os.environ.get("FXB200_CACHE") or tempfile.gettempdir(), f"fxb200-power-oracle-{os.getuid()}", tag)
    os.makedirs(d, exist_ok=True)
    return d


def _build(tag: str, sources: dict, cmd) -> str:
    """write `sources` (relative name -> text) into a cache directory keyed by their hash and compile once"""
    h = hashlib.sha256("".join(k + v for k, v in sorted(sources.items())).encode()).hexdigest()[:16]
    d = _cache_dir(f"{tag}-{h}")
    so = os.path.join(d, "lib.so")
    if not os.path.exists(so):
        for name, text in sources.items():
            os.makedirs(os.path.dirname(os.path.join(d, name)), exist_ok=True)
            with open(os.path.join(d, name), "w") as f:
                f.write(text)
        tmp = so + f".{os.getpid()}"
        subprocess.run(cmd(d, tmp), check=True, cwd=d, stdout=subprocess.DEVNULL)
        os.replace(tmp, so)
    return so


_port = None


def port() -> ou.Oracle:
    """the C port with the substitution (same compiler flags as oracle/Makefile)"""
    global _port
    if _port is None:
        src = _substituted(os.path.join(ou.ORACLE_DIR, "fx_oracle.c"), _PORT_ANCHOR, _PORT_SUBST)
        so = _build("port", {"fx_oracle_power.c": src},
                    lambda d, out: ["gcc", "-O2", "-std=c99", "-fPIC", "-shared", "-Wall", "-Wextra", "-I" + ou.ORACLE_DIR, "-o", out,
                                    "fx_oracle_power.c", "-lm", "-lpthread"])
        _port = ou.Oracle(so)
    return _port


def reference() -> ou.Oracle | None:
    """the reference's own classes over the substituted shim, where the reference sources exist"""
    if not os.path.isdir(REF_SRC):
        return None
    shim = _substituted(os.path.join(ou.ORACLE_DIR, "juce_shim", "JuceHeader.h"), _SHIM_ANCHOR, _SHIM_SUBST)
    drv = open(os.path.join(ou.ORACLE_DIR, "ref_driver.cpp")).read()
    so = _build("ref", {"juce_shim/JuceHeader.h": shim, "ref_driver.cpp": drv},
                lambda d, out: ["g++", "-O2", "-std=c++14", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable", "-Wno-unused-function",
                                "-Wno-return-type", "-Wno-sign-compare", "-Wno-switch", "-I" + d, "-I" + ou.ORACLE_DIR, "-I" + REF_SRC,
                                "-o", out, "ref_driver.cpp", "-lpthread"])
    return ou.Oracle(so)


class CheckedPowerOracle:
    """tests/oracle_util.py::CheckedOracle for the power mode: values from the reference's classes where they can be built,
    decision margins from the port (which must agree with them on every value)."""

    def __init__(self):
        self.ref = reference()
        self.port = port()
        self.kind = ("reference values + port margins" if self.ref is not None else "port (reference sources absent)") + ", power spectrum"

    def analyse(self, audio: np.ndarray, threads: int = 0, **cfg):
        p = self.port.analyse(audio, threads=threads, **cfg)
        if self.ref is None:
            return p
        r = self.ref.analyse(audio, threads=threads, **cfg)
        assert np.array_equal(r["raw"], p["raw"], equal_nan=True), "power-mode port and reference build disagree"
        assert np.array_equal(r["diag"][..., ou.D["lag"]], p["diag"][..., ou.D["lag"]])
        return {"raw": r["raw"], "smooth": r["smooth"], "diag": p["diag"], "frames": r["frames"]}
