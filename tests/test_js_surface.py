"""The JavaScript host cannot run in this image (no Node: SURVEY F1/F2), so these checks are structural: the B200
index.js exports every factory the reference's index.js exports, its contexts carry what the reference's carry, the raw
exports are synchronous, index.d.ts declares every name the reference's declares, and the N-API shim type-checks against the
Node-API signatures of the calls it makes (tests/napi_stub/node_api.h).  The behaviour of this surface is tested through its
Python twin (wat-fft_b200/contexts.py -- same design, same C ABI) in the GPU tests."""
import os
import re
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
JS = (ROOT / "wat-fft_b200" / "js" / "index.js").read_text()
DTS = (ROOT / "wat-fft_b200" / "js" / "index.d.ts").read_text()
REF = Path(os.environ["WATFFT_REFERENCE"]) if os.environ.get("WATFFT_REFERENCE") else None   # a wat-fft checkout

# the reference's public surface (index.js:28-178, index.d.ts:6-250), restated so the test also runs without a reference checkout
REF_FACTORIES = ["createFFTInstance", "createFFTf32Instance", "createRFFTInstance", "createRFFTf32Instance",
                 "createFFT", "createFFTf32", "createRFFT", "createRFFTf32"]
REF_TYPES = ["FFTExports", "FFTf32Exports", "RFFTExports", "RFFTf32Exports", "FFT", "FFTf32", "RFFT", "RFFTf32"]
REF_CONTEXT_FIELDS = ["size", "exports", "getInputBuffer", "getOutputBuffer", "forward", "inverse"]


def test_restated_surface_matches_the_reference():
    if REF is None:
        pytest.skip("reference checkout absent (set WATFFT_REFERENCE)")
    ref_js = (REF / "index.js").read_text()
    assert sorted(re.findall(r"export async function (\w+)", ref_js)) == sorted(REF_FACTORIES)
    ref_dts = (REF / "index.d.ts").read_text()
    assert sorted(re.findall(r"export interface (\w+)", ref_dts)) == sorted(REF_TYPES)
    assert sorted(re.findall(r"export function (\w+)", ref_dts)) == sorted(REF_FACTORIES)


def test_index_js_exports_every_reference_factory():
    exported = set(re.findall(r"export (?:async )?function (\w+)", JS)) | set(re.findall(r"export const (\w+)", JS))
    assert set(REF_FACTORIES) <= exported, set(REF_FACTORIES) - exported
    for name in REF_FACTORIES:                       # factories are async, as in the reference
        assert re.search(rf"export async function {name}\b", JS), name


def test_contexts_carry_the_reference_fields():
    body = JS[JS.index("function makeContext"):]
    for field in REF_CONTEXT_FIELDS:
        assert re.search(rf"\b(get )?{field}\b", body), field
    assert "get exports()" in body


def test_raw_exports_are_synchronous():
    """The reference's suites call `wasm.fft_split(n)` and read memory on the next line: no export may return a Promise."""
    inst = JS[JS.index("function makeInstanceSync"):JS.index("// Low-level instance factories")]
    assert "async" not in inst and "await" not in inst and "Promise" not in inst
    for name in ("precompute_twiddles", "fft", "ifft", "precompute_rfft_twiddles", "rfft", "irfft", "precompute_twiddles_split",
                 "precompute_rfft_twiddles_split", "fft_split", "ifft_split", "rfft_split", "irfft_split"):
        assert re.search(rf"\b{name}\(size\)", inst), name
    assert "REAL_OFFSET" in inst and "IMAG_OFFSET" in inst and "memory: { buffer }" in inst


def test_index_d_ts_declares_every_reference_name():
    for t in REF_TYPES:
        assert re.search(rf"export interface {t}\b", DTS), t
    for f in REF_FACTORIES:
        assert re.search(rf"export function {f}\(", DTS), f
    for t in ("FFT", "FFTf32", "RFFT", "RFFTf32"):
        iface = DTS[DTS.index(f"export interface {t} {{"):]
        iface = iface[:iface.index("\n}")]
        for field in REF_CONTEXT_FIELDS:
            assert re.search(rf"\b{field}\b", iface), (t, field)


def test_napi_shim_type_checks():
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-Wextra", "-Werror", "-I", str(ROOT / "tests" / "napi_stub"),
                        str(ROOT / "wat-fft_b200" / "napi" / "watfft_napi.cc")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    shim = (ROOT / "wat-fft_b200" / "napi" / "watfft_napi.cc").read_text()
    for js_call in re.findall(r"\bn\.(\w+)\(", JS):   # every native call index.js makes is registered by the shim
        assert f'"{js_call}"' in shim, js_call
