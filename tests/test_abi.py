"""CPU-side checks of the drop-in boundary: libkta_gpu.so builds/loads here without a GPU, exports
every symbol include/kta.h declares, and refuses to compute without CUDA (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

from kafka_topic_analyzer_b200 import _native, lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "kta.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(kta_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported():
    names = _declared_symbols()
    assert len(names) >= 30
    L = C.CDLL(_native.LIB_PATH) if os.path.exists(_native.LIB_PATH) else lib()
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing


def test_binding_table_covers_header():
    assert set(_declared_symbols()) <= set(_native.SYMBOLS), set(_declared_symbols()) - set(_native.SYMBOLS)


def test_abi_version_and_structs():
    L = lib()
    assert L.kta_abi_version() == 2
    assert C.sizeof(_native.Config) == 64 and C.sizeof(_native.Batch) == 88 and C.sizeof(_native.SynthSpec) == 56


def test_header_is_plain_c():
    """The boundary must be consumable from C (cgo / Rust bindgen / ctypes): compile it as C11."""
    src = '#include "kta.h"\nint main(void){kta_config c; c.struct_size=(int)sizeof c; return kta_abi_version()==KTA_ABI_VERSION?0:c.struct_size;}\n'
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), "-x", "c", "-"],
                       input=src, text=True, capture_output=True)
    assert r.returncode == 0, r.stderr


def _without_cuda():
    """Environment in which no CUDA device is visible, also on a machine that has one."""
    return dict(os.environ, CUDA_VISIBLE_DEVICES="")


def test_no_cpu_fallback_without_cuda():
    lib()                                   # make sure the library is built
    code = ("from kafka_topic_analyzer_b200 import KtaEngine, KtaError\n"
            "try:\n    KtaEngine(4)\nexcept KtaError as e:\n    print(e.code)\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=_without_cuda(), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == str(_native.ERR_CUDA), r.stdout


def test_product_never_touches_the_oracle():
    """Nothing under the package, include/ or bench-independent code may reference oracle/."""
    pkg = os.path.join(ROOT, "kafka_topic_analyzer_b200")
    bad = []
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".hpp")):
                txt = open(os.path.join(d, f), errors="replace").read()
                if re.search(r"kta_oracle|libkta_oracle|oracle_lib|kto_", txt):
                    bad.append(os.path.join(d, f))
    assert not bad, bad


def test_sass_has_bulk_copy_and_no_legacy_paths():
    """The fused kernel really uses the Blackwell/Hopper bulk async copy (UBLKCP) + mbarrier (SYNCS)."""
    r = subprocess.run(["cuobjdump", "-sass", _native.LIB_PATH], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "UBLKCP" in r.stdout and "SYNCS" in r.stdout and "ATOMS" in r.stdout
    assert "sm_100a" in r.stdout


def test_abi_rejects_bad_arguments_without_cuda():
    """Argument validation happens before any CUDA call, so it is checkable here (and never aborts the host)."""
    L = lib()
    h = C.c_void_p()
    cfg = _native.Config()
    cfg.struct_size = 12                      # wrong size: an ABI mismatch must be refused, not misread
    assert L.kta_create(C.byref(cfg), C.byref(h)) == _native.ERR_INVALID and not h
    assert b"struct_size" in L.kta_last_error()
    assert L.kta_create(None, C.byref(h)) == _native.ERR_INVALID
    out = C.c_uint64()
    assert L.kta_counter(None, 0, 0, C.byref(out)) == _native.ERR_INVALID
    assert L.kta_push(None, 0, 0, 0, None, -1, -1) == _native.ERR_INVALID
    assert L.kta_destroy(None) == 0
    assert L.kta_merge_words(None, 2) == -1
    spec = _native.SynthSpec()
    assert L.kta_synth_shard_records(C.byref(spec), 0, 1) == -1      # zero partitions


def _build_c_example(tmp_path):
    """integration/c/minimal.c: the boundary used from plain C11 (no C++, no torch)."""
    exe = str(tmp_path / "kta_minimal")
    libdir = os.path.join(ROOT, "kafka_topic_analyzer_b200")
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "integration", "c", "minimal.c"), "-L", libdir, "-lkta_gpu",
                        "-Wl,-rpath," + libdir, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_c_example_links_and_fails_loudly_without_cuda(tmp_path):
    from kafka_topic_analyzer_b200 import lib
    lib()                                   # make sure the library is built
    exe = _build_c_example(tmp_path)
    r = subprocess.run([exe], env=_without_cuda(), capture_output=True, text=True)
    assert r.returncode == 2 and r.stderr.startswith("kta_create:") and r.stdout == ""


@pytest.mark.gpu
def test_c_example_output(tmp_path):
    r = subprocess.run([_build_c_example(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout.splitlines() == [
        "partition 0: total 3 tombstones 1 key bytes 18 value bytes 120 dirty ratio 33.3333",
        "partition 1: total 2 tombstones 0 key bytes 6 value bytes 90 dirty ratio 0.0000",
        "alive keys: 2",
    ]


def test_reference_arm_never_maps_the_gpu_library():
    """bench.py --impl reference is a CPU arm: its topic comes from the host-only generator (libkta_synth.so) and the
    oracle; libkta_gpu.so must not even be loaded into that process."""
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '1', '--cpu-sample', '50000'];"
            "runpy.run_path(%r, run_name='__main__');"
            "maps = open('/proc/self/maps').read();"
            "assert 'libkta_synth.so' in maps and 'libkta_oracle.so' in maps, 'expected libraries missing';"
            "assert 'libkta_gpu' not in maps, 'the reference arm mapped the GPU library'") % os.path.join(ROOT, "bench.py")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = __import__("json").loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and d["config"]["config"] == "C1" and d["config"]["records_per_gpu"] == 100_000_000
