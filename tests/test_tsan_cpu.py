"""ThreadSanitizer over the host side of the C ABI (SURVEY 8(b) Threading, utils.rs:14-16: the error slot is thread-local,
distinct handles are independent).  A -fsanitize=thread build of the library (sourmash_rust_b200/build.py: build_tsan)
is driven by tests/host/tsan_host_calls.cpp from 8 threads: hashing, handle lifecycle and getters, the error slot,
signature JSON in and out (large enough for the reader's and the writer's own worker threads), the failure path of a
call that needs the device, private and shared handles.  Device work is outside what ThreadSanitizer can follow; the
concurrent GPU paths are covered by tests/test_gpu_round2.py (threads) for results."""
import json
import os
import random
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tsan_toolchain_works(tmp_path):
    if not shutil.which("g++"):
        return False
    src = tmp_path / "probe.cpp"
    src.write_text("#include <thread>\nint main(){ std::thread t([]{}); t.join(); return 0; }\n")
    exe = tmp_path / "probe"
    r = subprocess.run(["g++", "-fsanitize=thread", str(src), "-o", str(exe), "-lpthread"], capture_output=True)
    if r.returncode != 0:
        return False
    return subprocess.run([str(exe)], capture_output=True).returncode == 0


def test_host_calls_are_race_free(tmp_path):
    if not _tsan_toolchain_works(tmp_path):
        pytest.skip("no working -fsanitize=thread toolchain here")
    from sourmash_rust_b200 import build
    lib = build.build_tsan()
    lib_dir = os.path.dirname(lib)
    # 60 signatures x 2 sketches x 2000 hashes: ~5 MB of JSON, above the thresholds of the threaded reader (2 MiB) and
    # writer (100 000 hashes)
    rng = random.Random(5)
    sigs = []
    for i in range(60):
        sketches = []
        for k in (21, 31):
            mins = sorted(rng.sample(range(1, 1 << 62), 2000))
            d = {"num": 2000, "ksize": k, "seed": 42, "max_hash": 0, "md5sum": "0" * 32, "mins": mins, "molecule": "DNA"}
            if k == 31:
                d["abundances"] = [rng.randint(1, 9) for _ in mins]
            sketches.append(d)
        sigs.append({"class": "sourmash_signature", "email": "", "filename": "f%d.fa" % i, "name": "sample %d" % i,
                     "hash_function": "0.murmur64", "license": "CC0", "signatures": sketches, "version": 0.4})
    path = tmp_path / "sigs.json"
    path.write_text(json.dumps(sigs))
    assert path.stat().st_size > (2 << 20)
    exe = tmp_path / "tsan_host_calls"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=thread", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "host", "tsan_host_calls.cpp"), "-o", str(exe), "-L", lib_dir,
                           "-lsourmash_tsan", "-Wl,-rpath," + lib_dir, "-lpthread"])
    # (detect_deadlocks=0: signatures_save_buffer holds the lock of every handle it is given, 180 here, and the
    # sanitizer's lock-order checker gives up at 64 held locks; data-race detection is unaffected)
    # With a GPU present the device calls reach the CUDA driver, which is not instrumented: the sanitizer sees the
    # memcpy calls it makes into its own launch buffers from several threads but not the driver's own synchronisation,
    # and reports them as races.  called_from_lib ignores only calls made from inside the driver.
    supp = tmp_path / "tsan.supp"
    supp.write_text("called_from_lib:libcuda.so\n")
    env = dict(os.environ, SMB200_JSON_THREADS="4",
               TSAN_OPTIONS="halt_on_error=0 exitcode=66 detect_deadlocks=0 suppressions=%s" % supp)
    r = subprocess.run([str(exe), str(path), "8", "12"], capture_output=True, text=True, env=env, timeout=180)
    assert "ThreadSanitizer" not in r.stderr, r.stderr[-4000:]
    assert r.returncode == 0, (r.returncode, r.stdout[-2000:], r.stderr[-2000:])
    assert "0 failed checks" in r.stdout
