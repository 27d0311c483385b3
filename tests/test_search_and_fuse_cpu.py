"""The batched shim Fuse(vpKFs, vScw, vpPoints, th) + Fuse(search, k, vpReplacePoint) against the loop of single-target
Fuse(KF, Scw, ...) calls of LoopClosing::SearchAndFuse (tests/cpp/search_and_fuse_test.cpp), with the shim's host code
running on the CPU oracle port of the C ABI (tests/cpp/vsg_on_oracle.cpp, and tests/cpp/vsg_on_oracle_sim3_multi.cpp for
the multi-target search).  Needs no GPU; the same program linked with libvsg_cuda runs in tests/test_gpu_fuse_sim3_multi.py."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_batched_search_and_fuse_equals_the_loop_on_the_oracle(oracle, tmp_path):
    lib = os.path.join(ROOT, "oracle")
    exe = str(tmp_path / "search_and_fuse_test_cpu")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "search_and_fuse_test.cpp"),
                           os.path.join(ROOT, "tests", "cpp", "vsg_on_oracle.cpp"),
                           os.path.join(ROOT, "tests", "cpp", "vsg_on_oracle_sim3_multi.cpp"),
                           "-L" + lib, "-lorb_oracle", "-Wl,-rpath," + lib])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "SEARCH AND FUSE TEST OK" in out.stdout
