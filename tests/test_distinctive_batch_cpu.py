"""The batched shim ORBmatcher::ComputeDistinctiveDescriptors(vpMPs) against the loop of MapPoint::ComputeDistinctiveDescriptors
calls of LocalMapping (tests/cpp/distinctive_batch_test.cpp), with the shim's host code running on the CPU oracle port of
the C ABI (tests/cpp/vsg_on_oracle.cpp, and tests/cpp/vsg_on_oracle_distinctive.cpp for vsg_distinctive_descriptors).  Needs
no GPU; the same program linked with libvsg_cuda runs in tests/test_gpu_distinctive_descriptors.py."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_batched_distinctive_descriptors_equal_the_loop_on_the_oracle(oracle, tmp_path):
    lib = os.path.join(ROOT, "oracle")
    exe = str(tmp_path / "distinctive_batch_test_cpu")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "distinctive_batch_test.cpp"),
                           os.path.join(ROOT, "tests", "cpp", "vsg_on_oracle.cpp"),
                           os.path.join(ROOT, "tests", "cpp", "vsg_on_oracle_distinctive.cpp"),
                           "-L" + lib, "-lorb_oracle", "-Wl,-rpath," + lib])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "DISTINCTIVE BATCH TEST OK" in out.stdout
