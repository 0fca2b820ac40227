"""The C++ mirror's SolverCGMixedDevice without a GPU: a translation unit that uses it the way the
device plugins use SolverCGFullMergeDevice (solve_and_count in a run_cg_solver) compiles and links
against libbp4."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "mf_data_locality_b200")

SRC = r'''
#include "benchmark.h"
#include "solver_cg_device.h"

using DeviceVector = LinearAlgebra::distributed::Vector<double>;

template <typename Operator, typename Preconditioner>
unsigned int run_cg_solver(const Operator &A, DeviceVector &x, const DeviceVector &b, const Preconditioner &P)
{
  return solve_and_count<dealii::SolverCGMixedDevice<DeviceVector>>(A, x, b, P);
}

int main(int argc, char **argv)
{
  run(argc, argv);
}
'''


def test_mixed_device_solver_compiles_and_links(tmp_path):
    from mf_data_locality_b200 import build
    build.build_cuda()
    src = tmp_path / "mixed_plugin.cc"
    src.write_text(SRC)
    exe = tmp_path / "mixed_plugin"
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-pthread", "-Wall", "-Werror",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(PKG, "host"),
                           "-o", str(exe), str(src), "-L", PKG, "-lbp4", "-Wl,-rpath," + PKG])
    assert exe.exists()
