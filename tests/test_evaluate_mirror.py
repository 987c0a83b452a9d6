"""svnicp_evaluate through the header-only C++ mirror: SVGDICP::evaluate (inherited by SVNICP, reachable through
SVNICPBatch::stream) compiles and links against the C ABI.  Runs without a GPU: construction must then fail loudly."""
import os
import subprocess

from conftest import ROOT

SRC = r"""
#include "svnicp/SVNICP.hpp"
int main() {
  svnicp::SteinICPParam p;
  std::vector<double> ip(6 * 4, 0.0);
  int reached = 0;
  try {
    svnicp::SVNICP icp(p, ip);
    reached = 1;
    svnicp::SVGDICP &base = icp;
    svnicp::SVGDICP::Evaluation e = base.evaluate(std::vector<double>(6, 0.0), true, true);  // before stein_align: throws
    (void)e;
    return 3;
  } catch (const svnicp::Error &) {
  }
  try {
    svnicp::SVNICPBatch b(p, 2, 4, std::vector<double>(2 * 6 * 4, 0.0));
    auto e = b.stream(1).evaluate(std::vector<double>(12, 0.0), false);
    return e.n_poses == 2 ? 4 : 5;
  } catch (const svnicp::Error &) {
  }
  return reached ? 10 : 0;
}
"""


def test_mirror_evaluate_compiles(tmp_path):
    from svn_icp_b200 import build
    lib = build.build()
    src, exe = os.path.join(tmp_path, "eval.cpp"), os.path.join(tmp_path, "eval")
    open(src, "w").write(SRC)
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "svn_icp_b200", "include"), src,
                           "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib)])
    import torch
    assert subprocess.call([exe]) == (10 if torch.cuda.is_available() else 0)
