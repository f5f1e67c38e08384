"""The C-ABI library loads and exports every symbol include/vxs.h declares; without a GPU it fails loudly (no CPU fallback)."""
import ctypes as C
import os

import pytest
import torch

import synth
import voxel_slam_b200 as vx


SHIM_USE = r'''
#define VXS_SHIM_WITH_REFERENCE_TYPES
#include "voxel_slam_b200/csrc/shim/voxel_ba_shim.hpp"
// the call sites of voxelslam.cpp, with the reference's own argument types
void use(std::vector<IMUST>& xs, std::deque<IMU_PRE*>& imus, std::vector<Keyframe*>& smps, PVec& pvec, PVecPtr pptr, pcl::PointCloud<PointType>& pl,
         std::vector<std::vector<SlideWindow*>>& sws, PLV(3)& pwld, vxs_map_params& mpar) {
  vxs_shim::LidarFactor f(int(xs.size()));                                   // LidarFactor voxhess(win_size)            voxel_map.hpp:120
  std::vector<PointCluster> pcrs(xs.size()); PointCluster fix, add; Eigen::Vector3d ev; Eigen::Matrix3d U;
  vxs_shim::push_voxel(f, pcrs, fix, 1.0, ev, U, add);                        // voxel_map.hpp:1321
  Eigen::MatrixXd hess; std::vector<double> resis;
  vxs_shim::li_ba_damping_iter(xs, f, imus, &hess, 1e-4);                     // voxelslam.cpp:1652-1653
  vxs_shim::li_ba_gravity_damping_iter(xs, f, imus, resis, &hess, 5, 1e-4);   // voxelslam.cpp:632-634, 1643-1645
  vxs_shim::lidar_ba_damping_iter(xs, f, &hess, resis, 4, 2);                 // voxelslam.cpp:2381-2384
  vxs_shim::SurfMap surf_map(mpar, int(xs.size()));
  vxs_shim::cut_voxel_multi(surf_map, pptr, int(xs.size()) - 1, surf_map, int(xs.size()), pwld, sws);   // voxelslam.cpp:1612
  vxs_shim::cut_voxel(surf_map, pptr, int(xs.size()) - 1, surf_map, int(xs.size()), pwld, sws[0]);      // voxelslam.cpp:619, 1176
  vxs_shim::multi_recut(surf_map, int(xs.size()), xs, f, sws);                // voxelslam.cpp:1615
  vxs_shim::multi_margi(surf_map, 0.0, int(xs.size()), xs, f, sws[0]);        // voxelslam.cpp:1669
  vxs_shim::GbaMap oct_map(mpar);
  vxs_shim::OctreeGBA_cut_voxel(oct_map, xs[0], smps[0]->plptr, 0, int(xs.size()));   // voxelslam.cpp:2376
  vxs_shim::OctreeGBA_multi_recut(oct_map, f, 2);                             // voxelslam.cpp:2379
  vxs_shim::Context& c = vxs_shim::default_context();
  vxs_shim::down_sampling_voxel(c, pl, 0.1);
  vxs_shim::down_sampling_close(c, pl, 0.1);
  vxs_shim::down_sampling_pvec(c, pvec, 0.1, pl);
  vxs_shim::submap_merge(c, xs, smps, 1.0, pl);
  vxs_shim::var_init(c, xs[0], pl, pptr, 0.02, 0.05);                          // voxelslam.cpp:1246, 1584
  vxs_shim::pvec_update(c, pptr, xs[0], pwld);                                 // voxelslam.cpp:1250, 1594
  Eigen::Matrix<double, 6, 6> HTH; Eigen::Matrix<double, 6, 1> HTz; Eigen::Matrix3d nnt;
  int match_num = vxs_shim::odom_accumulate(surf_map, pptr, xs[0], true, HTH, HTz, nnt);   // voxelslam.cpp:876-918
  (void)match_num;
  std::vector<std::vector<IMUST>> win_xs; std::vector<int32_t> wf{0}, st;
  vxs_shim::hba_bottom_batch(c, mpar, smps, wf, 10, win_xs, st);               // voxelslam.cpp:2540-2557 (every HBA_add_edge(..., 1, 2, plptr) at once)
}
int main() { return 0; }
'''


def test_library_exports_every_declared_symbol():
    syms = vx.declared_symbols()
    assert len(syms) >= 25 and "vxs_li_ba" in syms and "vxs_build_window_factor" in syms
    lib = vx.lib()
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, missing
    assert lib.vxs_version() >= 100


def test_harness_library_loads():
    p = synth.true_pose(20.0, 3)
    assert p.shape == (12,) and abs(p[9] - 10.15) < 1e-12
    pts = synth.gen_scan(20.0, 0, 1000, synth.true_pose(20.0, 0))
    assert pts.shape == (1000, 3) and abs(pts).max() < 40
    assert (synth.gen_scan(20.0, 0, 1000, synth.true_pose(20.0, 0)) == pts).all()          # seeded, reproducible


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    with pytest.raises(vx.VxsError) as ei:
        vx.Context(0)
    assert ei.value.code == -1


def test_product_never_touches_the_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    bad = []
    for d, _, files in os.walk(os.path.join(root, "voxel_slam_b200")):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")) or fn == "Makefile":
                txt = open(os.path.join(d, fn), errors="ignore").read()
                if "oracle/" in txt or "liboracle" in txt or "oracle_api" in txt or "vxo_" in txt:
                    bad.append(os.path.join(d, fn))
    assert not bad, bad


def test_cpp_shim_plain_layer_compiles():
    """The header-only C++ shim with the reference's class names compiles (plain layer; the Eigen-typed layer needs the reference headers)."""
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with tempfile.NamedTemporaryFile("w", suffix=".cpp", delete=False) as f:
        f.write('#include "voxel_slam_b200/csrc/shim/voxel_ba_shim.hpp"\nint main() { vxs_shim::Lidar_BA_Optimizer o; return o.thd_num == 2 ? 0 : 1; }\n')
    r = subprocess.run(["g++", "-std=c++14", "-fsyntax-only", "-I", root, f.name], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_cpp_shim_typed_layer_type_checks_against_reference_signatures():
    """The Eigen/PCL-typed layer of the shim (push_voxel, damping_iter wrappers, IMU adapter, down-sampling, submap merge) type-checks against
    stand-ins that mirror the reference's names, members and call signatures (tests/shim_stubs/reference_stubs.hpp; Eigen/PCL are not
    installed here), instantiated the way voxelslam.cpp calls them."""
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = '#include "tests/shim_stubs/reference_stubs.hpp"\n' + SHIM_USE
    with tempfile.NamedTemporaryFile("w", suffix=".cpp", delete=False) as f:
        f.write(src)
    r = subprocess.run(["g++", "-std=c++14", "-fsyntax-only", "-I", root, f.name], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr




def test_bench_reference_arm_contract_on_cpu():
    """`bench.py --impl reference` needs no GPU: one JSON line with the contract keys (tiny window so that it runs in seconds)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--win", "6", "--pts-per-scan", "4000", "--L", "8", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, cwd=root, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "e2e", "cpu_baseline", "config"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 0 and d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["cpu_baseline"]["all_cores_variant"].get("value", 0) > 0


def test_every_entry_point_rejects_null_arguments_without_a_gpu():
    """Error behaviour of the boundary: every function of include/vxs.h called with all-NULL / zero arguments returns (VXS_ERR_ARG or another negative
    code; destroy / free of NULL are no-ops) instead of dereferencing anything — on a box without a GPU, so no compute call is involved.  One subprocess:
    a crash must fail this test, not take the suite down."""
    import json
    import re
    import subprocess
    import sys
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "vxs.h")).read()
    calls = []
    for s in vx.declared_symbols():
        m = re.search(r"\b" + s + r"\s*\(([^;]*?)\)\s*;", hdr, re.S)
        assert m, s
        a = m.group(1).strip()
        n, depth = (0 if a in ("", "void") else 1), 0
        for ch in a:
            depth += ch == "("; depth -= ch == ")"
            n += ch == "," and depth == 0
        calls.append((s, n))
    assert len(calls) >= 60
    code = "import ctypes as C, sys, json\nsys.path.insert(0, %r)\nimport voxel_slam_b200 as vx\nL = vx.lib()\nout = {}\nfor s, n in %r:\n    f = getattr(L, s); f.restype = C.c_int32\n" \
           "    print('CALL', s, flush=True)\n    out[s] = f(*([C.c_void_p(0)] * n))\nprint('RESULT', json.dumps(out))\n" % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), calls)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    last = [l for l in r.stdout.splitlines() if l.startswith("CALL")][-1:]
    assert r.returncode == 0, (r.returncode, last, r.stderr[-400:])
    res = json.loads([l for l in r.stdout.splitlines() if l.startswith("RESULT")][-1][7:])
    benign = {"vxs_version", "vxs_ctx_destroy", "vxs_factor_destroy", "vxs_map_destroy", "vxs_ctx_launch_count", "vxs_ctx_last_error", "vxs_host_free"}
    wrong = {s: v for s, v in res.items() if s not in benign and not v < 0}
    assert not wrong, wrong
