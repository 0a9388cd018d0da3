"""The C-ABI library loads and exports every symbol include/vloam_b200.h declares (no compute)."""
import ctypes
import json
import os
import re


def test_exports_match_header(pkg):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "vloam_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(vloam_b200_[a-z_0-9]+)\s*\(", hdr)))
    assert len(declared) >= 20
    lib_path = pkg._build.build_cuda()
    lib = ctypes.CDLL(lib_path)
    for sym in declared:
        assert hasattr(lib, sym), "missing export " + sym
    assert sorted(pkg.EXPORTS) == declared


def test_default_params(pkg):
    L = pkg.load_lib(build=True)
    p = pkg.Params()
    L.vloam_b200_default_params(ctypes.byref(p))
    # shipped KITTI values, loam_velodyne_HDL_64_kitti.launch:3-16
    assert (p.n_scans, p.mapping_skip_frame) == (64, 1)
    assert abs(p.minimum_range - 5.0) < 1e-7 and abs(p.line_res - 0.4) < 1e-7 and abs(p.plane_res - 0.8) < 1e-7


def test_no_oracle_in_product(pkg):
    """The product path must not reference the oracle."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pdir = os.path.join(root, "vloam-noted_b200")
    for dp, _, files in os.walk(pdir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle_py" not in txt and "liboracle" not in txt and "vloam_oracle" not in txt, f


def build_cpp_program(name, out_dir):
    """tests/cpp/<name>.cpp against vloam_adapter.hpp with the reference's include layout (ros_include/lidar_odometry_mapping/*.h)
    and the PCL / Eigen / ROS / tf2 / vloam_tf stand-ins of tests/cpp/stubs (none of those libraries is in this image), as
    C++14 like the reference (CMakeLists.txt:4-6), linked against the C-ABI library."""
    import subprocess
    import importlib
    pkg = importlib.import_module("vloam-noted_b200")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "vloam-noted_b200")
    pkg._build.build_cuda()
    exe = os.path.join(str(out_dir), name)
    subprocess.run(["g++", "-std=c++14", "-Wall", "-Werror", "-O1", "-I", os.path.join(root, "include"), "-I", os.path.join(libdir, "csrc"),
                    "-I", os.path.join(libdir, "ros_include"), "-I", os.path.join(root, "tests", "cpp", "stubs"),
                    os.path.join(root, "tests", "cpp", name + ".cpp"), "-o", exe, "-L", libdir, "-lvloam_b200", "-Wl,-rpath," + libdir], check=True)
    return exe


def test_reference_caller_compiles_against_the_adapter(tmp_path):
    """The boundary, compiled: the verbatim excerpt of vloam_main_node.cpp (construction with default constructors,
    init(std::shared_ptr<VloamTF>&), reset, the three IO calls) and the stage-by-stage driver both build and link."""
    for name in ("main_node_excerpt", "adapter_smoke"):
        assert os.path.exists(build_cpp_program(name, tmp_path))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "tests", "cpp", "main_node_excerpt.cpp")).read()
    # the marked statements really are the reference's lines (stored in tests/golden: the reference is not part of the repository)
    lines = json.load(open(os.path.join(root, "tests", "golden", "main_node_lines.json")))["lines"]
    marked = re.findall(r"^(.*?)\s*// \[MAIN\.cpp:(\d+)\]\s*$", src, re.M)
    assert len(marked) >= 11
    assert sorted(int(no) for _, no in marked) == sorted(int(no) for no in lines), "a stored reference line is no longer marked"
    for text, no in marked:
        assert lines[no] == text.strip(), (no, text, lines[no])
