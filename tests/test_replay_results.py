"""End-to-end witness (SURVEY 8f-1/2): results files written by the OpenCV-free C++ driver (host/cvg_replay: hot path
in libcvgraft, consumer restated in host/detect_objects.cpp) in the reference's layout
(output/<folder>/<scene>_results.txt, src/Output.cpp:46, src/utils.cpp:12-20).

tests/golden/replay_output/ is derived from cv2 itself: the inlier scene points cv2 4.13.0 returns for the 1 308 accepted pairs
of the loop nest (tests/golden/full_dataset_cv2.npz, tools/full_dataset_replay.py --cv2) pushed through the C++ consumer
(tools/make_replay_golden.py) — no GPU result is involved.  The files are checked against
 (0) a regeneration from the committed cv2 points on the CPU,
 (1) the survey's independent replay with cv2 (SURVEY App. C.3 detections, Mean IoU 0.351, accuracy 12/14, 2/14, 2/14),
and the GPU test runs the driver (one GPU; every GPU of the box behind cvg_create_multi) on the stored features of two of the
test images (tests/golden/features_small.npz) and compares their results files byte for byte."""
import os
import subprocess

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
GOLD = os.path.join(ROOT, "tests", "golden", "replay_output")

# SURVEY.md App. C.3 (oracle replay of the reference with cv2 4.13.0, sorted iteration order)
ANCHORS = {
    "004_sugar_box/4_0001_000121": {"004": [382, 281, 491, 482]},
    "004_sugar_box/4_0001_000956": {"004": [143, 186, 319, 420], "006": [449, 187, 514, 324]},
    "004_sugar_box/4_0014_001409": {"004": [152, 302, 460, 503]},
    "004_sugar_box/4_0025_000065": {"004": [358, 259, 535, 413]},
    "004_sugar_box/4_0049_000003": {"004": [248, 123, 432, 318]},
    "004_sugar_box/4_0049_000815": {"004": [195, 209, 414, 345]},
    "004_sugar_box/4_0054_000215": {"004": [188, 300, 386, 414]},
    "004_sugar_box/4_0058_000001": {"004": [417, 156, 556, 278]},
    "004_sugar_box/4_0058_001715": {"004": [353, 180, 527, 457]},
    "004_sugar_box/4_0077_000659": {"004": [284, 117, 368, 199]},
    "006_mustard_bottle/6_0008_001625": {"006": [395, 166, 521, 330]},
    "006_mustard_bottle/6_0046_000002": {"006": [302, 140, 413, 352]},
    "035_power_drill/35_0030_000046": {"006": [279, 257, 356, 357], "035": [160, 194, 357, 466]},
}
EMPTY = ["006_mustard_bottle/6_0026_000077", "035_power_drill/35_0010_000001", "035_power_drill/35_0010_000491",
         "035_power_drill/35_0010_001853", "035_power_drill/35_0038_002606"]


def read_results(path):
    out = {}
    for line in open(path):
        f = line.split()
        if len(f) == 5:
            out[f[0][:3]] = [int(v) for v in f[1:]]
    return out


def find(folder_scene):
    folder, scene = folder_scene.split("/")
    hits = [f for f in os.listdir(os.path.join(GOLD, folder)) if f.startswith(scene)]
    assert len(hits) == 1, folder_scene
    return os.path.join(GOLD, folder, hits[0])


def test_golden_results_are_the_consumer_on_cv2_points():
    """The committed results files = cv2's inlier points (full_dataset_cv2.npz) through host/libcvghost_consumer.so."""
    import sys
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_replay_golden as mg
    from computervision_objectdetection_featurematching_b200 import build
    build.build()                                               # the consumer library links against libcvgraft
    G = np.load(os.path.join(ROOT, "tests", "golden", "full_dataset_cv2.npz"))
    files = mg.results_from_points(G, mg.consumer())
    assert len(files) == 30
    for (folder, scene), text in files.items():
        assert open(os.path.join(GOLD, folder, scene + "_results.txt")).read() == text, (folder, scene)


def test_golden_results_match_survey_anchors():
    assert sum(len(fs) for _, _, fs in os.walk(GOLD)) == 30
    for key, boxes in ANCHORS.items():
        assert read_results(find(key)) == boxes, key
    for key in EMPTY:
        assert read_results(find(key)) == {}, key


@pytest.mark.gpu
def test_cpp_driver_reproduces_golden_results(tmp_path):
    import sys
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import export_feature_cache_bin
    small = os.path.join(ROOT, "tests", "golden", "features_small.npz")
    cache = export_feature_cache_bin.export(small, str(tmp_path / "features_small.bin"))
    Z = np.load(small)
    want = sorted(os.path.join(str(Z["model_names"][f]), f"{n}_results.txt") for f, n in zip(Z["scene_folder"], Z["scene_names"]))
    assert len(want) == 2 and all(os.path.exists(os.path.join(GOLD, f)) for f in want)
    exe = os.path.join(ROOT, "host", "cvg_replay")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "host"), "cvg_replay"])
    import torch
    runs = [["--sync"], []]                                       # synchronous calls; three images in flight from one thread
    if torch.cuda.device_count() >= 2:
        runs.append(["--gpus", str(torch.cuda.device_count())])   # cvg_create_multi: images dealt to the GPUs in turn
    for k, extra in enumerate(runs):
        out = str(tmp_path / f"output{k}")
        r = subprocess.run([exe, cache, out] + extra, capture_output=True, text=True, cwd=os.path.join(ROOT, "host"))
        assert r.returncode == 0, r.stdout + r.stderr
        written = sorted(os.path.relpath(os.path.join(d, f), out) for d, _, fs in os.walk(out) for f in fs)
        assert written == want, (extra, written)
        for f in want:
            assert open(os.path.join(out, f)).read() == open(os.path.join(GOLD, f)).read(), (extra, f)
