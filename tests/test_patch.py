"""patches/reference_cvgraft.patch only adds lines, to the three seam files, and carries the three hooks INTEGRATION.md
describes: the CMake option, the upload after the model loop, the fused call at the head of the view loop."""
import os

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
PATCH = os.path.join(ROOT, "patches", "reference_cvgraft.patch")


def test_patch_touches_only_the_three_seam_files():
    files = [l.split()[1][2:] for l in open(PATCH) if l.startswith("+++ b/")]
    assert sorted(files) == ["CMakeLists.txt", "src/ModelsDetector.cpp", "src/TestsDetector.cpp"]
    added = [l[1:] for l in open(PATCH) if l.startswith("+") and not l.startswith("+++")]
    removed = [l for l in open(PATCH) if l.startswith("-") and not l.startswith("---")]
    assert not removed                                           # nothing of the reference is deleted: the option OFF build is unchanged
    assert any("option(USE_CVGRAFT" in l for l in added)
    assert any("cvg::uploadModels(models, cvg::residentModels())" in l for l in added)
    assert any("cvg::detectAtScale(cvg::residentModels()" in l for l in added)


def test_added_source_lines_are_behind_the_option():
    """With USE_CVGRAFT off the preprocessor removes every line the patch adds to the two sources."""
    name, depth, checked = None, 0, 0
    for line in open(PATCH):
        if line.startswith("+++ b/"):
            name, depth = line.split()[1][2:], 0
        elif line.startswith("+") and name.endswith(".cpp"):
            text = line[1:].strip()
            if text == "#ifdef USE_CVGRAFT":
                depth += 1
            elif text == "#endif" and depth:
                depth -= 1
            else:
                assert depth > 0 or not text, (name, text)
                checked += 1
    assert checked > 0 and depth == 0
