"""d2d_episode_record as compiled from include/drone2d.h has the size and field offsets of the ctypes structure and the
numpy dtype the Python host reads the episode log with."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

import util

FIELDS = ["seed", "step", "tracked_steps", "env", "steps", "grid_discovered", "trackers", "state_machine", "collision_flag",
          "freezing_flag", "dead_lock_flag", "reserved"]


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs a C compiler")
def test_episode_record_layout_matches_header(tmp_path):
    from gym_drone2d_activeperception_b200 import _native
    src = tmp_path / "layout.c"
    src.write_text("#include <stdio.h>\n#include <stddef.h>\n#include \"drone2d.h\"\nint main(void) {\n"
                   "    printf(\"%zu\\n\", sizeof(d2d_episode_record));\n" +
                   "".join("    printf(\"%%zu\\n\", offsetof(d2d_episode_record, %s));\n" % f for f in FIELDS) +
                   "    return 0;\n}\n")
    exe = str(tmp_path / "layout")
    subprocess.run(["gcc", "-Wall", "-Werror", "-I", os.path.join(util.ROOT, "include"), str(src), "-o", exe], check=True)
    got = [int(x) for x in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert got[0] == 48 == C.sizeof(_native.D2DEpisodeRecord) == _native.EPISODE_DTYPE.itemsize
    assert [f[0] for f in _native.D2DEpisodeRecord._fields_] == FIELDS == list(_native.EPISODE_DTYPE.names)
    for f, off in zip(FIELDS, got[1:]):
        assert getattr(_native.D2DEpisodeRecord, f).offset == off, f
        assert _native.EPISODE_DTYPE.fields[f][1] == off, f
        assert C.sizeof(dict(_native.D2DEpisodeRecord._fields_)[f]) == _native.EPISODE_DTYPE.fields[f][0].itemsize, f
