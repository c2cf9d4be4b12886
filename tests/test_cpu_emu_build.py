"""The emulator library's build rule: every in-repo file the harness includes is a dependency of emu_lib.lib(), so that
an edit of any of them (e.g. include/prb_model.h regenerated from the model schema) rebuilds the library."""
import os
import subprocess

import emu_lib

ROOT = os.path.realpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))


def test_every_included_file_is_a_dependency():
    src = os.path.join(ROOT, 'tests', 'emu', 'prb_emu.cpp')
    out = subprocess.check_output(['g++', '-MM', '-std=c++17', src], cwd=ROOT, text=True)
    listed = {os.path.realpath(os.path.join(ROOT, f)) for f in out.replace('\\\n', ' ').split()[1:]}
    in_repo = {f for f in listed if f.startswith(ROOT + os.sep)}
    assert os.path.join(ROOT, 'include', 'prb_model.h') in in_repo
    assert in_repo <= set(emu_lib.deps()), sorted(in_repo - set(emu_lib.deps()))
