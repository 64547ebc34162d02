"""compute-sanitizer over small end-to-end solves (every kernel family, narrow and wide instantiations):
memcheck and racecheck must be clean.  SURVEY.md section 5: the reference has no race detection at all."""
import os
import shutil
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('tool', ['memcheck', 'racecheck'])
def test_compute_sanitizer_clean(tool):
    exe = shutil.which('compute-sanitizer') or '/usr/local/cuda/bin/compute-sanitizer'
    if not os.path.exists(exe):
        pytest.skip('compute-sanitizer not installed')
    try:
        out = subprocess.run([exe, '--tool', tool, '--error-exitcode', '9', sys.executable, os.path.join(ROOT, 'scripts', 'sanitize_target.py')],
                             cwd=ROOT, capture_output=True, text=True, timeout=900)
    except PermissionError:
        pytest.skip('compute-sanitizer is installed but this user may not run it')
    text = out.stdout + out.stderr
    assert out.returncode == 0, text[-3000:]
    assert ('ERROR SUMMARY: 0 errors' in text) or ('0 hazards displayed (0 errors, 0 warnings)' in text), text[-2000:]
