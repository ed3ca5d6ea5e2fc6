"""CPU (only where $SWEEPTT_REFERENCE names a checkout of the original project): the binding of INTEGRATION.md 1
applied mechanically to a TEMPORARY copy of the reference's serial_new/sweep-tt-multistart.c -- include the header after
the file's own struct definitions, replace the sweep loop (:150-170) by one sweeptt_solve call -- builds with the
reference's flags, links against libsweeptt.so, and runs the reference's own main() up to our call: without a GPU the
call must fail loudly with the library's message, on a GPU machine it must run.  Without the checkout the test is
skipped and the CLI test covers the run.  Nothing of the reference is copied into the repository."""
import os
import pathlib
import re
import subprocess

import pytest
import torch

import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import workloads as W

from conftest import ROOT

REF_DIR = pathlib.Path(os.environ["SWEEPTT_REFERENCE"]) if os.environ.get("SWEEPTT_REFERENCE") else None
REF = REF_DIR / "serial_new" / "sweep-tt-multistart.c" if REF_DIR else None

CALL = r'''
  {
    float *out[STARTMAX];
    sweeptt_opts opts;
    sweeptt_stats st;
    memset(&opts, 0, sizeof opts);
    opts.struct_size = sizeof opts;
    opts.device = -1;
    for (s = 0; s < numstart; s++) out[s] = ttboxes[s].flat;
    if (!sweeptt_solve(vbox.box.flat, nx, ny, nz, fs, starsize, start, numstart, out, &opts, &st)) {
      printf("sweep failed: %s\n", sweeptt_last_error());
      exit(1);
    }
    printf("sweep %d finished: anychange = %d\n", st.rounds, 0);
  }
'''


@pytest.mark.skipif(REF is None or not os.path.isfile(REF), reason="needs a checkout of the original project in $SWEEPTT_REFERENCE")
def test_binding_patch_builds_links_and_reaches_our_call(tmp_path):
    src = REF.read_text()
    # 1. our header after the file's own struct definitions
    marker = "int\t\tchanged[STARTMAX];"
    assert marker in src
    src = src.replace(marker, '#include <string.h>\n#define SWEEPTT_NO_STRUCTS\n#include "sweeptt.h"\n' + marker, 1)
    # 2. the sweep loop -> one call
    a = src.index("  /* sweep until no change in travel times occur */")
    b = src.index("  /* TODO: Remove exit statement so output can complete. */")
    src = src[:a] + CALL + src[b:]
    patched = tmp_path / "sweep-tt-multistart.c"
    patched.write_text(src)
    exe = tmp_path / "sweep-tt-multistart"
    lib = P.lib_path()
    subprocess.run(["gcc", "-O3", "-Wfatal-errors", "-w", f"-I{REF_DIR / 'include'}", f"-I{ROOT / 'include'}", "-o", str(exe),
                    str(patched), f"-L{lib.parent}", "-lsweeptt", f"-Wl,-rpath,{lib.parent}", "-lm"], check=True)
    v = W.heterogeneous_field((12, 11, 9), 3)
    P.vbox_store(tmp_path / "m.vbox", v, origin=(1, 1, 1))
    W.write_star_file(tmp_path / "fs.txt", W.star("3"))
    W.write_start_file(tmp_path / "start.txt", [(5, 5, 4)])
    r = subprocess.run([str(exe), "m.vbox", "fs.txt", "start.txt"], cwd=tmp_path, capture_output=True, text=True, timeout=120)
    assert "Velocity model dimensions: 12 x 11 x 9" in r.stdout and "Starting points read" in r.stdout
    if torch.cuda.is_available():
        assert r.returncode == 0 and re.search(r"sweep \d+ finished: anychange = 0", r.stdout)
        assert (tmp_path / "output.tt").exists()
    else:
        assert r.returncode == 1 and "sweep failed: no CUDA device" in r.stdout
