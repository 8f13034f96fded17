"""CPU: the quad kernel source with the border of M kept the way the device keeps it (tensor memory there): outside the
private slots, behind the policy's mb_load_row / mb_store_row, both of them collectives over the whole warp.  Four cars
as one warp of quads with a staged solve must finish (a border access that not every quad reaches dead-locks the
harness, in a subprocess that is killed) and reproduce the single-quad results bit for bit, with the border scribbled
over between the two launches so that it has to come back from the record."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "tests", "host_harness")


def test_border_accessors_are_warp_collectives_and_travel_with_the_record():
    src = os.path.join(HARNESS, "step_quad_border_host.cpp")
    out = os.path.join(HARNESS, "libstep_quad_border_host.so")
    deps = [src, os.path.join(HARNESS, "step_quad_host.cpp")] + [
        os.path.join(ROOT, "ft_grandprix_b200", "csrc", f)
        for f in ("mushr_step_quad.cuh", "mushr_step.cuh", "mushr_consts.h", "mushr_mesh.h", "hfield_contact.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-pthread", "-o", out, src])
    script = os.path.join(HARNESS, "warp_lockstep_check.py")
    res = subprocess.run([sys.executable, script, ROOT, out, "60"], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.startswith("ok") and int(res.stdout.split()[1]) > 100          # suspensions really happened
