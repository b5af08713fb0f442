"""CPU: the package reads no environment variable that picks a code path or a tuning constant.  A variant that is
parity-clean and faster becomes the only path, and the switch that selected it goes (DESIGN.md, "Environment switches"):
a switch is a second code path that nothing runs and no test checks.  The reads that stay are listed with their reason."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "ladder-vae-pytorch_b200")

ALLOWED = {
    ("build.py", "NVCC"),        # which nvcc builds the library
    ("_capi.py", "LVAE_PDL"),    # LVAE_PDL=0: no programmatic dependent launch, for back-to-back kernel durations; same results
}


def env_reads():
    """(path relative to the package, line number, variable name or None) of every environment read."""
    sources = [(p, r"os\.environ|getenv") for p in glob.glob(os.path.join(PKG, "**", "*.py"), recursive=True)]
    sources += [(p, r"getenv\(") for p in glob.glob(os.path.join(PKG, "csrc", "*"))]
    for path, pattern in sources:
        with open(path, encoding="utf-8") as fh:
            for n, line in enumerate(fh, 1):
                if re.search(pattern, line):
                    name = re.search(r"""["']([A-Za-z_][A-Za-z0-9_]*)["']""", line)
                    yield os.path.relpath(path, PKG), n, name.group(1) if name else None


def test_only_listed_environment_reads():
    hits = list(env_reads())
    extra = ["%s:%d %s" % h for h in hits if (h[0], h[2]) not in ALLOWED]
    assert not extra, "environment switches outside the allow-list: %s" % extra
    assert {(f, v) for f, _, v in hits} == ALLOWED       # the scan does see the reads that stay
