"""Run the REFERENCE's own finite-volume unit tests (tests/numerics/fv/test_{mpfa,mpsa,biot}.py of the
read-only tree) with pp.Mpfa / pp.Mpsa / pp.Biot rebound to the porepy_b200 plugin classes.

    python tools/run_reference_tests.py            # wherever the reference (or its copy under oracle/_ref) is
    python tools/run_reference_tests.py functional/test_terzaghi.py [--stock] [pytest options]

With a GPU the plugin runs the CUDA path; without one the device plan is replaced by the host build of the
same node routines (tests/emu) so that the drop-in wiring can be checked in the build container.  Prints
how many discretize() calls ran on the porepy_b200 path and, with the reason, every call the plugin handed
to the reference (this tool opts into ``allow_reference_fallback``; the default plugin re-raises).  Nothing is copied
from the reference; its test files are collected where they lie."""
import collections
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
COUNTS = collections.Counter()


class Rebind:
    """pytest plugin object: rebinding happens before collection imports the test modules."""

    def pytest_configure(self, config):
        from ref_loader import load_porepy
        pp = load_porepy()
        from porepy_b200 import _lib, fv
        from porepy_b200.porepy_plugin import plugin
        try:
            gpu = _lib.load().pb_device_count() > 0
        except Exception:
            gpu = False
        if not gpu:
            from emu_binding import EmuBackedFaceGrid, EmuBackedPlan
            fv.DevicePlan = EmuBackedPlan
            fv.FaceGrid = EmuBackedFaceGrid
            import emu_binding
            fv.interface_upwind_masks = emu_binding.emu_interface_upwind_masks
        COUNTS["backend: " + ("cuda" if gpu else "host build of the node routines")] = 1
        for name in ("Mpfa", "Mpsa", "Biot", "Tpfa", "Upwind"):
            for owner, tag in ((getattr(fv, name), "porepy_b200"), (getattr(pp, name), "reference")):
                stock = owner.discretize

                def counted(self, sd, data, _stock=stock, _tag=tag, _name=name):
                    out = _stock(self, sd, data)   # counted only when it returns (no NotImplementedError)
                    COUNTS[f"{_name}.discretize on the {_tag} path"] += 1
                    return out
                owner.discretize = counted
        if "--stock" in sys.argv:  # control run: the unmodified reference in the same environment
            COUNTS["classes: stock reference (control run)"] = 1
            return
        # the reference's tests also cover what porepy_b200 refuses (periodic faces, sub-face boundary
        # conditions): opt into the counted hand-over so that those tests still run, and report every reason
        self.b200 = plugin(pp, allow_reference_fallback=True)
        self.b200.install()

    def pytest_terminal_summary(self, terminalreporter):
        terminalreporter.write_line("")
        for k in sorted(COUNTS):
            terminalreporter.write_line(f"[porepy_b200] {k}: {COUNTS[k]}")
        for k, v in sorted(getattr(getattr(self, "b200", None), "fallback_calls", {}).items()):
            terminalreporter.write_line(f"[porepy_b200] handed to the reference ({v}x): {k}")


if __name__ == "__main__":
    import pytest
    from ref_loader import REF_TESTS
    if REF_TESTS is None:
        sys.exit("reference tests not present (run oracle/make_ref.sh)")
    # extra arguments: reference test files (relative to the reference's tests/) and pytest options
    extra = [a for a in sys.argv[1:] if a.endswith(".py") or "::" in a]
    opts = [a for a in sys.argv[1:] if a not in extra and a != "--stock"]
    if extra:
        files = [os.path.join(REF_TESTS, a) for a in extra]
    else:
        files = [os.path.join(REF_TESTS, "numerics", "fv", f) for f in ("test_mpfa.py", "test_mpsa.py", "test_biot.py")]
    os.chdir("/tmp")
    sys.exit(pytest.main(files + ["-p", "no:cacheprovider", "-o", "addopts=", "-q", "--rootdir", "/tmp", *opts],
                         plugins=[Rebind()]))
