"""Kept for the tools' imports: the loader of the unmodified reference lives in oracle/ref_loader.py."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.ref_loader import REF_SRC, REF_TESTS, load_porepy, reference_available  # noqa: E402,F401
