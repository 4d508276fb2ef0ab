"""The original Moby sources (github.com/PositronicsLab/Moby) are not part of this repository.  The tests that read its example
scenes take the tree from the MOBY_SOURCE_DIR environment variable and skip without it."""
import os

import pytest

ROOT = os.environ.get("MOBY_SOURCE_DIR", "")
EXAMPLE = os.path.join(ROOT, "example")
needed = pytest.mark.skipif(not ROOT or not os.path.isdir(EXAMPLE), reason="needs the original Moby sources: set MOBY_SOURCE_DIR")
