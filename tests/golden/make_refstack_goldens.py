"""Re-records tests/golden/refstack/*.npz: runs tests/test_refpin_vector.py once against the live reference stack (the
reference package on oracle/refshim), logging what the reference returns to every test (tests/refreplay.py).

  python tests/golden/make_refstack_goldens.py <reference checkout, the directory that holds the `metaworld` package>
"""
import os
import sys

import pytest

if __name__ == "__main__":
    os.environ["MW_REFSTACK_RECORD"] = os.path.abspath(sys.argv[1])
    test = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "test_refpin_vector.py")
    sys.exit(pytest.main(["-q", "-p", "no:cacheprovider", test]))
