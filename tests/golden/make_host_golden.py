#!/usr/bin/env python
"""Generate host_vs_reference.npz from the REAL reference (regeirk/pycwt).

    python tests/golden/make_host_golden.py /path/to/pycwt-checkout

Runs the seeded calls of tests/test_host_vs_reference.py on the unmodified reference package
and stores its records, reduced as `reduce_record` there describes and packed by `pack`.
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def main(ref_root):
    sys.path.insert(0, ref_root)
    sys.path.insert(0, os.path.dirname(HERE))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import pycwt  # the reference
        from pycwt import helpers, mothers
    import test_host_vs_reference as T

    records = (T.mother_records(mothers) + T.helper_records(helpers)
               + T.significance_records(pycwt, mothers) + T.transform_records(pycwt))
    arrays = {}
    for key, rule, value in records:
        arrays.update(T.reduce_record(key, rule, value))
    path = os.path.join(HERE, T.FIXTURE + ".npz")
    np.savez_compressed(path, **T.pack(arrays))
    print("%-28s %8.1f KB, %d records" % (T.FIXTURE, os.path.getsize(path) / 1024, len(records)))


if __name__ == "__main__":
    main(sys.argv[1])
