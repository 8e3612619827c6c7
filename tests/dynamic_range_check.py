"""Helper of test_gpu_dynamic_range.py: runs the device on high-dynamic-range cases in a fresh process, so that the
library reads the SSPSD_* kernel switches (at handle creation; two of them are process-wide statics).

    python dynamic_range_check.py SIGNAL_DIR OUT.npz CASE_ID...

reads each case's input from SIGNAL_DIR/<id>.npy and writes, per case, the per-stage rows of the cascade's readout
(merged units) and, for the hbf cases, the decimated samples of Psd(n).process.  The comparison against the float64
model is made by the caller, which already holds it."""
import os
import sys

import numpy as np

import dynamic_range_cases as D
import stabilizer_stream_b200 as sp


def main(signal_dir, out, ids):
    res = {}
    opts = sp.MergeOpts(keep_overlap=True, min_count=0, keep_transition_band=True)
    for cid in ids:
        case = D.case_by_id(cid)
        x = np.load(os.path.join(signal_dir, cid + ".npy"))
        c = sp.PsdCascade(case.n, hbf=sp.Hbf(case.hbf))
        c.set_detrend(sp.Detrend(case.detrend))
        c.process(x)
        for i, row in enumerate(D.merged_rows(*c.psd(opts))):
            res["%s:rows%d" % (cid, i)] = row
        if case.group == "hbf":
            res[cid + ":samples"] = sp.Psd(case.n, hbf=sp.Hbf(case.hbf)).process(x)
    np.savez(out, **res)
    print("dynamic range run ok", len(ids))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2], sys.argv[3:])
