#!/usr/bin/env python
"""Generate tests/golden/*.npz from the REFERENCE's own dsp headers (oracle/_ref/libsdrpp_ref.so, built from
/root/reference by oracle/Makefile).  Runs only in the authoring container; the fixtures are committed so that
the oracle restatement (and through it the CUDA path) stays pinned to the reference's control flow on machines
where /root/reference does not exist.  Inputs are regenerated from the seeds stored in each file, so the fixtures
hold outputs only (kept small: heads/tails + order-sensitive checksums for the long streams).

  reference_path.npz  run_cases on the reference build
  oracle_vs_ref.npz   a SHA-256 of every output of the VS_REF cases on the reference build, the RDS group chain's symbols
                      in full, and what the reference's own RDS group decoder (rds.cpp) reads from the bit streams"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle.oracle import Block, Oracle  # noqa: E402
from golden_cases import VS_REF, rds_group_signal, run_cases, sha256, vs_ref_blocks  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def vs_ref(R):
    g = {}
    for case, fn in VS_REF.items():
        for name, a in fn(R).items():
            g[case + "__" + name] = sha256(a)
    # the reference's stereo branch behind the same discriminator gives the same RDS output as its mono branch
    R.lib.orc_wfm_rds_stereo_create.restype = C.c_void_p
    R.lib.orc_wfm_rds_stereo_create.argtypes = [C.c_double, C.c_double]
    for seed in (1, 2):
        y = vs_ref_blocks(R, seed)["vfo_in"]
        g["blocks_seed%d__wfm_rds_stereo_branch" % seed] = sha256(
            Block(R.lib, R.lib.orc_wfm_rds_stereo_create(75e3, 250e3), 2, 2).process_chunks(y, 1250))
    bits, _ = rds_group_signal()
    chain = VS_REF["rds_groups"](R)
    g["rds_groups__soft_full"] = chain["soft"]
    g["rds_groups__hard_full"] = chain["hard"]
    for what, b in (("generator", bits), ("chain", chain["hard"])):
        pi, ps = R.rds_group_decode(b)
        g["rds_decoder__%s_pi" % what] = np.array(-1 if pi is None else pi, np.int64)
        g["rds_decoder__%s_ps" % what] = np.array("" if ps is None else ps)
    return g


def main():
    os.makedirs(OUT, exist_ok=True)
    R = Oracle("reference")
    assert R.impl() == "reference-headers"
    for name, g in (("reference_path.npz", run_cases(R)), ("oracle_vs_ref.npz", vs_ref(R))):
        np.savez_compressed(os.path.join(OUT, name), **g)
        sz = os.path.getsize(os.path.join(OUT, name))
        print("wrote tests/golden/%s: %d arrays, %d bytes" % (name, len(g), sz))


if __name__ == "__main__":
    main()
