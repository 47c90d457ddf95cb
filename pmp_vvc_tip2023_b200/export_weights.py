"""Export the reference's ``.pkl`` weights to ``.pmpw`` files, which ``pmp_weights_load`` reads from C/C++ without Python.

    python -m pmp_vvc_tip2023_b200.export_weights --modelDir DIR --outDir DIR [--missingBD error|seeded]

For every ``<comp>_Q_<qp>.pkl`` / ``<comp>_BD_<qp>.pkl`` of the reference's naming (Inference_QBD.py:219-220) it writes
``<comp>_Q_<qp>.pmpw`` / ``<comp>_BD_<qp>.pmpw``.  ``--missingBD seeded`` writes the seeded MSBD weights that
``PartitionPredictor.load_pkls(missing_bd="seeded")`` uses where a BD file is absent.  A missing tensor or a wrong shape
is an error: unlike ``load_pretrain_model``, nothing is skipped.
"""
import argparse
import os

from . import weights
from .netspec import QPS

COMPS = ("Luma", "Chroma")


def export(model_dir, out_dir, missing_bd="error", comps=COMPS, qps=QPS):
    """Returns the paths written."""
    os.makedirs(out_dir, exist_ok=True)
    paths = []
    for comp in comps:
        for qp in qps:
            sd_q, sd_bd = weights.reference_state_dicts(model_dir, comp, qp, missing_bd)
            for net, tag, sd in (("%s_Q" % comp, "Q", sd_q), ("%s_MSBD" % comp, "BD", sd_bd)):
                path = os.path.join(out_dir, "%s_%s_%d.pmpw" % (comp, tag, qp))
                weights.write_pmpw(path, net, sd)
                paths.append(path)
    return paths


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--modelDir", required=True, help="directory of the reference's <comp>_Q_<qp>.pkl / <comp>_BD_<qp>.pkl")
    ap.add_argument("--outDir", required=True)
    ap.add_argument("--missingBD", default="error", choices=["error", "seeded"],
                    help="seeded: write seeded MSBD weights where a BD .pkl is absent (benchmarking and tests only)")
    a = ap.parse_args(argv)
    for p in export(a.modelDir, a.outDir, a.missingBD):
        print(p)


if __name__ == "__main__":
    main()
