"""`python -m mcgra_b200.main ARGS` for the command-line tests, single-process or under torchrun, that also saves what
this rank computed to <out>/rank<RANK>.npz: the returned whole-graph AUC and the top-k pairs of recovered_edges().

    python tests/cli_rank_run.py <out> ARGS..."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    out, argv = sys.argv[1], sys.argv[2:]
    from mcgra_b200 import main as cli
    from mcgra_b200.topology_attack import PGDAttack
    got = {}
    recovered = PGDAttack.recovered_edges

    def keep(self, k):
        rows, cols, scores = recovered(self, k)
        got.update(rows=rows.cpu().numpy(), cols=cols.cpu().numpy(), scores=scores.cpu().numpy())
        return rows, cols, scores
    PGDAttack.recovered_edges = keep
    auc_all = cli.main(argv)
    np.savez(os.path.join(out, f"rank{os.environ.get('RANK', '0')}.npz"), auc_all=np.float64(auc_all), **got)


if __name__ == "__main__":
    main()
