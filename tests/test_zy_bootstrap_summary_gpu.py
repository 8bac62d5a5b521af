"""Bootstrap summaries at full size: C2 (80k loci x 8 haplotypes x 5M classes, with genes), model 4, 100 replicates,
every statistic against the host computation from the replicates (tests/boot_summary_checks.py)."""
import numpy as np
import pytest

from gbrs_b200 import synth
from gbrs_b200.emfactory import EMfactory
from tests import boot_summary_checks as bs

pytestmark = pytest.mark.gpu


def test_c2_summary_against_the_host():
    d = synth.generate(T=80_000, N=5_000_000, H=8)
    em = EMfactory(synth.to_apm(d))
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    summary = em.bootstrap_summary(100, model=4, seed=0, keep_replicates=True)
    assert len(summary) == 100 and np.all(summary.num_iters > 0)
    # sums over 640k values (the TPM normaliser) in different orders: a looser bound for the derived values
    worst = bs.check_summary(em, summary, summary.result, derive_rtol=1e-12)
    print(f"SUMMARY C2 B=100: derived values within {worst:.2e} of the host")
