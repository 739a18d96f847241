"""CPU only, and only with a checkout of the reference project named by SCD_REFERENCE_DIR (it is not part of this
repository; skipped without it): the committed fixtures are what the REAL reference code produces today - regenerate
every family into a scratch directory with oracle/gen_golden.py and compare array by array."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('SCD_REFERENCE_DIR', '')

pytestmark = pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, 'local_utils')),
                                reason='needs a checkout of the reference project (SCD_REFERENCE_DIR)')


@pytest.mark.parametrize('family,files', [
    ('kmeans', ['kmeans_blobs_demo.npz', 'kmeans_small.npz', 'kmeans_empty_cluster.npz']),
    ('constrained', ['kmeans_constrained.npz']),
    ('hungarian', ['hungarian.npz']),
    ('naming', ['naming_small.npz']),
    ('naming_strings', ['naming_ptsup_strings.npz']),
    ('eval', ['eval_small.npz']),
])
def test_fixture_family_regenerates_bit_identically(tmp_path, golden_dir, family, files):
    from oracle.gen_golden import PTSUP_STRINGS_HASH_SEED
    r = subprocess.run([sys.executable, '-m', 'oracle.gen_golden', '--ref', REF, '--only', family, '--out', str(tmp_path)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, PYTHONHASHSEED=PTSUP_STRINGS_HASH_SEED))
    assert r.returncode == 0, r.stderr[-2000:]
    for f in files:
        new, old = np.load(tmp_path / f), np.load(os.path.join(golden_dir, f))
        assert sorted(new.files) == sorted(old.files)
        for k in old.files:
            same = np.array_equal(old[k], new[k], equal_nan=True) if old[k].dtype.kind == 'f' else np.array_equal(old[k], new[k])
            assert old[k].dtype == new[k].dtype and same, (f, k)


def test_ptsup_loop_with_string_names_matches_the_reference_loop():
    """ADVICE round 1: `sorted(cand_names)` (main_ptsup.py:659) sorts NAME STRINGS and `nouns.index` resolves duplicates
    to the first column.  The real loop text is exec'd here with a string vocabulary that is NOT in lexicographic order
    and contains duplicate names, in the same interpreter as the oracle (the loop's `list(set(...) - set(...))` order
    depends on the process's string hashing; tests/golden/naming_ptsup_strings.npz holds the trace under a fixed
    PYTHONHASHSEED) - voted names, candidate lists and the re-assigned clusters must agree round by round."""
    from oracle import gen_golden as gg, naming_oracle
    _, _, lang, _ = gg.import_reference(REF)
    c = gg.ptsup_strings_case()
    trace = gg.run_reference_ptsup_strings(REF, lang, c)
    m = c['mask_lab']
    got = naming_oracle.naming_loop_ptsup(c['idx_top'][~m], c['all_preds'].copy(), m, c['feats'][~m], c['W'], c['lab_idx'],
                                          c['k_true'], top_k=5, num_common_vote=20, num_common_linear=4, nouns=c['nouns'])
    assert len(trace) >= 2 and len(got) == len(trace)
    for (names, cand, p, nu), r in zip(trace, got):
        assert r['voted'] == names and r['cand'] == cand and r['n_unique'] == nu
        assert np.array_equal(r['u_preds'], p)
    # and the index-named shortcut would NOT have produced this: the lexicographic order differs from the column order
    nouns = c['nouns']
    assert [nouns.index(s) for s in got[0]['cand']] != sorted(nouns.index(s) for s in got[0]['cand'])
