"""Input readers and their lowering to batch tensors (raoteh_b200/io.py; reference
examples/p53/app_helper.py:23-184, p53.py:76-100, blink.py:229-270)."""
import io
import os

import numpy as np
import pytest

from helpers import GOLDEN
from raoteh_b200 import io as rio
from raoteh_b200.lowering import TreeSchedule

CODE = """0\tala\tgct
1\tala\tgcc
2\targ\tcgt
3\tcys\ttgc
4\ttyr\ttac
5\tstop\ttaa
"""


def test_read_newick_numbering_and_weights():
    T, root, leaves = rio.read_newick(io.StringIO("((A:0.1,'B b':0.2)x:0.3,[c]C:0.4);"))
    assert leaves == [(0, 'A'), (1, 'B b'), (2, 'C')]
    assert root == 4 and sorted(T) == [0, 1, 2, 3, 4]
    assert T[3][0]['weight'] == 0.1 and T[3][1]['weight'] == 0.2
    assert T[4][3]['weight'] == 0.3 and T[4][2]['weight'] == 0.4
    with pytest.raises(ValueError):
        rio.read_newick(io.StringIO('((A,B),C)'))


def test_read_genetic_code_and_maps():
    code = rio.read_genetic_code(io.StringIO(CODE))
    assert (5, 'STOP', 'TAA') not in code and len(code) == 5
    c2s, s2r, r2p, s2p = rio.codon_state_maps(code)
    assert c2s['TGC'] == 3 and s2r[4] == 'TYR'
    assert r2p == {'ALA': 0, 'ARG': 1, 'CYS': 2, 'TYR': 3} and s2p[1] == 0


def test_read_phylip_both_layouts_and_lowering():
    T, root, leaves = rio.read_newick(io.StringIO('((Has:0.1,Ptr:0.2):0.3,Mmu:0.4);'))
    code = rio.read_genetic_code(io.StringIO(CODE))
    c2s = rio.codon_state_maps(code)[0]
    a = "3 9\n\nHas  GCTTGCTAC\n\nPtr  gccTGCnnn\n\nMmu  CGT---TAC\n"
    b = "3 9\n\nHas\nGCT TGC TAC\n\nPtr\ngcc TGC\nnnn\n\nMmu\nCGT --- TAC\n"
    sched = TreeSchedule.from_nx(T, root)
    want = np.array([[0, 3, 4], [1, 3, 255], [2, 255, 4]], dtype=np.uint8)
    for text in (a, b):
        rows = list(rio.read_phylip(io.StringIO(text), ntaxa=3, ncodons=3))
        assert [r[0] for r in rows] == ['Has', 'Ptr', 'Mmu']
        codes, leaf_nodes = rio.alignment_to_codes(rows, leaves, sched, c2s)
        assert np.array_equal(codes, want)
        assert [sched.nodes[i] for i in leaf_nodes] == [0, 1, 2]
    with pytest.raises(Exception):
        list(rio.read_phylip(io.StringIO(a), ntaxa=4))


def test_read_disease_data_and_tolerance_observations():
    text = "467 135 5 TGC TAC Cys Tyr\n470 136 5 TGC TGCINS Cys Cys2\n12 2 1 GCT CGT Ala Arg\n"
    d = rio.read_disease_data(io.StringIO(text))
    assert d == {134: {'TYR'}, 1: {'ARG'}}
    r2p = {'ALA': 0, 'ARG': 1, 'CYS': 2, 'TYR': 3}
    tol = rio.disease_to_tol_obs(d, r2p, 4, 140)
    assert tol.shape == (1, 4, 140)
    assert tol[0, 3, 134] == 1 and tol[0, 1, 1] == 1 and int((tol == 1).sum()) == 2
    assert tol[0, 0, 0] == 2                      # no data: tolerated
    with pytest.raises(Exception):
        rio.read_disease_data(io.StringIO("1 1 1 GCT GCC Ala Ala\n"))


@pytest.mark.reference
def test_reference_p53_inputs_parse():
    from oracle import ref_shim
    base = os.path.join(ref_shim.REFERENCE_ROOT, 'examples', 'p53')
    with open(os.path.join(base, 'p53S.const.tree')) as f:
        T, root, leaves = rio.read_newick(f)
    assert len(T) == 49 and len(leaves) == 25 and leaves[0][1] == 'Has'
    np.testing.assert_allclose(T.size(weight='weight'), 4.8)
    with open(os.path.join(base, 'universal.code.txt')) as f:
        code = rio.read_genetic_code(f)
    assert len(code) == 61
    with open(os.path.join(base, 'alignment.for.codeml.phylip')) as f:
        rows = list(rio.read_phylip(f, ntaxa=25, ncodons=393))
    c2s, s2r, r2p, s2p = rio.codon_state_maps(code)
    sched = TreeSchedule.from_nx(T, root)
    codes, leaf_nodes = rio.alignment_to_codes(rows, leaves, sched, c2s)
    assert codes.shape == (25, 393) and len(r2p) == 20
    assert (codes[0] != 255).all()                # the human sequence has no gaps or stops


def test_mg94_matches_reference_recipe():
    # the standard genetic code as an index / residue / codon table like the reference's
    # examples/p53/universal.code.txt, residues in alphabetical order, the stop codons last
    with open(os.path.join(GOLDEN, 'universal.code.txt')) as f:
        code = rio.read_genetic_code(f)
    assert len(code) == 61
    Q, distn, s2r, r2p = rio.mg94_from_genetic_code(0.25039, 0.30126, 0.25952, 0.18883, 3.17632,
                                                    0.21925, code, target_expected_rate=1.0)
    np.testing.assert_allclose(Q.sum(axis=1), 0, atol=1e-12)
    np.testing.assert_allclose(-(distn * np.diag(Q)).sum(), 1.0)
    np.testing.assert_allclose(distn @ Q, 0, atol=1e-12)      # reversible: distn is stationary
    # same model as the synthetic generator, up to the state order
    from raoteh_b200 import synth
    Q2, pi2, res2 = synth.mg94()
    codons2, _ = synth.universal_code()
    order = [codons2.index(c) for s, r, c in code]
    np.testing.assert_allclose(Q, Q2[np.ix_(order, order)], rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(distn, pi2[order], rtol=1e-12)
