"""A7, nucleotide gapped aligner.  CPU: oracle/oracle_ksw.c against the reference fixture (tests/golden/nucl_v1.npz) and against
the reference's own ksw_extz2_sse / BandedNucleotideAligner on seeded random inputs (the `ref` fixture).
GPU (-m gpu): b200_nucl_align against the fixture and the oracle."""
import numpy as np
import pytest

from mmseqs2_b200 import synth
from oracle.pyoracle import KswOracle


@pytest.fixture(scope="module")
def nucl():
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return np.load(os.path.join(root, "tests", "golden", "nucl_v1.npz"))


@pytest.fixture(scope="module")
def kso(oracle):
    d = np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden", "blosum62.npz"))
    return KswOracle(d["nucl_mat"])


def _seqs(data, off):
    return [data[int(off[i]):int(off[i + 1])] for i in range(len(off) - 1)]


def test_oracle_matches_reference_fixture(nucl, kso):
    reads, targets = _seqs(nucl["qdata"], nucl["qoff"]), _seqs(nucl["tdata"], nucl["toff"])
    gaps = 0
    for i, (qi, ti, dg) in enumerate(nucl["tasks"]):
        o, cg, bt = kso.align(reads[qi], targets[ti], int(dg))
        assert np.array_equal(o, nucl["out"][i]), i
        assert np.array_equal(cg, nucl["cigars"][int(nucl["cigar_off"][i]):int(nucl["cigar_off"][i + 1])]), i
        assert bt == str(nucl["bt"][i]), i
        gaps += o[6] > 1
    assert gaps > 100


def test_ksw_restatement_vs_reference_random(kso, ref):
    nmat = kso.mat
    rng = np.random.default_rng(77)
    for it in range(240):
        ql = int(rng.integers(1, 350))
        q = synth.nucl_genome(rng, ql)
        if it % 3 == 0:
            t = synth.nucl_genome(rng, int(rng.integers(1, 500)))
        else:
            t = np.concatenate([synth.nucl_mutate(rng, q, 0.02 + 0.2 * rng.random(), 0.05 * rng.random()),
                                synth.nucl_genome(rng, int(rng.integers(0, 200)))])
        if it % 7 == 0:
            q[::5] = 4
        for flag in (0x41, 0x40, 0x00, 0x42):
            w = 64 if it % 5 else int(rng.integers(1, 100))
            zd = 40 if it % 3 else int(rng.integers(5, 100))
            a, ca = ref.ksw_extz2(q, t, nmat, 5, 2, w, zd, flag)
            b, cb = kso.extz2(q, t, 5, 2, w, zd, flag)
            assert [a[0], a[8], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[10]] == list(b), (it, flag)
            assert np.array_equal(ca, cb), (it, flag)


def test_aligner_restatement_vs_reference_random(kso, ref):
    rng = np.random.default_rng(78)
    targets = [synth.nucl_genome(rng, int(n)) for n in rng.integers(100, 2000, 20)]
    reads, tasks = synth.nucl_reads(rng, targets, 300, 120, subst=0.06, indel=0.02)
    for i, (qi, ti, dg) in enumerate(tasks):
        dg = (int(dg) + (int(rng.integers(-4, 5)) if i % 4 == 0 else 0)) & 0xffff
        a, ca, bta = ref.nucl_align(reads[qi], targets[ti], dg if dg < 32768 else dg - 65536)
        b, cb, btb = kso.align(reads[qi], targets[ti], dg)
        assert np.array_equal(a, b) and np.array_equal(ca, cb) and bta == btb, i


@pytest.mark.gpu
def test_gpu_matches_reference_fixture(ctx, nucl):
    reads = _seqs(nucl["qdata"], nucl["qoff"])
    ctx.load_db(nucl["tdata"], nucl["toff"].astype(np.uint64), 5)
    out, cigars, bts = ctx.nucl_align(reads, nucl["tasks"])
    got = np.stack([out[f] for f in ("score", "qstart", "qend", "dbstart", "dbend", "identical", "n_cigar")], 1)
    bad = np.nonzero((got != nucl["out"]).any(1))[0]
    assert len(bad) == 0, (bad[:5], got[bad[:3]], nucl["out"][bad[:3]])
    for i in range(len(reads)):
        assert np.array_equal(cigars[i], nucl["cigars"][int(nucl["cigar_off"][i]):int(nucl["cigar_off"][i + 1])]), i
        assert bts[i] == str(nucl["bt"][i]), i


@pytest.mark.gpu
def test_gpu_matches_oracle_random(ctx, kso):
    rng = np.random.default_rng(79)
    targets = [synth.nucl_genome(rng, int(n)) for n in rng.integers(50, 6000, 60)]
    targets[1][::9] = 4
    reads, tasks = synth.nucl_reads(rng, targets, 1500, 150, subst=0.03, indel=0.01)
    for i in range(0, 1500, 6):      # long reads, tiny reads, shifted seeds
        tasks[i, 2] = (int(tasks[i, 2]) + int(rng.integers(-8, 9))) & 0xffff
    for i in range(3, 1500, 100):
        t = int(tasks[i, 1]); reads[i] = synth.nucl_mutate(rng, targets[t][:min(len(targets[t]), 900)], 0.05, 0.01); tasks[i, 2] = 0
    for i in range(7, 1500, 90):
        reads[i] = reads[i][:int(rng.integers(1, 20))]
    from oracle.pyoracle import pack_targets
    td, to = pack_targets(targets)
    ctx.load_db(td, to.astype(np.uint64), 5)
    out, cigars, bts = ctx.nucl_align(reads, tasks)
    for i, (qi, ti, dg) in enumerate(tasks):
        o, cg, bt = kso.align(reads[qi], targets[ti], int(dg))
        got = [out[f][i] for f in ("score", "qstart", "qend", "dbstart", "dbend", "identical", "n_cigar")]
        assert got == list(o), (i, got, list(o))
        assert np.array_equal(cigars[i], cg) and bts[i] == bt, i
