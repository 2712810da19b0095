"""Core-genome FASTA written on the device: byte-for-byte equality with the numpy formatter of download_core()
(tests/fasta_reference.py) in whole and SNP mode, the cross-checks with the CSV, the diversity reduction and the
allele counts, the deferred recombination materialised before reading, column shards and groups, errors, and
--print_fasta / --print_snp_alignment in both command lines."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import pansim_b200 as pb
from fasta_reference import CODES, fasta_columns, fasta_letters, fasta_text

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _sim(N, L, **kw):
    return pb.Pansim.from_params(pb.Params(pop_size=N, core_size=L, pan_genes=40, core_genes=10, HR_rate=0.0,
                                           HGT_rate=0.0, **kw))


def forced_state(rng, N, L, anc):
    """Random rows with columns forced on purpose: all ancestral, fixed for another letter, exactly 2, 3 and 4
    letters, and a polymorphic last site."""
    core = (1 << rng.integers(0, 4, (N, L))).astype(np.uint8)
    code = np.searchsorted(CODES, anc)

    def others(s, k):
        return [int(CODES[(code[s % L] + 1 + i) % 4]) for i in range(k)]

    def force(col, letters):
        s = col % L
        core[:, s] = np.array(letters, np.uint8)[np.arange(N) % len(letters)]

    force(0, [anc[0]])                                  # every row ancestral: a constant site
    force(1, others(1, 1))                              # fixed for another letter: whole mode only
    force(2, [anc[2 % L]] + others(2, 1))               # 2 letters
    force(4, others(4, 3))                              # 3 letters
    force(6, [anc[6 % L]] + others(6, 3))               # all 4 letters
    core[:, 7::5] = anc[7::5]                           # more constant sites
    force(L - 1, [1, 8])                                # polymorphic last site (N >= 2)
    return core


def check_against_reference(sim, core, tmp_path):
    """Both modes of write_core_fasta and export_core_fasta_rows against the numpy formatter of `core`."""
    N = core.shape[0]
    for snps in (False, True):
        path = str(tmp_path / f"a{int(snps)}.fasta")
        want, cols, const = fasta_text(core, snps)
        res = sim.write_core_fasta(path, snps_only=snps)
        got = open(path, "rb").read()
        assert got == want, snps
        assert res.bytes == len(want) and res.columns == cols and res.const_counts.tolist() == const.tolist()
        assert int(res.const_counts.sum()) + res.columns == core.shape[1]
        r0 = N // 3
        let = sim.export_core_fasta_rows(r0, N, snps_only=snps)
        assert let.shape == (N - r0, cols) and (let == fasta_letters(core, fasta_columns(core, snps)[0])[r0:]).all()
    return res


SHAPES = [(3, 9), (1, 1), (2, 1), (5, 16), (1, 17), (7, 8191), (4, 8192), (4, 8193), (2, 70001), (33, 1024 * 3 + 1),
          (130, 8192 * 2 + 5), (300, 2049), (600, 70001), (1100, 8193)]


@pytest.mark.parametrize("N,L", SHAPES)
def test_bytes_match_numpy(N, L, tmp_path):
    rng = np.random.default_rng(N * 7919 + L)
    anc = (1 << rng.integers(0, 4, L)).astype(np.uint8)
    with _sim(N, L) as sim:
        sim.set_initial(anc, np.zeros(30, np.uint8))
        res = check_against_reference(sim, np.tile(anc, (N, 1)), tmp_path)     # clonal: no column in SNP mode
        assert res.columns == 0 and open(str(tmp_path / "a1.fasta"), "rb").read() == b"".join(b">ind_%d\n\n" % i for i in range(N))
        core = forced_state(rng, N, L, anc)
        sim.upload(core)
        res = check_against_reference(sim, core, tmp_path)
        # cross-checks with the other readers of the state
        assert res.columns == sim.core_diversity().segregating
        counts = sim.core_allele_counts().astype(np.int64)
        const = (counts > 0).sum(axis=1) == 1
        assert res.const_counts.tolist() == np.bincount(counts[const].argmax(axis=1), minlength=4).tolist()
        csv = sim.export_core_csv(0, N).replace(b",", b"").split(b"\n")[:-1]
        assert sim.write_core_fasta(str(tmp_path / "w.fasta")).columns == L
        whole = open(str(tmp_path / "w.fasta"), "rb").read().split(b"\n")[:-1]
        assert whole[1::2] == csv and whole[0::2] == [b">ind_%d" % i for i in range(N)]


def _evolved(N, L, n_gen, seed, **kw):
    p = pb.Params(pop_size=N, core_size=L, pan_genes=300, core_genes=100, n_gen=n_gen, seed=seed, **kw)
    d = pb.derive(p)
    rng = np.random.default_rng(seed)
    core_row = (1 << rng.integers(0, 4, L)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.3).astype(np.uint8)
    return p, core_row, acc_row, rng.normal(0, 0.05, d.pan_size)


def test_evolved_hr_state_is_materialised_before_writing(tmp_path):
    p, core_row, acc_row, sel = _evolved(150, 8192 * 4 + 999, 4, 11, HR_rate=0.5, core_mu=0.01, prop_positive=0.1,
                                         competition_strength=0.4)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        for g in range(p.n_gen):
            sim.step(g)                                 # recombination stays deferred
        path = str(tmp_path / "e.fasta")
        sim.write_core_fasta(path, snps_only=True)      # the FASTA first: it must materialise
        core = sim.download_core()
        assert open(path, "rb").read() == fasta_text(core, True)[0]
        check_against_reference(sim, core, tmp_path)


def test_sparse_state_has_few_columns(tmp_path):
    p, core_row, acc_row, sel = _evolved(500, 200_003, 20, 3, core_mu=1e-6)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        sim.run_generations(0, p.n_gen)
        core = sim.download_core()
        res = check_against_reference(sim, core, tmp_path)
        assert 0 < res.columns < p.core_size // 50
        assert res.columns == sim.core_diversity().segregating


def _bounds(L, n, i):
    import ctypes as C
    b, e = C.c_uint64(), C.c_uint64()
    assert pb._ffi.lib().pansim_shard_bounds(L, n, i, C.byref(b), C.byref(e)) == 0
    return b.value, e.value


def test_shards_and_groups_write_the_whole_file(tmp_path):
    import torch
    p, core_row, acc_row, sel = _evolved(90, 8192 * 5 + 321, 4, 6, HR_rate=0.5, core_mu=0.01, prop_positive=0.1,
                                         competition_strength=0.3)
    want = {}
    with pb.Pansim.from_params(p) as whole:
        whole.set_initial(core_row, acc_row)
        whole.set_selection(sel)
        whole.run_generations(0, p.n_gen)
        for snps in (False, True):
            path = str(tmp_path / f"whole{int(snps)}.fasta")
            want[snps] = (whole.write_core_fasta(path, snps_only=snps), open(path, "rb").read())
        core = whole.download_core()
    assert want[True][1] == fasta_text(core, True)[0] and 0 < want[True][0].columns < p.core_size
    for n in (2, 3):
        parts = {False: [], True: []}
        for i in range(n):
            b, e = _bounds(p.core_size, n, i)
            assert 0 < e - b < p.core_size
            with pb.Pansim.from_params(p, site_begin=b, site_end=e) as s:
                s.set_initial(core_row, acc_row)
                s.set_selection(sel)
                s.run_generations(0, p.n_gen)
                for snps in (False, True):
                    res = s.write_core_fasta(str(tmp_path / f"shard{i}.fasta"), snps_only=snps)
                    let = s.export_core_fasta_rows(0, p.pop_size, snps_only=snps)
                    assert let.shape == (p.pop_size, res.columns)
                    parts[snps].append((res, let))
        for snps in (False, True):
            let = np.concatenate([x[1] for x in parts[snps]], axis=1)
            text = b"".join(b">ind_%d\n" % r + let[r].tobytes() + b"\n" for r in range(p.pop_size))
            assert text == want[snps][1], (n, snps)
            assert sum(x[0].columns for x in parts[snps]) == want[snps][0].columns
            assert (sum(x[0].const_counts for x in parts[snps]) == want[snps][0].const_counts).all()
    for n_dev in (1, 2, 3):
        if n_dev > torch.cuda.device_count():
            continue
        with pb.PansimGroup(p, n_dev) as g:
            g.set_initial(core_row, acc_row)
            g.set_selection(sel)
            g.run_generations(0, p.n_gen)
            for snps in (False, True):
                path = str(tmp_path / f"group{n_dev}_{int(snps)}.fasta")
                res = g.write_core_fasta(path, snps_only=snps)
                assert open(path, "rb").read() == want[snps][1], (n_dev, snps)
                assert res.bytes == len(want[snps][1]) and res.columns == want[snps][0].columns
                assert (res.const_counts == want[snps][0].const_counts).all()


def _gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif(_gpus() < 2, reason="needs two GPUs")
def test_group_fasta_as_the_first_text_export(tmp_path):
    """Every shard's staging chunks are made by the FASTA writer itself, on the shard's own device: no CSV or VCF
    export has sized them before."""
    p, core_row, acc_row, sel = _evolved(64, 8192 * 3 + 77, 3, 8, HR_rate=0.5, core_mu=0.01)
    want = {}
    with pb.Pansim.from_params(p) as whole:
        whole.set_initial(core_row, acc_row)
        whole.set_selection(sel)
        whole.run_generations(0, p.n_gen)
        for snps in (False, True):
            path = str(tmp_path / f"whole{int(snps)}.fasta")
            whole.write_core_fasta(path, snps_only=snps)
            want[snps] = open(path, "rb").read()
    for n_dev in range(2, min(_gpus(), 3) + 1):
        for snps in (True, False):
            with pb.PansimGroup(p, n_dev) as g:
                g.set_initial(core_row, acc_row)
                g.set_selection(sel)
                g.run_generations(0, p.n_gen)
                path = str(tmp_path / f"group{n_dev}_{int(snps)}.fasta")
                assert g.write_core_fasta(path, snps_only=snps).bytes == len(want[snps])
                assert open(path, "rb").read() == want[snps], (n_dev, snps)


def test_errors(tmp_path):
    N, L = 6, 300
    rng = np.random.default_rng(2)
    with _sim(N, L) as sim:
        path = str(tmp_path / "x.fasta")
        for snps in (False, True):
            with pytest.raises(pb.PansimError) as e:
                sim.write_core_fasta(path, snps_only=snps)     # no state at all
            assert e.value.code == -5
        with pytest.raises(pb.PansimError) as e:
            sim.export_core_fasta_rows(0, N)
        assert e.value.code == -5
        core = (1 << rng.integers(0, 4, (N, L))).astype(np.uint8)
        sim.upload(core, np.zeros((N, 30), np.uint8))       # no ancestral row: not needed
        assert sim.write_core_fasta(path).bytes == len(fasta_text(core, False)[0])
        with pytest.raises(pb.PansimError) as e:
            sim.write_core_fasta(str(tmp_path / "no_such_dir" / "x.fasta"))
        assert e.value.code == -1
        for r0, r1 in ((0, N + 1), (4, 3), (N + 1, N + 2)):
            with pytest.raises(pb.PansimError) as e:
                sim.export_core_fasta_rows(r0, r1)
            assert e.value.code == -1
        if os.path.exists("/dev/full"):
            with pytest.raises(pb.PansimError):
                sim.write_core_fasta("/dev/full", snps_only=True)
        check_against_reference(sim, core, tmp_path)         # the context still works after refused calls
    p = pb.Params(pop_size=N, core_size=8192 * 3, pan_genes=40, core_genes=10)
    big = (1 << rng.integers(0, 4, (N, p.core_size))).astype(np.uint8)
    with pb.Pansim.from_params(p) as sim:
        sim.upload(big, np.zeros((N, 30), np.uint8))
        if os.path.exists("/dev/full"):
            with pytest.raises(pb.PansimError):             # large enough to fail inside the chunk stream
                sim.write_core_fasta("/dev/full")
        assert sim.write_core_fasta(str(tmp_path / "b.fasta")).bytes == os.path.getsize(str(tmp_path / "b.fasta"))


CLI_COMMON = ["--pop_size", "40", "--core_size", "8300", "--pan_genes", "90", "--core_genes", "30", "--n_gen", "5",
              "--max_distances", "60", "--HR_rate", "0.5", "--core_mu", "0.01", "--competition_strength", "0.3",
              "--prop_positive", "0.2", "--seed", "9", "--print_dist", "--print_matrices", "--print_diversity",
              "--print_vcf", "--print_genealogy"]
OTHER_FILES = (".tsv", "_per_gen.tsv", "_freqs.txt", "_diversity.tsv", "_core_sfs.txt", "_core_genome.csv",
               "_pangenome.csv", "_core_genome.vcf", "_genealogy.nwk", "_tmrca.tsv")
NEW_FILES = ("_core_genome.fasta", "_core_snps.fasta", "_core_snps_fconst.txt")


def _records(path):
    lines = open(path, "rb").read().split(b"\n")
    assert lines[-1] == b""
    return [x.decode() for x in lines[0:-1:2]], lines[1:-1:2]


def _check_cli(run, tmp_path, tag):
    plain, fa = str(tmp_path / f"{tag}_plain"), str(tmp_path / f"{tag}_fa")
    run(*CLI_COMMON, "--outpref", plain)
    run(*CLI_COMMON, "--print_fasta", "--print_snp_alignment", "--outpref", fa)
    for suffix in NEW_FILES:
        assert not os.path.exists(plain + suffix)
    for suffix in OTHER_FILES:
        assert open(plain + suffix, "rb").read() == open(fa + suffix, "rb").read(), suffix
    rows = [r.replace(",", "").encode() for r in open(fa + "_core_genome.csv").read().splitlines()]
    names, seqs = _records(fa + "_core_genome.fasta")
    assert seqs == rows
    assert names == [">ind_%d" % i for i in range(40)]
    assert sorted(n[1:] for n in names) == sorted(re.findall(r"ind_\d+", open(fa + "_genealogy.nwk").read()))
    vcf_samples = [l for l in open(fa + "_core_genome.vcf").read().splitlines() if l.startswith("#CHROM")][0].split("\t")[9:]
    assert [n[1:] for n in names] == vcf_samples
    letters = np.array([list(r.decode()) for r in rows])                      # [N, L]
    poly = np.array([len(set(letters[:, s])) >= 2 for s in range(letters.shape[1])])
    snp_names, snp_seqs = _records(fa + "_core_snps.fasta")
    assert snp_names == names and snp_seqs == ["".join(r).encode() for r in letters[:, poly]]
    consts = [int((letters[0, ~poly] == ch).sum()) for ch in "ACGT"]
    assert open(fa + "_core_snps_fconst.txt").read() == ",".join(map(str, consts)) + "\n"
    assert sum(consts) + int(poly.sum()) == 8300 and 0 < poly.sum() < 8300
    div = [int(x.split("\t")[0]) for x in open(fa + "_diversity.tsv").read().splitlines()]
    assert poly.sum() == div[-1]
    return fa


def test_python_cli_print_fasta(tmp_path):
    def run(*args):
        r = subprocess.run([sys.executable, "-m", "pansim_b200", *args], cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    _check_cli(run, tmp_path, "py")


def test_cpp_cli_print_fasta(tmp_path):
    binary = os.path.join(ROOT, "pansim_b200", "pansim")
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)

    def run(*args):
        r = subprocess.run([binary, *args], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    fa = _check_cli(run, tmp_path, "cpp")
    import torch
    if torch.cuda.device_count() >= 2:
        two = str(tmp_path / "cpp_two")
        run(*CLI_COMMON, "--print_fasta", "--print_snp_alignment", "--gpus", "2", "--outpref", two)
        for suffix in NEW_FILES:
            assert open(two + suffix, "rb").read() == open(fa + suffix, "rb").read(), suffix
        # the FASTA files as the only text outputs: no CSV or VCF export sizes the shards' staging first
        only = str(tmp_path / "cpp_two_only")
        run(*[a for a in CLI_COMMON if a not in ("--print_matrices", "--print_vcf")], "--print_fasta",
            "--print_snp_alignment", "--gpus", "2", "--outpref", only)
        for suffix in NEW_FILES:
            assert open(only + suffix, "rb").read() == open(fa + suffix, "rb").read(), suffix
