"""Core-genome VCF written on the device: byte-for-byte equality with a numpy formatter of download_core() and
the ancestral row, the deferred recombination materialised before reading, the tie to the independent SFS
path, column shards and groups, errors, and --print_vcf in both command lines."""
import os
import subprocess
import sys

import numpy as np
import pytest

import pansim_b200 as pb

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CODES = np.array([1, 2, 4, 8], np.uint8)
LETTERS = "ACGT"


def vcf_header(L, N):
    return ("##fileformat=VCFv4.2\n##source=pansim_b200\n" f"##contig=<ID=core,length={L}>\n"
            '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n'
            "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT" + "".join(f"\tind_{i}" for i in range(N)) + "\n").encode()


def np_vcf_body(core, anc, site_begin=0):
    """The VCF lines of one-hot rows core [N, Ll] against the ancestral one-hot row anc [Ll]."""
    N, Ll = core.shape
    codes = np.searchsorted(CODES, core).astype(np.int64)                  # [N, Ll] in 0..3
    ref = np.searchsorted(CODES, anc).astype(np.int64)                     # [Ll]
    present = np.stack([(codes == a).any(axis=0) for a in range(4)], axis=1)   # [Ll, 4]
    is_ref = np.arange(4)[None, :] == ref[:, None]
    alt = present & ~is_ref
    digit = np.where(is_ref, 0, np.cumsum(alt, axis=1) - alt + 1)          # genotype of each letter
    written = np.flatnonzero(alt.any(axis=1))
    out = []
    for s0 in range(0, len(written), 4096):
        ws = written[s0:s0 + 4096]
        gt = digit[ws[:, None], codes[:, ws].T] + ord("0")                 # [sites, N]
        span = np.empty((len(ws), 2 * N), np.uint8)
        span[:, 0::2] = ord("\t")
        span[:, 1::2] = gt
        for k, s in enumerate(ws):
            alts = ",".join(LETTERS[a] for a in range(4) if alt[s, a])
            out.append(f"core\t{site_begin + s + 1}\t.\t{LETTERS[ref[s]]}\t{alts}\t.\t.\t.\tGT".encode()
                       + span[k].tobytes() + b"\n")
    return b"".join(out)


def parse_body(body, N):
    """(positions, REF letters, ALT lists, genotype digits [lines, N] uint8) of a VCF body."""
    if not body:
        return np.zeros(0, np.int64), [], [], np.zeros((0, N), np.uint8)
    buf = np.frombuffer(body, np.uint8)
    nl = np.flatnonzero(buf == ord("\n"))
    idx = nl[:, None] - 2 * N + 1 + 2 * np.arange(N)[None, :]
    gt = (buf[idx] - ord("0")).astype(np.uint8)
    assert (buf[idx - 1] == ord("\t")).all()
    starts = np.concatenate([[0], nl[:-1] + 1])
    pos, refs, alts = [], [], []
    for a, e in zip(starts, nl - 2 * N):
        f = body[a:e].split(b"\t")
        assert f[0] == b"core" and f[2] == b"." and f[5:9] == [b".", b".", b".", b"GT"], f
        pos.append(int(f[1]))
        refs.append(f[3].decode())
        alts.append(f[4].decode().split(","))
    return np.array(pos, np.int64), refs, alts, gt


def _sim(N, L, **kw):
    return pb.Pansim.from_params(pb.Params(pop_size=N, core_size=L, pan_genes=40, core_genes=10, HR_rate=0.0,
                                           HGT_rate=0.0, **kw))


def forced_state(rng, N, L, anc):
    """Random rows with columns forced on purpose: all REF, fixed for another letter, and exactly 2, 3 and 4
    letters with and without REF present."""
    core = (1 << rng.integers(0, 4, (N, L))).astype(np.uint8)
    code = np.searchsorted(CODES, anc)

    def others(s, k):
        return [int(CODES[(code[s] + 1 + i) % 4]) for i in range(k)]

    def force(col, letters):
        s = col % L
        core[:, s] = np.array(letters, np.uint8)[np.arange(N) % len(letters)]

    force(0, [anc[0]])                                  # every row REF: not written
    force(1, others(1, 1))                              # fixed for another letter: ALT of one letter, all 1
    force(2, [anc[2 % L]] + others(2, 1))               # 2 letters with REF
    force(3, others(3, 2))                              # 2 letters without REF
    force(4, [anc[4 % L]] + others(4, 2))               # 3 letters with REF
    force(5, others(5, 3))                              # 3 letters without REF
    force(6, [anc[6 % L]] + others(6, 3))               # all 4 letters
    core[:, 7::5] = anc[7::5]                           # more sites that are not written
    return core


SHAPES = [(3, 9), (7, 8191), (4, 8193), (2, 70001), (1, 17), (5, 16), (33, 1024 * 3 + 1), (130, 8192 * 2 + 5),
          (300, 2049), (600, 70001)]


@pytest.mark.parametrize("N,L", SHAPES)
def test_bytes_match_numpy(N, L, tmp_path):
    rng = np.random.default_rng(N * 7919 + L)
    anc = (1 << rng.integers(0, 4, L)).astype(np.uint8)
    path = str(tmp_path / "a.vcf")
    with _sim(N, L) as sim:
        sim.set_initial(anc, np.zeros(30, np.uint8))
        n = sim.write_core_vcf(path)
        assert open(path, "rb").read() == vcf_header(L, N) and n == len(vcf_header(L, N))     # clonal: no line
        core = forced_state(rng, N, L, anc)
        sim.upload(core)
        want = np_vcf_body(core, anc)
        n = sim.write_core_vcf(path)
        got = open(path, "rb").read()
        assert n == len(got)
        assert got == vcf_header(L, N) + want
        assert sim.write_core_vcf(path, header=False) == len(want)
        assert open(path, "rb").read() == want
        # line lengths: 19 + digits(POS) + 2 |ALT| + 2 N
        pos, refs, alts, gt = parse_body(want, N)
        assert sum(19 + len(str(p)) + 2 * len(a) + 2 * N for p, a in zip(pos, alts)) == len(want)


def test_evolved_state_is_materialised_before_writing(tmp_path):
    p = pb.Params(pop_size=150, core_size=8192 * 4 + 999, pan_genes=300, core_genes=100, n_gen=4, HR_rate=0.5,
                  core_mu=0.01, prop_positive=0.1, competition_strength=0.4, seed=11)
    d = pb.derive(p)
    rng = np.random.default_rng(11)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.3).astype(np.uint8)
    path = str(tmp_path / "e.vcf")
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(rng.normal(0, 0.05, d.pan_size))
        for g in range(p.n_gen):
            sim.step(g)                                 # recombination stays deferred
        sim.write_core_vcf(path)                        # the VCF first: it must materialise
        core = sim.download_core()
    assert open(path, "rb").read() == vcf_header(p.core_size, p.pop_size) + np_vcf_body(core, core_row)


def test_lines_and_genotypes_match_the_sfs(tmp_path):
    N, L, n_gen = 1000, 100_003, 5
    p = pb.Params(pop_size=N, core_size=L, pan_genes=300, core_genes=100, n_gen=n_gen, seed=4)
    d = pb.derive(p)
    rng = np.random.default_rng(4)
    core_row = (1 << rng.integers(0, 4, L)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.3).astype(np.uint8)
    path = str(tmp_path / "s.vcf")
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(np.zeros(d.pan_size))
        sim.run_generations(0, n_gen)
        n = sim.write_core_vcf(path, header=False)
        _, sfs = sim.core_diversity(sfs=True)
    body = open(path, "rb").read()
    assert n == len(body) > 100_000_000
    buf = np.frombuffer(body, np.uint8)
    nl = np.flatnonzero(buf == ord("\n"))
    assert len(nl) == L - int(sfs[0])
    hist = np.zeros(N + 1, np.int64)
    for a in range(0, len(nl), 8192):
        idx = nl[a:a + 8192, None] - 2 * N + 1 + 2 * np.arange(N)[None, :]
        hist += np.bincount((buf[idx] != ord("0")).sum(axis=1), minlength=N + 1)
    assert hist[0] == 0 and (hist[1:] == sfs[1:].astype(np.int64)).all()


def _shard_case():
    p = pb.Params(pop_size=90, core_size=8192 * 5 + 321, pan_genes=300, core_genes=100, n_gen=4, HR_rate=0.5,
                  core_mu=0.01, seed=6, prop_positive=0.1, competition_strength=0.3)
    d = pb.derive(p)
    rng = np.random.default_rng(6)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.25).astype(np.uint8)
    sel = rng.normal(0, 0.05, d.pan_size)
    return p, core_row, acc_row, sel


def _bounds(L, n, i):
    import ctypes as C
    b, e = C.c_uint64(), C.c_uint64()
    assert pb._ffi.lib().pansim_shard_bounds(L, n, i, C.byref(b), C.byref(e)) == 0
    return b.value, e.value


def test_shards_and_groups_write_the_whole_file(tmp_path):
    import torch
    p, core_row, acc_row, sel = _shard_case()
    whole_path, body_path = str(tmp_path / "whole.vcf"), str(tmp_path / "whole_body.vcf")
    with pb.Pansim.from_params(p) as whole:
        whole.set_initial(core_row, acc_row)
        whole.set_selection(sel)
        whole.run_generations(0, p.n_gen)
        whole.write_core_vcf(whole_path)
        whole.write_core_vcf(body_path, header=False)
        want = np_vcf_body(whole.download_core(), core_row)
    assert open(body_path, "rb").read() == want and len(want) > 0
    parts = []
    for i in range(2):
        b, e = _bounds(p.core_size, 2, i)
        assert 0 < e - b < p.core_size
        with pb.Pansim.from_params(p, site_begin=b, site_end=e) as s:
            s.set_initial(core_row, acc_row)
            s.set_selection(sel)
            s.run_generations(0, p.n_gen)
            path = str(tmp_path / f"shard{i}.vcf")
            s.write_core_vcf(path, header=False)
            parts.append(open(path, "rb").read())
    assert parts[0] + parts[1] == want
    for n_dev in (1, 2):
        if n_dev > torch.cuda.device_count():
            continue
        path = str(tmp_path / f"group{n_dev}.vcf")
        with pb.PansimGroup(p, n_dev) as g:
            g.set_initial(core_row, acc_row)
            g.set_selection(sel)
            g.run_generations(0, p.n_gen)
            n = g.write_core_vcf(path)
        assert open(path, "rb").read() == open(whole_path, "rb").read() and n == os.path.getsize(whole_path)


def test_errors(tmp_path):
    N, L = 6, 300
    rng = np.random.default_rng(2)
    with _sim(N, L) as sim:
        path = str(tmp_path / "x.vcf")
        with pytest.raises(pb.PansimError) as e:
            sim.write_core_vcf(path)                    # no state at all
        assert e.value.code == -5
        core = (1 << rng.integers(0, 4, (N, L))).astype(np.uint8)
        sim.upload(core, np.zeros((N, 30), np.uint8))
        with pytest.raises(pb.PansimError) as e:
            sim.write_core_vcf(path)                    # uploads give no ancestral row
        assert e.value.code == -5
        sim.set_initial(core[0], np.zeros(30, np.uint8))
        sim.upload(core)
        if os.path.exists("/dev/full"):
            with pytest.raises(pb.PansimError):
                sim.write_core_vcf("/dev/full")
        assert sim.write_core_vcf(path) == os.path.getsize(path)   # the context still works after a failed write
    p = pb.Params(pop_size=N, core_size=8192 * 3, pan_genes=40, core_genes=10)
    big = 1 << rng.integers(0, 4, (N, p.core_size))
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(big[0].astype(np.uint8), np.zeros(30, np.uint8))
        sim.upload(big.astype(np.uint8))
        if os.path.exists("/dev/full"):
            with pytest.raises(pb.PansimError):         # large enough to fail inside the chunk stream
                sim.write_core_vcf("/dev/full", header=False)


CLI_COMMON = ["--pop_size", "40", "--core_size", "8300", "--pan_genes", "90", "--core_genes", "30", "--n_gen", "5",
              "--max_distances", "60", "--HR_rate", "0.5", "--core_mu", "0.01", "--competition_strength", "0.3",
              "--prop_positive", "0.2", "--seed", "9"]
OTHER_FILES = (".tsv", "_per_gen.tsv", "_freqs.txt", "_diversity.tsv", "_core_sfs.txt", "_core_genome.csv", "_pangenome.csv")


def _check_cli(run, tmp_path, tag):
    plain, vcf = str(tmp_path / f"{tag}_plain"), str(tmp_path / f"{tag}_vcf")
    run(*CLI_COMMON, "--print_dist", "--print_matrices", "--print_diversity", "--outpref", plain)
    run(*CLI_COMMON, "--print_dist", "--print_matrices", "--print_diversity", "--print_vcf", "--outpref", vcf)
    assert not os.path.exists(plain + "_core_genome.vcf")
    for suffix in OTHER_FILES:
        assert open(plain + suffix, "rb").read() == open(vcf + suffix, "rb").read(), suffix
    text = open(vcf + "_core_genome.vcf", "rb").read()
    head = vcf_header(8300, 40)
    assert text.startswith(head)
    pos, refs, alts, gt = parse_body(text[len(head):], 40)
    letters = np.array([l.split(",") for l in open(vcf + "_core_genome.csv").read().splitlines()])   # [N, L]
    assert (np.diff(pos) > 0).all()
    for k, s in enumerate(pos - 1):
        table = np.array([refs[k]] + alts[k])
        assert (table[gt[k]] == letters[:, s]).all()
    sfs = np.array([int(x) for x in open(vcf + "_core_sfs.txt").read().splitlines()])
    assert len(pos) == 8300 - sfs[0]
    hist = np.bincount((gt != 0).sum(axis=1), minlength=41)
    assert hist[0] == 0 and (hist[1:] == sfs[1:]).all()
    # sites left out are those where every row carries the ancestral letter
    unwritten = np.setdiff1d(np.arange(8300), pos - 1)
    assert all(len(set(letters[:, s])) == 1 for s in unwritten[:200])
    return vcf


def test_python_cli_print_vcf(tmp_path):
    def run(*args):
        r = subprocess.run([sys.executable, "-m", "pansim_b200", *args], cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    _check_cli(run, tmp_path, "py")


def test_cpp_cli_print_vcf(tmp_path):
    binary = os.path.join(ROOT, "pansim_b200", "pansim")
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)

    def run(*args):
        r = subprocess.run([binary, *args], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    vcf = _check_cli(run, tmp_path, "cpp")
    import torch
    if torch.cuda.device_count() >= 2:
        two = str(tmp_path / "cpp_two")
        run(*CLI_COMMON, "--print_dist", "--print_matrices", "--print_diversity", "--print_vcf", "--gpus", "2",
            "--outpref", two)
        assert open(two + "_core_genome.vcf", "rb").read() == open(vcf + "_core_genome.vcf", "rb").read()
