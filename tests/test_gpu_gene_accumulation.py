"""Pangenome accumulation on the device: the orders, the four curves, the gene frequency spectrum and the gene classes
equal, exactly, a numpy reference (uploaded, crafted and evolved states, with and without core genes); the global-memory
order draw; repeated calls reuse their buffers; NULL outputs; groups equal the single context; errors leave the
context working; --print_gene_accumulation in both command lines."""
import dataclasses
import os
import subprocess
import sys

import numpy as np
import pytest

import pansim_b200 as pb

from gene_accumulation_reference import np_classes, np_curves, np_orders, np_spectrum

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cfg(N, G, c0):
    """A context of N rows, G accessory genes and c0 core genes (one gene compartment)."""
    cfg = pb.make_config(pb.Params(pop_size=N, core_size=64, pan_genes=G + 10, core_genes=10, HR_rate=0.0, HGT_rate=0.0,
                                   prop_genes2=0.0))
    cfg.core_genes = c0
    return cfg


def _upload(sim, pres):
    sim.upload(acc=np.asarray(pres, np.uint8).reshape(sim.N, sim.G))


def assert_matches(sim, pres, n_perms, seed, c0):
    got = sim.gene_accumulation(n_perms, seed)
    orders = np_orders(seed, n_perms, sim.N)
    assert got.orders.dtype == np.uint32 and got.orders.shape == (n_perms, sim.N)
    assert np.array_equal(got.orders, orders)
    for name, want in zip(("pan", "core", "new", "unique"), np_curves(pres, orders, c0)):
        assert np.array_equal(getattr(got, name), want), name
    assert (np.cumsum(got.new.astype(np.int64), axis=1) == got.pan).all()
    return got


def assert_spectrum(sim, pres, c0):
    spec = sim.gene_spectrum()
    want = np_spectrum(pres, c0)
    assert spec.dtype == np.uint64 and np.array_equal(spec, want)
    assert pb.pangenome_classes(spec, sim.N) == np_classes(want, sim.N)


def random_presence(rng, N, G):
    """Random presence at a spread of gene frequencies, with genes present everywhere, absent everywhere and in one row."""
    pres = rng.random((N, G)) < rng.random(G)[None, :] ** 2
    pres[:, 0::11] = True
    pres[:, 1::13] = False
    for g in range(2, G, 17):
        pres[:, g] = False
        pres[rng.integers(0, N), g] = True
    return pres


@pytest.mark.parametrize("G", [0, 1, 31, 32, 33, 4000])
@pytest.mark.parametrize("N", [1, 2, 31, 32, 33, 1000, 1100])
def test_uploaded_states_match_numpy(N, G):
    rng = np.random.default_rng(N * 7919 + G)
    pres = random_presence(rng, N, G)
    for c0 in (0, 13):
        with pb.Pansim(_cfg(N, G, c0)) as sim:
            _upload(sim, pres)
            for n_perms, seed in ((1, 0), (7, 0xDEADBEEF_12345678), (100, 2 ** 64 - 1 - N)):
                assert_matches(sim, pres, n_perms, seed, c0)
            assert_spectrum(sim, pres, c0)


@pytest.mark.parametrize("G", [4097, 9000])
def test_several_word_slices_match_numpy(G):
    # 129 and 282 words: two and three slices of 128 words adding into the same per-step counts, with several row
    # chunks at one order and at 100 orders for G = 4 097, one chunk at 100 orders for G = 9 000
    N = 1100
    pres = random_presence(np.random.default_rng(G), N, G)
    with pb.Pansim(_cfg(N, G, 11)) as sim:
        _upload(sim, pres)
        for n_perms, seed in ((1, 5), (100, 6)):
            assert_matches(sim, pres, n_perms, seed, 11)
        assert_spectrum(sim, pres, 11)


def test_seed_keys_the_orders():
    N, G = 200, 300
    pres = random_presence(np.random.default_rng(1), N, G)
    with pb.Pansim(_cfg(N, G, 4)) as sim:
        _upload(sim, pres)
        a = sim.gene_accumulation(20, 11)
        assert np.array_equal(sim.gene_accumulation(20, 11).orders, a.orders)
        b = sim.gene_accumulation(20, 12)
        assert not np.array_equal(a.orders, b.orders)
        assert (a.orders[0] != a.orders[1]).any()                    # orders differ from each other
        assert all(sorted(o.tolist()) == list(range(N)) for o in b.orders)
        # the orders are a pure function of (seed, p): fewer orders are a prefix
        assert np.array_equal(sim.gene_accumulation(5, 11).orders, a.orders[:5])
        # None is the context's seed
        assert np.array_equal(sim.gene_accumulation(3).orders, np_orders(sim.cfg.seed, 3, N))


def test_global_memory_order_draw():
    # 8 N bytes do not fit in a CTA's shared memory: the orders are drawn in global memory, the same permutations
    N, G, c0 = 30000, 40, 2
    rng = np.random.default_rng(3)
    pres = rng.random((N, G)) < 0.01
    with pb.Pansim(_cfg(N, G, c0)) as sim:
        _upload(sim, pres)
        assert_matches(sim, pres, 3, 99, c0)


def test_crafted_matrices():
    N, G, c0 = 70, 70, 5
    with pb.Pansim(_cfg(N, G, c0)) as sim:
        _upload(sim, np.ones((N, G), bool))
        got = sim.gene_accumulation(9, 1)
        assert (got.pan == G + c0).all() and (got.core == G + c0).all()
        assert (got.new[:, 0] == G + c0).all() and (got.new[:, 1:] == 0).all()
        assert (got.unique[:, 0] == G + c0).all() and (got.unique[:, 1:] == 0).all()
        assert sim.gene_spectrum().tolist() == [0] * N + [G + c0]

        _upload(sim, np.zeros((N, G), bool))
        got = sim.gene_accumulation(9, 1)
        assert (got.pan == c0).all() and (got.core == c0).all() and (got.unique[:, 1:] == 0).all()
        assert sim.gene_spectrum().tolist() == [G] + [0] * (N - 1) + [c0]

        eye = np.eye(N, dtype=bool)                                  # every genome has one gene of its own
        _upload(sim, eye)
        got = assert_matches(sim, eye, 9, 1, c0)
        k = np.arange(1, N + 1)
        assert (got.pan == c0 + k).all() and (got.new[:, 1:] == 1).all()
        assert (got.core[:, 0] == c0 + 1).all() and (got.core[:, 1:] == c0).all()
        assert (got.unique[:, 1:] == k[1:]).all()
        assert pb.pangenome_classes(sim.gene_spectrum(), N) == (c0, 0, 0, G, G + c0)

        one = np.zeros((N, G), bool)
        one[37, 41] = True                                           # a single gene in a single row
        _upload(sim, one)
        got = assert_matches(sim, one, 9, 1, c0)
        pos = np.argmax(got.orders == 37, axis=1)
        for p in range(9):
            assert got.new[p].tolist() == [c0 + (pos[p] == 0)] + [int(i == pos[p]) for i in range(1, N)]
            assert (got.pan[p] == c0 + (np.arange(N) >= pos[p])).all()
        assert_spectrum(sim, one, c0)


EVOLVED = {
    "neutral": dict(pop_size=300, pan_genes=1300, core_genes=100, n_gen=6),
    "selection": dict(pop_size=257, pan_genes=1130, core_genes=100, n_gen=6, prop_positive=0.2, competition_strength=0.4,
                      genome_size_penalty=0.9),
    "low_flip_hgt": dict(pop_size=400, pan_genes=2100, core_genes=100, n_gen=30, rate_genes1=1e-4, rate_genes2=1e-2,
                         HGT_rate=0.5),
}


def _evolved(kind, seed=3):
    p = pb.Params(core_size=8192, HR_rate=0.0, core_mu=0.001, seed=seed, **{"HGT_rate": 0.0, **EVOLVED[kind]})
    d = pb.derive(p)
    rng = np.random.default_rng(seed)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.5).astype(np.uint8)
    sel = rng.normal(0, 0.05, d.pan_size)
    return p, d, core_row, acc_row, sel


@pytest.mark.parametrize("kind", list(EVOLVED))
def test_evolved_states(kind):
    p, d, core_row, acc_row, sel = _evolved(kind)
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        sim.run_generations(0, p.n_gen - 1)
        sim.step(p.n_gen - 1)                            # the last accessory step, then the call
        pres = sim.download_acc().astype(bool)
        assert_matches(sim, pres, 50, 77, p.core_genes)
        assert_spectrum(sim, pres, p.core_genes)


def test_repeated_calls_reuse_buffers_and_null_outputs():
    p, d, core_row, acc_row, sel = _evolved("low_flip_hgt")
    with pb.Pansim.from_params(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        sim.run_generations(0, p.n_gen)
        pres = sim.download_acc().astype(bool)
        counts = sim.gene_counts()
        first = assert_matches(sim, pres, 100, 5, p.core_genes)
        for n_perms in (7, 200, 1, 100):
            got = assert_matches(sim, pres, n_perms, 5, p.core_genes)
            k = min(n_perms, 100)
            assert all(np.array_equal(getattr(got, f)[:k], getattr(first, f)[:k]) for f in first._fields)
        spec = sim.gene_spectrum()
        assert np.array_equal(sim.gene_spectrum(), spec) and (sim.gene_counts() == counts).all()
        # NULL outputs: each array alone, and none at all
        lib, N = sim._lib, sim.N
        for keep in range(5):
            outs = [np.zeros((100, N), np.uint32) if i == keep else None for i in range(5)]
            sim._check(lib.pansim_gene_accumulation(sim._h, 5, 100, *[pb.population._ptr(a) for a in outs]))
            assert np.array_equal(outs[keep], first[keep])
        sim._check(lib.pansim_gene_accumulation(sim._h, 5, 100, None, None, None, None, None))
        o_ms, a_ms, nbytes = sim.gene_accumulation_kernel_ms(100, 5, 3)
        assert o_ms > 0 and a_ms > 0 and nbytes == 100 * N * -(-sim.G // 32) * 4
        assert_matches(sim, pres, 100, 5, p.core_genes)


@pytest.mark.parametrize("n_dev", [1, 2])
def test_group_matches_single_context(n_dev):
    import torch
    if n_dev > torch.cuda.device_count():
        pytest.skip(f"needs {n_dev} GPUs")
    p, d, core_row, acc_row, sel = _evolved("low_flip_hgt")
    p = dataclasses.replace(p, core_size=8192 * 3)
    core_row = np.resize(core_row, p.core_size)
    with pb.Pansim.from_params(p) as whole:
        whole.set_initial(core_row, acc_row)
        whole.set_selection(sel)
        whole.run_generations(0, p.n_gen)
        want, want_spec = whole.gene_accumulation(33), whole.gene_spectrum()
    with pb.PansimGroup(p, n_dev) as g:
        g.set_initial(core_row, acc_row)
        g.set_selection(sel)
        g.run_generations(0, p.n_gen)
        got, spec = g.gene_accumulation(33), g.gene_spectrum()
    assert all(np.array_equal(getattr(got, f), getattr(want, f)) for f in want._fields)
    assert np.array_equal(spec, want_spec)


def test_errors_and_the_context_still_works():
    N, G, c0 = 50, 140, 3
    pres = random_presence(np.random.default_rng(2), N, G)
    with pb.Pansim(_cfg(N, G, c0)) as sim:
        for call in (lambda: sim.gene_accumulation(10, 1), sim.gene_spectrum):
            with pytest.raises(pb.PansimError) as e:
                call()                                   # no state
            assert e.value.code == -5
        _upload(sim, pres)                               # the accessory matrix alone is enough
        assert_matches(sim, pres, 10, 1, c0)
        for n_perms in (0, 10001, 2 ** 32 - 1):
            with pytest.raises(pb.PansimError) as e:
                sim.gene_accumulation(n_perms, 1)
            assert e.value.code == -1
            assert_matches(sim, pres, 10, 1, c0)
            assert_spectrum(sim, pres, c0)
        assert_matches(sim, pres, 10000, 1, c0)        # the largest n_perms


CLI_COMMON = ["--pop_size", "60", "--core_size", "9192", "--pan_genes", "700", "--core_genes", "30", "--n_gen", "12",
              "--max_distances", "60", "--HGT_rate", "0.3", "--rate_genes1", "0.001", "--rate_genes2", "0.05",
              "--competition_strength", "0.3", "--prop_positive", "0.2", "--seed", "9"]
OTHER_FILES = (".tsv", "_per_gen.tsv", "_freqs.txt", "_core_genome.csv", "_pangenome.csv", "_diversity.tsv")
CURVE_FILES = ("genes_in_pan_genome", "conserved_genes", "new_genes", "unique_genes")
ROARY_LABELS = ("Core genes\t(99% <= strains <= 100%)", "Soft core genes\t(95% <= strains < 99%)",
                "Shell genes\t(15% <= strains < 95%)", "Cloud genes\t(0% <= strains < 15%)",
                "Total genes\t(0% <= strains <= 100%)")


def _check_cli(run, tmp_path, tag, extra=()):
    plain, ga = str(tmp_path / f"{tag}_plain"), str(tmp_path / f"{tag}_ga")
    common = [*CLI_COMMON, *extra, "--print_dist", "--print_matrices", "--print_diversity"]
    run(*common, "--outpref", plain)
    run(*common, "--print_gene_accumulation", "--gene_accumulation_perms", "9", "--outpref", ga)
    assert not os.path.exists(plain + "_gene_spectrum.txt")
    for suffix in OTHER_FILES:
        assert open(plain + suffix, "rb").read() == open(ga + suffix, "rb").read(), suffix
    rows = [line.split(",")[30:] for line in open(ga + "_pangenome.csv").read().splitlines()]
    pres = np.array(rows, dtype=np.int64).astype(bool)
    curves = np_curves(pres, np_orders(9, 9, 60), 30)
    got = b""
    for name, want in zip(CURVE_FILES, curves):
        text = open(f"{ga}_number_of_{name}.Rtab", "rb").read()
        assert text == "".join("\t".join(str(int(x)) for x in row) + "\n" for row in want).encode(), name
        got += text
    spec = np_spectrum(pres, 30)
    assert spec[1:60].sum() > 0
    text = open(ga + "_gene_spectrum.txt", "rb").read()
    assert text == "".join(f"{int(x)}\n" for x in spec).encode()
    got += text
    text = open(ga + "_summary_statistics.txt", "rb").read()
    assert text == "".join(f"{label}\t{n}\n" for label, n in zip(ROARY_LABELS, np_classes(spec, 60))).encode()
    return got + text


def test_python_cli_print_gene_accumulation(tmp_path):
    def run(*args):
        r = subprocess.run([sys.executable, "-m", "pansim_b200", *args], cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    _check_cli(run, tmp_path, "py")


def test_cpp_cli_print_gene_accumulation(tmp_path):
    binary = os.path.join(ROOT, "pansim_b200", "pansim")
    subprocess.run(["make", "-C", os.path.join(ROOT, "pansim_b200", "host")], check=True, stdout=subprocess.DEVNULL)

    def run(*args):
        r = subprocess.run([binary, *args], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    one = _check_cli(run, tmp_path, "cpp")
    import torch
    if torch.cuda.device_count() >= 2:
        two = _check_cli(run, tmp_path, "cpp2", extra=("--gpus", "2"))
        assert two == one
