"""GPU parity tests: the CUDA path (through the C ABI) against the oracle on the
same inputs. Integer / byte / index results must be bit-exact; f64 results are
bit-exact where the summation order is reproduced, otherwise rtol is stated."""
import dataclasses

import numpy as np
import pytest

import pansim_b200 as pb
from oracle import binding as ob
from helpers import oracle_apply_gpu_events, random_state, sample_pairs, small_params

pytestmark = pytest.mark.gpu


def make(p, **kw):
    return pb.Pansim.from_params(p, **kw)


# ---------------------------------------------------------------- T: layout
@pytest.mark.parametrize("N,L,G", [(3, 9, 10), (5, 16, 32), (7, 8191, 33), (4, 8193, 1), (6, 20000, 4000),
                                   (2, 70001, 95)])
def test_upload_download_round_trip(N, L, G):
    rng = np.random.default_rng(N * L + G)
    core, acc = random_state(rng, N, L, G)
    p = pb.Params(pop_size=N, core_size=L, pan_genes=G + 5, core_genes=5)
    with make(p) as sim:
        sim.upload(core, acc)
        assert (sim.download_core() == core).all()
        assert (sim.download_acc() == acc).all()


def test_upload_rejects_non_onehot():
    p = pb.Params(pop_size=2, core_size=40, pan_genes=12, core_genes=2)
    core = np.ones((2, 40), np.uint8)
    core[1, 7] = 3
    with make(p) as sim:
        with pytest.raises(pb.PansimError) as e:
            sim.upload(core_onehot=core)
        assert e.value.code == -1


def test_set_initial_is_clonal():
    p = small_params()
    d = pb.derive(p)
    rng = np.random.default_rng(0)
    row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    arow = (rng.random(d.pan_size) < 0.25).astype(np.uint8)
    with make(p) as sim:
        sim.set_initial(row, arow)
        assert (sim.download_core() == row[None, :]).all()
        assert (sim.download_acc() == arow[None, :]).all()


def test_export_core_csv_matches_int_to_base():
    # population.rs:877-879, 154-162
    rng = np.random.default_rng(4)
    core, acc = random_state(rng, 5, 37, 8)
    p = pb.Params(pop_size=5, core_size=37, pan_genes=10, core_genes=2)
    with make(p) as sim:
        sim.upload(core, acc)
        txt = sim.export_core_csv(0, 5).decode()
    lut = {1: "A", 2: "C", 4: "G", 8: "T"}
    want = "".join(",".join(lut[int(x)] for x in row) + "\n" for row in core)
    assert txt == want


# ------------------------------------------------------------ D: distances
def test_KAT_H1_J1_through_cabi():
    r1 = np.array([1, 2, 4, 8, 1, 2, 4, 8, 1], np.uint8)
    r2 = np.array([1, 4, 4, 2, 8, 2, 4, 8, 2], np.uint8)
    x = np.array([1, 0, 1, 1, 0, 0, 1, 0, 1, 1], np.uint8)
    y = np.array([1, 1, 0, 1, 0, 0, 0, 0, 1, 0], np.uint8)
    p = pb.Params(pop_size=2, core_size=9, pan_genes=12, core_genes=2)
    with make(p) as sim:
        sim.upload(np.stack([r1, r2]), np.stack([x, y]))
        cd, it, un = sim.pair_counts([0], [1])
        assert (cd[0], it[0], un[0]) == (4, 3, 7)
        core_d, acc_d = sim.pairwise_distances([0, 1], [1, 0])
        assert core_d.tolist() == [0.4444444444444444] * 2
        assert acc_d.tolist() == [0.4444444444444444] * 2


@pytest.mark.parametrize("N,L,G,P", [(2, 1, 1, 4), (9, 100, 31, 200), (33, 8192, 64, 500), (17, 50001, 333, 400),
                                     (64, 300000, 4000, 1000)])
def test_pair_counts_match_oracle(N, L, G, P):
    rng = np.random.default_rng(L + G)
    core, acc = random_state(rng, N, L, G)
    # make some rows near-identical so small distances occur too
    core[1] = core[0]
    core[1, ::7] = 8
    r1, r2 = sample_pairs(rng, N, P)
    p = pb.Params(pop_size=N, core_size=L, pan_genes=G + 3, core_genes=3)
    with make(p) as sim:
        sim.upload(core, acc)
        cd, it, un = sim.pair_counts(r1, r2)
        core_d, acc_d = sim.pairwise_distances(r1, r2)
    ocore = ob.Population(core, True, 3)
    opan = ob.Population(acc, False, 3)
    assert (cd == ocore.pair_counts(r1, r2)).all()
    oi, ou = opan.pair_counts(r1, r2)
    assert (it == oi).all() and (un == ou).all()
    assert (core_d == ocore.pairwise_distances(r1, r2)).all()       # bit-exact f64
    assert (acc_d == opan.pairwise_distances(r1, r2)).all()


def test_pair_counts_self_and_repeated_pairs():
    rng = np.random.default_rng(8)
    core, acc = random_state(rng, 6, 1000, 40)
    p = pb.Params(pop_size=6, core_size=1000, pan_genes=40, core_genes=0)
    r1 = np.array([0, 0, 3, 3, 5], np.uint32)
    r2 = np.array([0, 1, 2, 2, 5], np.uint32)
    with make(p) as sim:
        sim.upload(core, acc)
        cd, it, un = sim.pair_counts(r1, r2)
    assert cd[0] == 0 and cd[4] == 0 and cd[2] == cd[3]
    assert it[0] == un[0] == acc[0].sum()


# ------------------------------------------------------------- Q: reductions
def test_gene_counts_and_frequencies():
    rng = np.random.default_rng(5)
    core, acc = random_state(rng, 37, 64, 1001)
    p = pb.Params(pop_size=37, core_size=64, pan_genes=1011, core_genes=10)
    with make(p) as sim:
        sim.upload(core, acc)
        opan = ob.Population(acc, False, 10)
        assert (sim.gene_counts() == opan.gene_counts()).all()
        assert (sim.gene_frequencies() == opan.gene_frequencies()).all()
        assert sim.calc_gene_freq() == opan.calc_gene_freq()


# ------------------------------------------------------------ G: gather
def test_next_generation_matches_oracle():
    rng = np.random.default_rng(6)
    N, L, G = 21, 25000, 130
    core, acc = random_state(rng, N, L, G)
    parents = rng.integers(0, N, N).astype(np.uint32)
    p = pb.Params(pop_size=N, core_size=L, pan_genes=G, core_genes=0)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.next_generation(parents)
        assert (sim.download_core() == core[parents]).all()
        assert (sim.download_acc() == acc[parents]).all()
        with pytest.raises(pb.PansimError):
            sim.next_generation(np.full(N, N, np.uint32))


# ---------------------------------------------------- F, C, W: selection
def test_fitness_and_average_distance_bit_exact():
    rng = np.random.default_rng(7)
    N, G = 80, 700
    core, acc = random_state(rng, N, 50, G, 0.25)
    acc[5] = acc[4]                       # identical rows -> small distances
    sel = rng.normal(0, 0.1, G)
    sel[3] = -1.0                          # lethal gene (population.rs:312-318)
    p = pb.Params(pop_size=N, core_size=50, pan_genes=G + 50, core_genes=50, competition_strength=0.7,
                  genome_size_penalty=0.98)
    d = pb.derive(p)
    opan = ob.Population(acc, False, 50)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.set_selection(sel)
        avg = sim.average_distance()
        assert (avg == opan.average_distance()).all()          # bit-exact (same f64 op order)
        sim.sample_indices(0)
        w, ng, lf = sim.weights()
    ow, ong, olf = opan.selection_weights(d.avg_gene_num, opan.average_distance(), sel, False, 0.98, 0.7)
    assert (ng == ong).all()
    assert (lf == olf).all()                                    # bit-exact column-order sum
    assert (lf[acc[:, 3] == 1] == 0.0).all()
    # softmax chain: CUDA libm exp/log differ from glibc by ulps -> rtol 1e-12
    np.testing.assert_allclose(w / w.sum(), ow / ow.sum(), rtol=1e-12)


@pytest.mark.parametrize("N,G,dens", [(200, 4000, 0.25), (131, 1030, 0.5), (65, 31, 0.3), (300, 33, 0.9), (2, 5, 0.5),
                                      (1100, 70, 0.5), (1024, 2100, 0.75)])
def test_competition_and_fitness_kernels_over_shapes(N, G, dens):
    """The intersection counts run on the tensor cores over 128 x 128 pair tiles (tcgen05, select.cuh
    K2a), the distances and the fitness sum as per-row sequential f64 chains fed from shared memory
    in rounds of 256 / 1024 values: shapes with several tiles, ragged last tiles,
    a ragged last word and fewer rows than one tile must all stay bit-exact. Parent selection has a
    register/shared-memory kernel up to 1024 individuals and a global-memory one above."""
    rng = np.random.default_rng(N + G)
    core, acc = random_state(rng, N, 20, G, dens)
    sel = rng.normal(0, 0.2, G).clip(-0.95, None)
    p = pb.Params(pop_size=N, core_size=20, pan_genes=G + 7, core_genes=7, competition_strength=1.0)
    opan = ob.Population(acc, False, 7)
    with make(p) as sim:
        sim.upload(core, acc)
        # neutral fast path first (all coefficients 0: popcounts only, log-fitness +0.0) ...
        sim.sample_indices(0, np.ones(N))
        _, ng0, lf0 = sim.weights()
        assert (ng0 == acc.sum(1)).all() and (lf0 == 0.0).all() and not np.signbit(lf0).any()
        # ... then the sequential chain
        sim.set_selection(sel)
        oavg = opan.average_distance()
        assert (sim.average_distance() == oavg).all()
        sim.sample_indices(1)
        w, ng, lf = sim.weights()
    ow, ong, olf = opan.selection_weights(pb.derive(p).avg_gene_num, oavg, sel, False, p.genome_size_penalty, 1.0)
    assert (ng == ong).all() and (lf == olf).all()
    np.testing.assert_allclose(w / w.sum(), ow / ow.sum(), rtol=1e-11)


@pytest.mark.parametrize("N,pan,cg,dens", [
    (300, 900, 200, 0.5), (130, 37, 0, 0.9), (1025, 4229, 100, 0.02), (257, 300, 0, 1.0), (5, 40, 37, 0.3),
    (1000, 6000, 2000, 0.25), (640, 12800, 0, 0.4),
    (2, 1, 0, 1.0), (128, 128, 0, 0.5), (129, 129, 0, 0.5), (384, 641, 1, 0.5),
    (200, 131072, 131000, 0.5), (300, 131100, 131000, 0.5)])
def test_competition_kernel_variants_are_bit_exact(N, pan, cg, dens):
    """The competition term gives the oracle's bits: intersection counts on tcgen05.mma with the operands expanded in
    the CTA, mean distances from the reciprocal-table quotient (tools/check_recip_division.c) while G + core_genes <=
    131072 and from the IEEE division above. Shapes: several 128-row tiles with a ragged last one, gene counts off the
    128-gene stage size, exactly one tile and one stage and one past each, more stages than the ring holds, fewer rows
    than a tile, no core genes (denominator 0 is not reachable here), the last shape of the table and the first past it."""
    rng = np.random.default_rng(N + pan)
    G = pan - cg
    core, acc = random_state(rng, N, 20, G, dens)
    p = pb.Params(pop_size=N, core_size=20, pan_genes=pan, core_genes=cg, competition_strength=0.5)
    oavg = ob.Population(acc, False, cg).average_distance()
    with make(p) as sim:
        sim.upload(core, acc)
        avg = sim.average_distance()
    assert np.array_equal(avg, oavg), (N, pan, cg, dens, int((avg != oavg).sum()))


def test_average_distance_identical_population_is_min_positive():
    p = pb.Params(pop_size=5, core_size=16, pan_genes=40, core_genes=8, competition_strength=1.0)
    with make(p) as sim:
        sim.upload(np.ones((5, 16), np.uint8), np.ones((5, 32), np.uint8))
        assert (sim.average_distance() == np.finfo(np.float64).tiny).all()


def test_parent_draws_follow_weights_and_are_reproducible():
    rng = np.random.default_rng(9)
    N, G = 40, 64
    core, acc = random_state(rng, N, 50, G, 0.5)
    sel = rng.normal(0, 0.3, G).clip(-0.9, None)
    p = pb.Params(pop_size=N, core_size=50, pan_genes=G, core_genes=0, seed=5)
    counts = np.zeros(N)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.set_selection(sel)
        first = sim.sample_indices(0)
        assert (sim.sample_indices(0) == first).all()          # counter-based: same key, same draw
        assert (sim.parents() == first).all()
        w, _, _ = sim.weights()
        n_gen = 400
        for g in range(n_gen):
            counts += np.bincount(sim.sample_indices(g), minlength=N)
    expected = w / w.sum() * N * n_gen
    chi2 = ((counts - expected) ** 2 / expected).sum()
    assert chi2 < 100          # 39 dof: mean 39, sd 8.8


def test_sample_indices_error_where_reference_panics():
    # WeightedIndex::new(...).unwrap() panics on NaN weights (population.rs:440)
    p = pb.Params(pop_size=4, core_size=16, pan_genes=8, core_genes=0, competition_strength=1.0)
    with make(p) as sim:
        sim.upload(np.ones((4, 16), np.uint8), np.ones((4, 8), np.uint8))
        with pytest.raises(pb.PansimError) as e:
            sim.sample_indices(0, np.array([1.0, -1.0, 1.0, 1.0]))     # ln(-1) = NaN
        assert e.value.code == -4
        assert sim.sample_indices(0, np.ones(4)).max() < 4              # context still usable


# ------------------------------------------------------- K6: replay mode
@pytest.mark.parametrize("seed", [0, 1])
def test_replay_step_bit_exact_vs_oracle(seed):
    rng = np.random.default_rng(seed)
    N, L, G = 24, 20000, 300
    core, acc = random_state(rng, N, L, G)
    ocore, opan = ob.Population(core, True, 0), ob.Population(acc, False, 0)
    p = pb.Params(pop_size=N, core_size=L, pan_genes=G, core_genes=0)
    main_rng = ob.make_rng(seed)
    with make(p) as sim:
        sim.upload(core, acc)
        for gen in range(3):
            parents = rng.integers(0, N, N).astype(np.uint32)
            ocore.next_generation(parents)
            opan.next_generation(parents)
            ev = ob.EventLog()
            # oracle generate mode = the reference's event loops (population.rs:467-751)
            ocore.mutate_alleles([3000.0], [(0, L)], seed, gen, ev)
            opan.mutate_alleles([40.0, 300.0], [(0, 250), (250, G)], seed, gen, ev)
            ocore.recombine([1500.0], [(0, L)], main_rng, seed, gen, ev)
            opan.recombine([30.0, 10.0], [(0, 250), (250, G)], main_rng, seed, gen, ev)
            a = ev.arrays()
            # force same-cell collisions: repeat a block of events with other alleles
            sim.step_replay(parents,
                            core_mut=(a["core_mut_row"], a["core_mut_site"], a["core_mut_allele"]),
                            acc_flip=(a["acc_flip_row"], a["acc_flip_gene"]),
                            hr=(a["hr_recipient"], a["hr_locus"], a["hr_value"]),
                            hgt=(a["hgt_recipient"], a["hgt_gene"]))
            assert (sim.download_core() == ocore.m).all()
            assert (sim.download_acc() == opan.m).all()


def test_replay_last_writer_wins_with_forced_collisions():
    N, L, G = 4, 100, 8
    core = np.ones((N, L), np.uint8)
    acc = np.zeros((N, G), np.uint8)
    p = pb.Params(pop_size=N, core_size=L, pan_genes=G, core_genes=0)
    rng = np.random.default_rng(3)
    M = 5000
    row = rng.integers(0, N, M).astype(np.uint32)
    site = rng.integers(0, 10, M).astype(np.uint32)            # 40 cells, 5000 writes
    val = (1 << rng.integers(1, 4, M)).astype(np.uint8)
    hrow = rng.integers(0, N, 700).astype(np.uint32)
    hsite = rng.integers(0, 12, 700).astype(np.uint32)
    hval = (1 << rng.integers(0, 4, 700)).astype(np.uint8)
    frow = rng.integers(0, N, 999).astype(np.uint32)
    fgene = rng.integers(0, G, 999).astype(np.uint32)
    parents = np.arange(N, dtype=np.uint32)
    ocore, opan = ob.Population(core, True), ob.Population(acc, False)
    ocore.apply_core_writes(row, site, val)
    ocore.apply_core_writes(hrow, hsite, hval)
    opan.apply_acc_flips(frow, fgene)
    opan.apply_acc_sets(np.array([1, 1], np.uint32), np.array([2, 2], np.uint32))
    with make(p) as sim:
        sim.upload(core, acc)
        sim.step_replay(parents, core_mut=(row, site, val), acc_flip=(frow, fgene), hr=(hrow, hsite, hval),
                        hgt=([1, 1], [2, 2]))
        assert (sim.download_core() == ocore.m).all()
        assert (sim.download_acc() == opan.m).all()


def test_replay_empty_events_is_gather():
    rng = np.random.default_rng(2)
    core, acc = random_state(rng, 5, 77, 9)
    parents = np.array([4, 4, 0, 1, 2], np.uint32)
    with make(pb.Params(pop_size=5, core_size=77, pan_genes=9, core_genes=0)) as sim:
        sim.upload(core, acc)
        sim.step_replay(parents)
        assert (sim.download_core() == core[parents]).all()


# ----------------------------------------- K4/K5: generate mode vs oracle
@pytest.mark.parametrize("kw", [
    dict(),                                                       # defaults-like rates
    dict(HR_rate=1.0, HGT_rate=1.0, rate_genes2=1000.0),          # cfg3: heavy recombination
    dict(core_mu=0.9, HR_rate=0.5),                               # many events per block
    dict(core_size=8192 * 3 + 5, HR_rate=0.3),                    # ragged last region
    dict(HR_rate=0.0, HGT_rate=0.0),                              # recombination off (main.rs:459-464)
    dict(prop_genes2=0.0), dict(prop_genes2=1.0),                 # single compartment
    dict(prop_positive=0.2, competition_strength=0.5),            # cfg2: selection on
])
def test_generate_step_equals_oracle_replay_of_its_own_events(kw):
    """The fused generate-mode step draws events from Philox and applies them in
    one pass. Dumping those events and replaying them on the ORACLE with the
    reference's operator order / snapshot / last-writer semantics must give the
    same state bit for bit (this checks gather, SNP apply, the HR snapshot
    recomputation, flips and HGT application)."""
    p = small_params(**kw)
    d = pb.derive(p)
    rng = np.random.default_rng(11)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < d.avg_gene_freq_adj).astype(np.uint8)
    sel = ob.selection_coefficients(ob.default_params(prop_positive=p.prop_positive), d.pan_size, ob.make_rng(1))
    ocore = ob.Population(np.tile(core_row, (p.pop_size, 1)), True, p.core_genes)
    opan = ob.Population(np.tile(acc_row, (p.pop_size, 1)), False, p.core_genes)
    with make(p) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        sim.enable_event_dump(4_000_000)
        for gen in range(p.n_gen):
            sim.step(gen)
            ev = sim.fetch_event_dump()
            oracle_apply_gpu_events(ev, sim.parents(), ocore, opan)
            assert (sim.download_core() == ocore.m).all(), f"core differs at gen {gen}"
            assert (sim.download_acc() == opan.m).all(), f"accessory differs at gen {gen}"
            if p.HR_rate > 0:
                assert len(ev["hr_recipient"]) > 0
                assert (ev["hr_recipient"] != ev["hr_donor"]).all()      # population.rs:616-619
            assert set(np.unique(ev["core_mut_allele"])) <= {2, 4, 8}   # population.rs:531 quirk


def test_hr_value_is_donor_post_mutation_snapshot():
    # population.rs:693-695: value = donor row after mutate_alleles, before any HR apply
    p = small_params(HR_rate=1.0, core_mu=0.3, n_gen=1)
    d = pb.derive(p)
    rng = np.random.default_rng(12)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.enable_event_dump(4_000_000)
        parents = rng.integers(0, p.pop_size, p.pop_size).astype(np.uint32)
        sim.step_with_parents(0, parents)
        ev = sim.fetch_event_dump()
    snap = ob.Population(core, True)
    snap.next_generation(parents)
    o = np.lexsort((ev["core_mut_seq"], ev["core_mut_row"]))
    snap.apply_core_writes(ev["core_mut_row"][o], ev["core_mut_site"][o], ev["core_mut_allele"][o])
    assert (snap.m[ev["hr_donor"], ev["hr_locus"]] == ev["hr_value"]).all()
    assert len(ev["hr_value"]) > 1000


def test_generate_mode_event_rates():
    """Event counts follow the reference's Poisson means (main.rs:275-280, 348-366)."""
    p = small_params(pop_size=64, core_size=200000, n_gen=1, HR_rate=0.5, HGT_rate=0.5)
    d = pb.derive(p)
    rng = np.random.default_rng(13)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size, 0.25)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.enable_event_dump(8_000_000)
        sim.step_with_parents(0, np.arange(p.pop_size, dtype=np.uint32))
        ev = sim.fetch_event_dump()
        rates = sim.rates()
    N = p.pop_size
    n_mut, n_hr = len(ev["core_mut_row"]), len(ev["hr_recipient"])
    exp_mut, exp_hr = N * d.n_core_mutations, N * d.n_recombinations_core
    assert abs(n_mut - exp_mut) < 5 * np.sqrt(exp_mut)
    assert abs(n_hr - exp_hr) < 5 * np.sqrt(exp_hr)
    # uniform positions: chi-square over 50 bins of the site coordinate
    h = np.bincount((ev["core_mut_site"].astype(np.int64) * 50) // p.core_size, minlength=50)
    assert ((h - n_mut / 50) ** 2 / (n_mut / 50)).sum() < 110
    # alleles uniform on {C,G,T}
    a = np.bincount(ev["core_mut_allele"], minlength=9)[[2, 4, 8]]
    assert ((a - n_mut / 3) ** 2 / (n_mut / 3)).sum() < 20
    # donors uniform over the other rows
    hd = np.bincount(ev["hr_donor"], minlength=N)
    assert ((hd - n_hr / N) ** 2 / (n_hr / N)).sum() < 2 * N
    # flips: per-gene probability (1 - exp(-2 rate)) / 2
    for c, (lo, hi) in enumerate(d.comp):
        f = ev["acc_flip_mask"][:, lo:hi].mean()
        sd = np.sqrt(rates[2 + c] * (1 - rates[2 + c]) / (N * (hi - lo)))
        assert abs(f - rates[2 + c]) < 5 * sd
    assert abs(rates[0] - (1 - np.exp(-d.n_core_mutations / p.core_size))) < 1e-15


def test_hgt_gain_probability_matches_event_process():
    """Gain probability of an absent gene = 1 - exp(-lambda_c/(N-1) * sum_d x_dg / K_dc)
    (derived from population.rs:616-680)."""
    p = small_params(pop_size=200, core_size=64, pan_genes=120, core_genes=20, HGT_rate=20.0, core_mu=0.5,
                     rate_genes1=0.0, rate_genes2=0.0, n_gen=1)
    d = pb.derive(p)
    rng = np.random.default_rng(14)
    N, G = p.pop_size, d.pan_size
    core = np.ones((N, 64), np.uint8)
    freq = np.linspace(0.05, 0.9, G)
    acc = (rng.random((N, G)) < freq[None, :]).astype(np.uint8)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.enable_event_dump(1 << 16)
        sim.step_with_parents(0, np.arange(N, dtype=np.uint32))
        gain = sim.fetch_event_dump()["acc_gain_mask"]
        new = sim.download_acc()
    assert (new == (acc | gain)).all()
    assert (gain & acc).sum() == 0
    z = 0.0
    for c, (lo, hi) in enumerate(d.comp):
        K = acc[:, lo:hi].sum(axis=1).astype(np.float64)
        S = ((acc[:, lo:hi] == 1) / np.where(K > 0, K, 1)[:, None]).sum(axis=0)
        pg = 1 - np.exp(-d.n_recombinations_pan[c] / (N - 1) * S)
        absent = (acc[:, lo:hi] == 0)
        exp_gain = (absent * pg[None, :]).sum()
        var = (absent * (pg * (1 - pg))[None, :]).sum()
        got = gain[:, lo:hi].sum()
        z = max(z, abs(got - exp_gain) / np.sqrt(var))
        assert exp_gain > 100
    assert z < 5


# ------------------------------------------------- E: column sharding
def test_column_shards_reproduce_single_context():
    """Results do not depend on how the core columns are split over contexts/GPUs:
    the RNG is keyed by (seed, gen, row, site block)."""
    p = small_params(core_size=8192 * 5 + 77, HR_rate=0.5, n_gen=3, prop_positive=0.1)
    d = pb.derive(p)
    rng = np.random.default_rng(15)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < 0.25).astype(np.uint8)
    sel = rng.normal(0, 0.05, d.pan_size)
    r1, r2 = sample_pairs(rng, p.pop_size, 200)
    cuts = [0, 8192 * 2, 8192 * 3, p.core_size]
    with make(p) as whole:
        shards = [make(p, site_begin=a, site_end=b) for a, b in zip(cuts[:-1], cuts[1:])]
        for s in [whole] + shards:
            s.set_initial(core_row, acc_row)
            s.set_selection(sel)
            s.run_generations(0, p.n_gen)
        full = whole.download_core()
        got = np.concatenate([s.download_core() for s in shards], axis=1)
        assert (got == full).all()
        for s in shards:
            assert (s.download_acc() == whole.download_acc()).all()
            assert (s.parents() == whole.parents()).all()
        cd, it, un = whole.pair_counts(r1, r2)
        part = sum(s.pair_counts(r1, r2)[0].astype(np.int64) for s in shards)
        assert (part == cd).all()
        for s in shards:
            s.close()


def test_run_generations_equals_repeated_step():
    p = small_params(n_gen=4, competition_strength=0.3, prop_positive=0.3)
    d = pb.derive(p)
    rng = np.random.default_rng(16)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    sel = rng.normal(0, 0.05, d.pan_size)
    with make(p) as a, make(p) as b:
        for s in (a, b):
            s.upload(core, acc)
            s.set_selection(sel)
        a.run_generations(0, 4)
        for g in range(4):
            b.step(g)
        assert (a.download_core() == b.download_core()).all()
        assert (a.download_acc() == b.download_acc()).all()
        # host-driven loop (reference call order, main.rs:435-464) gives the same result
    with make(p) as c:
        c.upload(core, acc)
        c.set_selection(sel)
        for g in range(4):
            avg = c.average_distance()
            parents = c.sample_indices(g, avg)
            c.step_with_parents(g, parents)
        with make(p) as a2:
            a2.upload(core, acc)
            a2.set_selection(sel)
            a2.run_generations(0, 4)
            assert (a2.download_core() == c.download_core()).all()
            assert (a2.download_acc() == c.download_acc()).all()


def test_state_required_and_error_codes():
    p = small_params()
    with make(p) as sim:
        with pytest.raises(pb.PansimError) as e:
            sim.step(0)
        assert e.value.code == -5
    with pytest.raises(pb.PansimError):
        make(pb.Params(pop_size=1, core_size=1000, pan_genes=10, core_genes=0, HR_rate=1.0))   # HR needs N >= 2


@pytest.mark.parametrize("kw", [dict(HR_rate=1.0, core_mu=0.2), dict(HR_rate=0.05, core_mu=0.05),
                                dict(HR_rate=4.0, core_mu=0.6)])
def test_recombination_list_pass_last_event_of_a_cell_wins(kw):
    """Recombination runs as collect + apply on the mutated rows (core_hr.cuh). Same-cell
    events are resolved inside the collect kernel (window of 32 events: highest lane; across
    windows: claim map, last window first); the oracle replays ALL dumped events in draw
    order with population.rs:745 store semantics and must end in the same state. The third
    parameter set puts ~2000 events on every 8192-site region (60+ windows, many repeats)."""
    p = small_params(core_size=8192 * 2 + 999, n_gen=2, pop_size=40, **kw)
    d = pb.derive(p)
    rng = np.random.default_rng(21)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    ocore = ob.Population(core.copy(), True, p.core_genes)
    opan = ob.Population(acc.copy(), False, p.core_genes)
    repeats = 0
    with make(p) as sim:
        sim.upload(core, acc)
        sim.enable_event_dump(8_000_000)
        for gen in range(p.n_gen):
            sim.step(gen)
            ev = sim.fetch_event_dump()
            cell = ev["hr_recipient"].astype(np.int64) * p.core_size + ev["hr_locus"]
            repeats += len(cell) - len(np.unique(cell))
            assert ev["hr_locus"].max() < p.core_size          # ragged last region: nothing beyond the end
            oracle_apply_gpu_events(ev, sim.parents(), ocore, opan)
            assert (sim.download_core() == ocore.m).all(), f"core differs at gen {gen}"
    if kw["HR_rate"] >= 1.0:
        assert repeats > 0


@pytest.mark.parametrize("kw", [
    dict(pop_size=200, core_size=8192 * 40 + 77, HR_rate=0.05),            # default rates, ragged last region
    dict(pop_size=64, core_size=8192 * 9, HR_rate=1.0, core_mu=0.2),       # several windows of 32 events per item
    dict(pop_size=40, core_size=8192 * 2 + 999, HR_rate=4.0, core_mu=0.6), # ~2000 events per region, many same-cell repeats
    dict(pop_size=3000, core_size=8192 * 12 + 5, HR_rate=0.05),
    dict(pop_size=2, core_size=100, HR_rate=1.0, core_mu=0.5),             # the only possible donor is the other row
])
def test_deferred_recombination_equals_immediate(monkeypatch, kw):
    """Default mode defers the recombination events of generation g: the next core step applies them
    to every region it gathers (donor cells read from the old, read-only buffer), and a reader of
    the state materialises them first (core_mut.cuh header). The state seen by download / distances
    after every generation must equal the one left by the immediate mode (PANSIM_HR_DEFER=0: collect +
    apply launches right after each gather+SNP pass), which the event-dump tests pin to the oracle."""
    p = small_params(n_gen=5, **kw)
    d = pb.derive(p)
    rng = np.random.default_rng(23)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    r1, r2 = sample_pairs(rng, p.pop_size, 50)
    out = {}
    for defer in ("0", "1"):
        monkeypatch.setenv("PANSIM_HR_DEFER", defer)
        with make(p) as sim:
            sim.upload(core, acc)
            sim.run_generations(0, 3)                    # two deferred applications inside the batch
            mid = sim.download_core()                    # materialises generation 2's events
            sim.run_generations(3, 1)
            cd = sim.pair_counts(r1, r2)[0]              # materialises generation 3's events
            sim.run_generations(4, 1)
            last, par = sim.download_core(), sim.parents()
            sim.run_generations(5, 1)                    # events pending again ...
            sim.next_generation(np.arange(p.pop_size, dtype=np.uint32)[::-1].copy())   # ... when a plain gather follows
            out[defer] = (mid, cd, last, par, sim.download_core())
    for a, b in zip(out["0"], out["1"]):
        assert (a == b).all()
    assert (out["0"][2] != core).any()


def test_recombination_is_reproducible_and_seed_dependent():
    p = small_params(HR_rate=1.0, n_gen=2)
    d = pb.derive(p)
    rng = np.random.default_rng(22)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    out = []
    for seed in (1, 1, 2):
        with make(dataclasses.replace(p, seed=seed)) as sim:
            sim.upload(core, acc)
            sim.run_generations(0, p.n_gen)
            out.append(sim.download_core())
    assert (out[0] == out[1]).all()
    assert (out[0] != out[2]).any()


def test_all_pairs_mode_matches_oracle():
    rng = np.random.default_rng(23)
    N, L, G = 37, 5000, 90
    core, acc = random_state(rng, N, L, G)
    ocore, opan = ob.Population(core, True, 4), ob.Population(acc, False, 4)
    seen = 0
    with make(pb.Params(pop_size=N, core_size=L, pan_genes=G + 4, core_genes=4)) as sim:
        sim.upload(core, acc)
        for ii, jj, cd, it, un in sim.iter_all_pairs(chunk_pairs=200):
            assert (ii < jj).all()
            assert (cd == ocore.pair_counts(ii, jj)).all()
            oi, ou = opan.pair_counts(ii, jj)
            assert (it == oi).all() and (un == ou).all()
            seen += len(ii)
        assert seen == N * (N - 1) // 2
        # the device-generated plan of a row block must not leak into a later sampled-pair call
        r1, r2 = sample_pairs(rng, N, 500)
        cd, it, un = sim.pair_counts(r1, r2)
        assert (cd == ocore.pair_counts(r1, r2)).all()
        cd2, _, _ = sim.pair_counts_rows(30, 37)
        assert len(cd2) == sum(N - 1 - i for i in range(30, 37))
        assert (sim.pair_counts(r1, r2)[0] == cd).all()


def test_all_pairs_row_blocks_larger_shape():
    """Row blocks of the exact all-pairs mode (pair list and row-stationary groups generated on the
    device): groups of 8 partners with ragged tails, several column chunks, empty last row."""
    rng = np.random.default_rng(29)
    N, L, G = 203, 70001, 40
    core, acc = random_state(rng, N, L, G)
    ocore, opan = ob.Population(core, True, 0), ob.Population(acc, False, 0)
    with make(pb.Params(pop_size=N, core_size=L, pan_genes=G, core_genes=0)) as sim:
        sim.upload(core, acc)
        blocks = list(sim.row_blocks(6000))
        assert blocks[0][0] == 0 and blocks[-1][1] == N - 1 and all(a[1] == b[0] for a, b in zip(blocks, blocks[1:]))
        for i0, i1 in blocks[::3] + [(N - 1, N), (5, 5)]:
            cd, it, un = sim.pair_counts_rows(i0, i1)
            ii = np.repeat(np.arange(i0, i1, dtype=np.uint32), [N - 1 - i for i in range(i0, i1)]).astype(np.uint32)
            jj = (np.concatenate([np.arange(i + 1, N, dtype=np.uint32) for i in range(i0, i1)])
                  if len(ii) else np.zeros(0, np.uint32))
            assert len(cd) == len(ii)
            if len(ii):
                assert (cd == ocore.pair_counts(ii, jj)).all()
                oi, ou = opan.pair_counts(ii, jj)
                assert (it == oi).all() and (un == ou).all()
        with pytest.raises(pb.PansimError):
            sim.pair_counts_rows(0, N + 1)


def test_no_accessory_genome_and_tiny_shapes():
    """pan_genes == core_genes -> zero accessory columns (population.rs:296 skips the fitness
    term); single-site / single-gene shapes; one pair."""
    p = pb.Params(pop_size=6, core_size=40, pan_genes=5, core_genes=5, n_gen=2, HGT_rate=0.0, core_mu=0.5, HR_rate=1.0)
    assert pb.derive(p).pan_size == 0
    rng = np.random.default_rng(3)
    core = (1 << rng.integers(0, 4, (6, 40))).astype(np.uint8)
    with make(p) as sim:
        sim.upload(core, np.zeros((6, 0), np.uint8))
        sim.run_generations(0, 3)
        parents = sim.parents()
        assert parents.max() < 6
        out = sim.download_core()
        assert set(np.unique(out)) <= {1, 2, 4, 8} and out.shape == (6, 40)
        cd, it, un = sim.pair_counts([0], [1])
        assert it[0] == 0 and un[0] == 0 and cd[0] == (out[0] != out[1]).sum()
        assert sim.gene_frequencies().tolist() == [1.0] * 5
    p1 = pb.Params(pop_size=2, core_size=1, pan_genes=2, core_genes=1, HR_rate=0.0, HGT_rate=0.0)
    with make(p1) as sim:
        sim.upload(np.array([[1], [8]], np.uint8), np.array([[1], [0]], np.uint8))
        cd, it, un = sim.pair_counts([0, 1], [1, 0])
        assert cd.tolist() == [1, 1] and it.tolist() == [0, 0] and un.tolist() == [1, 1]
        sim.run_generations(0, 2)
        assert sim.download_core().shape == (2, 1)


def test_empty_pair_list_and_large_pair_batch():
    rng = np.random.default_rng(4)
    core, acc = random_state(rng, 50, 3000, 64)
    with make(pb.Params(pop_size=50, core_size=3000, pan_genes=64, core_genes=0)) as sim:
        sim.upload(core, acc)
        cd, it, un = sim.pair_counts(np.zeros(0, np.uint32), np.zeros(0, np.uint32))
        assert len(cd) == 0
        r1, r2 = sample_pairs(rng, 50, 30000)        # many repeats of the same pairs
        cd, it, un = sim.pair_counts(r1, r2)
        assert (cd == ob.Population(core, True).pair_counts(r1, r2)).all()
        with pytest.raises(pb.PansimError):
            sim.pair_counts([0], [50])


def test_blocked_fitness_sum_for_large_shapes(monkeypatch):
    """Above 2^25 accessory cells the fitness sum uses a fixed blocked association instead of the
    strictly sequential chain: same gene counts, log-fitness within 1e-12 (relative) of the oracle."""
    monkeypatch.setenv("PANSIM_FITNESS_BLOCKED", "1")
    rng = np.random.default_rng(31)
    N, G = 70, 2500
    core, acc = random_state(rng, N, 40, G, 0.25)
    sel = rng.normal(0, 0.1, G)
    sel[7] = -1.0
    p = pb.Params(pop_size=N, core_size=40, pan_genes=G, core_genes=0)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.set_selection(sel)
        sim.sample_indices(0)
        w, ng, lf = sim.weights()
    ow, ong, olf = ob.Population(acc, False, 0).selection_weights(pb.derive(p).avg_gene_num, np.ones(N), sel)
    assert (ng == ong).all()
    np.testing.assert_allclose(lf, olf, rtol=1e-12, atol=1e-12)
    assert (lf[acc[:, 7] == 1] == 0.0).all()
    np.testing.assert_allclose(w / w.sum(), ow / ow.sum(), rtol=1e-10)


def test_zero_core_mutation_rate_is_pure_gather():
    """core_mu = 0 (hence no recombination either, main.rs:275-279): the generate-mode core step is
    next_generation alone (population.rs:450-465); every child row equals its parent's row."""
    rng = np.random.default_rng(5)
    N, L, G = 40, 20000, 64
    core, acc = random_state(rng, N, L, G)
    p = pb.Params(pop_size=N, core_size=L, pan_genes=G, core_genes=0, core_mu=0.0, HR_rate=0.05)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.run_generations(0, 1)
        parents = sim.parents()
        assert (sim.download_core() == core[parents]).all()


# ------------------------------------------------ the benchmarked kernel instance vs the oracle chain
@pytest.mark.parametrize("kw", [
    dict(pop_size=48, core_size=30000, HR_rate=0.05),
    dict(pop_size=64, core_size=8192 * 9 + 17, HR_rate=1.0, core_mu=0.2),      # several windows of 32 events per item
    dict(pop_size=33, core_size=8192 * 3 + 999, HR_rate=4.0, core_mu=0.6, prop_positive=0.1, competition_strength=0.5),
])
def test_event_dump_run_equals_default_run(kw):
    """bench.py times core_mut_kernel<RNG, no dump> with recombination deferred into the next launch
    (hr_window_fetch/apply); the oracle replay tests above pin core_mut_kernel<RNG, DUMP> +
    hr_collect_kernel<DUMP> (the event dump forces the immediate mode). Same Params and seed with and
    without the dump must leave identical states and parents: this ties the benchmarked instance to
    the oracle-verified one."""
    p = small_params(n_gen=3, **kw)
    d = pb.derive(p)
    rng = np.random.default_rng(41)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    sel = rng.normal(0, 0.05, d.pan_size)
    out = []
    for dump in (False, True):
        with make(p) as sim:
            sim.upload(core, acc)
            sim.set_selection(sel)
            if dump:
                sim.enable_event_dump(6_000_000)
            per_gen = []
            for g in range(3):
                sim.step(g)
                per_gen.append(sim.parents())
            out.append((sim.download_core(), sim.download_acc(), np.stack(per_gen)))
    for a, b in zip(*out):
        assert (a == b).all()
    assert (out[0][0] != core).any()


@pytest.mark.parametrize("name,kw", [
    ("cfg1", dict()),
    ("cfg3", dict(HR_rate=1.0, HGT_rate=1.0, rate_genes2=1000.0)),
])
def test_parity_at_the_benchmark_shape(monkeypatch, name, kw):
    """N = 1000, L = 1.2 Mbp, G = 4000 (BASELINE configs 1-3): the row-stationary pair plan, the
    L2-sized column chunks and the batch launch shape (8 items per warp) only exist at this size.
    Two generations, then (i) pair counts of 500 sampled pairs against the oracle's byte-per-site
    popcount path on the downloaded state, (ii) deferred == immediate recombination, (iii) event
    dump run == default run (the oracle-pinned instance, see test_event_dump_run_equals_default_run)."""
    p = pb.Params(pop_size=1000, core_size=1_200_000, pan_genes=6000, core_genes=2000, n_gen=2, max_distances=500,
                  seed=7, **kw)
    d = pb.derive(p)
    rng = np.random.default_rng(5)
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < d.avg_gene_freq_adj).astype(np.uint8)
    r1, r2 = sample_pairs(rng, p.pop_size, p.max_distances)

    def run(defer, dump=False):
        monkeypatch.setenv("PANSIM_HR_DEFER", defer)
        with make(p) as sim:
            sim.set_initial(core_row, acc_row)
            if dump:
                sim.enable_event_dump(140_000_000 if name == "cfg3" else 70_000_000)
                for g in range(2):
                    sim.step(g)
            else:
                sim.run_generations(0, 2)
            cd, it, un = sim.pair_counts(r1, r2)
            return sim.download_core(), sim.download_acc(), cd, it, un

    core, acc, cd, it, un = run("1")
    assert (core != core_row[None, :]).any()
    ocore = ob.Population(core, True, p.core_genes)
    assert (cd == ocore.pair_counts(r1, r2)).all()
    oi, ou = ob.Population(acc, False, p.core_genes).pair_counts(r1, r2)
    assert (it == oi).all() and (un == ou).all()
    del ocore
    core0, acc0, cd0, _, _ = run("0")
    assert (cd0 == cd).all() and (acc0 == acc).all()
    assert np.array_equal(core0, core)
    del core0
    if name == "cfg1":
        cored, accd, cdd, _, _ = run("1", dump=True)
        assert (cdd == cd).all() and (accd == acc).all()
        assert np.array_equal(cored, core)


def test_entry_point_orders_that_rotate_parents_without_a_core_step():
    """A generate-mode step returns with the core kernel still in flight; every later reader must
    join THAT launch even when pansim_sample_indices / pansim_next_generation have rotated the
    parents buffers in between (the join event is per launch, not per parents slot)."""
    p = small_params(pop_size=300, core_size=8192 * 60 + 5, n_gen=3, HR_rate=0.5)
    d = pb.derive(p)
    rng = np.random.default_rng(61)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    par = [rng.integers(0, p.pop_size, p.pop_size).astype(np.uint32) for _ in range(3)]
    rev = np.arange(p.pop_size, dtype=np.uint32)[::-1].copy()

    def reference_run():
        with make(p) as sim:
            sim.upload(core, acc)
            sim.step_with_parents(0, par[0])
            a = sim.download_core()                       # joins right after the step
            sim.step_with_parents(1, par[1])
            b = sim.download_core()
            sim.next_generation(rev)
            return a, b, sim.download_core()

    a, b, c3 = reference_run()
    with make(p) as sim:
        sim.upload(core, acc)
        sim.step_with_parents(0, par[0])
        sim.sample_indices(7)                             # rotates the parents slot, launches no core step
        assert (sim.download_core() == a).all()
        sim.step_with_parents(1, par[1])
        sim.sample_indices(8)
        sim.sample_indices(9)
        cd = sim.pair_counts([0, 5], [1, 6])[0]
        assert cd[0] == (b[0] != b[1]).sum() and cd[1] == (b[5] != b[6]).sum()
        assert (sim.download_core() == b).all()
    with make(p) as sim:
        sim.upload(core, acc)
        sim.step_with_parents(0, par[0])
        sim.step_with_parents(1, par[1])
        sim.next_generation(rev)                          # plain gather right behind an in-flight generate step
        assert (sim.download_core() == c3).all()


def test_step_with_parents_consumes_the_vector_before_returning():
    """The header's 'valid for the call' contract: the parents vector may be overwritten as soon as
    the call returns (it is staged through the context's pinned buffer)."""
    p = small_params(pop_size=500, core_size=8192 * 30, n_gen=2, HR_rate=0.0)
    d = pb.derive(p)
    rng = np.random.default_rng(62)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    par = rng.integers(0, p.pop_size, p.pop_size).astype(np.uint32)
    with make(dataclasses.replace(p, core_mu=0.0)) as sim:
        sim.upload(core, acc)
        buf = par.copy()
        sim.step_with_parents(0, buf)
        buf[:] = 0                                        # scribble over it immediately
        assert (sim.download_core() == core[par]).all()


# ------------------------------------------------ per-generation statistics on the device (8f-4)
@pytest.mark.parametrize("N,L,G,P", [(9, 100, 31, 7), (40, 20011, 333, 1024), (64, 8192 * 3, 500, 5000), (17, 501, 64, 1025)])
def test_pair_stats_equal_reference_order_sums(N, L, G, P):
    """pansim_pair_stats = pairwise_distances x2 + standard_deviation x2 (main.rs:502-519,
    population.rs:87-94). The oracle sums left to right like `iter().sum::<f64>()`; the device chain
    does the same, so all four doubles are bit-identical (also with P not a multiple of the chunk)."""
    rng = np.random.default_rng(N + P)
    core, acc = random_state(rng, N, L, G)
    r1, r2 = sample_pairs(rng, N, P)
    p = pb.Params(pop_size=N, core_size=L, pan_genes=G + 5, core_genes=5)
    with make(p) as sim:
        sim.upload(core, acc)
        avg_core, std_core, avg_acc, std_acc = sim.pair_stats(r1, r2)
        core_d, acc_d = sim.pairwise_distances(r1, r2)
    o_std_c, o_avg_c = ob.standard_deviation(core_d)
    o_std_a, o_avg_a = ob.standard_deviation(acc_d)
    assert (avg_core, std_core, avg_acc, std_acc) == (o_avg_c, o_std_c, o_avg_a, o_std_a)
    assert (std_core, avg_core) == pb.standard_deviation(core_d)


def test_run_generations_stats_equals_host_loop():
    """The --print_dist loop as one device-resident batch: states, parents and the per-generation
    statistics equal those of the host-driven loop (step, distance pass, host-side sums)."""
    p = small_params(pop_size=60, core_size=8192 * 5 + 77, n_gen=5, HR_rate=0.5, prop_positive=0.1, competition_strength=0.3)
    d = pb.derive(p)
    rng = np.random.default_rng(71)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    sel = rng.normal(0, 0.05, d.pan_size)
    r1, r2 = sample_pairs(rng, p.pop_size, 700)
    with make(p) as a, make(p) as b:
        for s in (a, b):
            s.upload(core, acc)
            s.set_selection(sel)
        stats = a.run_generations_stats(0, 5, r1, r2)
        want = []
        for g in range(5):
            b.step(g)
            core_d, acc_d = b.pairwise_distances(r1, r2)
            sc, ac = ob.standard_deviation(core_d)
            sa, aa = ob.standard_deviation(acc_d)
            want.append((ac, sc, aa, sa))
        assert stats.tolist() == [list(w) for w in want]
        assert (a.download_core() == b.download_core()).all() and (a.download_acc() == b.download_acc()).all()
        assert (a.parents() == b.parents()).all()


def test_select_parents_is_average_distance_plus_sample_indices():
    p = small_params(pop_size=200, prop_positive=0.1, competition_strength=0.5)
    d = pb.derive(p)
    rng = np.random.default_rng(72)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    sel = rng.normal(0, 0.05, d.pan_size)
    with make(p) as a, make(p) as b:
        for s in (a, b):
            s.upload(core, acc)
            s.set_selection(sel)
        for g in range(3):
            avg, par = a.select_parents(g)
            avg2 = b.average_distance()
            par2 = b.sample_indices(g, avg2)
            assert (avg == avg2).all() and (par == par2).all()
            a.step_with_parents(g, par)
            b.step_with_parents(g, par2)
        assert (a.download_core() == b.download_core()).all()
    with make(dataclasses.replace(p, competition_strength=0.0)) as c:
        c.upload(core, acc)
        avg, par = c.select_parents(0)
        assert (avg == 1.0).all() and par.max() < p.pop_size          # main.rs:435


@pytest.mark.parametrize("N", [1500, 5000])
def test_selection_weights_for_large_populations(N):
    """N > 1024 uses the global-memory selection kernel (256 threads up to 4096 individuals, 1024
    beyond): weights within 1e-12 of the oracle's three-softmax product (population.rs:325-393),
    the cumulative table consistent with them, the draws a pure function of (seed, gen)."""
    rng = np.random.default_rng(N)
    G = 96
    core, acc = random_state(rng, N, 64, G, 0.4)
    sel = rng.normal(0, 0.08, G)
    p = pb.Params(pop_size=N, core_size=64, pan_genes=G, core_genes=0, competition_strength=0.7)
    avg = rng.uniform(0.05, 0.9, N)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.set_selection(sel)
        par = sim.sample_indices(3, avg)
        w, ng, lf = sim.weights()
        par2 = sim.sample_indices(3, avg)
    ow, ong, olf = ob.Population(acc, False, 0).selection_weights(pb.derive(p).avg_gene_num, avg, sel, competition_strength=0.7)
    assert (ng == ong).all() and (lf == olf).all()
    np.testing.assert_allclose(w, ow, rtol=1e-12)
    assert (par == par2).all() and par.max() < N
    # the favoured individuals are drawn more often: mean weight of the drawn parents exceeds the plain mean
    assert w[par].mean() > w.mean()


@pytest.mark.parametrize("kw", [
    dict(pop_size=120, core_size=8192 * 6 + 5, HR_rate=0.5, prop_positive=0.1, competition_strength=0.4),
    dict(pop_size=64, core_size=30000, HR_rate=0.0),                       # no recombination: nothing pending between generations
    dict(pop_size=90, core_size=8192 * 3, HR_rate=1.0, core_mu=0.2, pan_genes=100, core_genes=100),   # no accessory genome
])
def test_graph_replay_equals_launch_by_launch(monkeypatch, kw):
    """Device-resident batches launch the selection chain + accessory step of every generation as ONE CUDA
    graph (six phases of the buffer rotation, relative generation numbers + a device counter the graph
    advances). States, parents, pair counts and per-generation statistics must equal those of the same
    batches enqueued kernel by kernel (PANSIM_GRAPH=0), across several calls (graph cache, all phases, a
    reader between the calls that materialises the pending recombination)."""
    p = small_params(n_gen=3, **kw)
    d = pb.derive(p)
    rng = np.random.default_rng(81)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    sel = rng.normal(0, 0.05, d.pan_size)
    r1, r2 = sample_pairs(rng, p.pop_size, 200)
    out = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("PANSIM_GRAPH", mode)
        with make(p) as sim:
            sim.upload(core, acc)
            sim.set_selection(sel)
            sim.run_generations(0, 60)
            a = (sim.download_core(), sim.download_acc(), sim.parents())
            sim.run_generations(60, 26)              # starts in another phase of the buffer rotation
            cd = sim.pair_counts(r1, r2)[0]
            sim.run_generations(86, 25)
            sim.run_generations(111, 7)              # short batch: launch by launch
            st = sim.run_generations_stats(118, 9, r1, r2)
            b = (sim.download_core(), sim.download_acc(), sim.parents())
            out[mode] = a + (cd, st) + b
    for x, y in zip(out["0"], out["1"]):
        assert (x == y).all()


def test_write_core_csv_streams_the_same_text(tmp_path):
    """pansim_write_core_csv (GPU text expansion, two pinned chunks in flight) writes exactly the rows
    pansim_export_core_csv returns, over several chunks and with pending recombination materialised first."""
    p = small_params(pop_size=600, core_size=40000, n_gen=2, HR_rate=0.5)
    d = pb.derive(p)
    rng = np.random.default_rng(91)
    core, acc = random_state(rng, p.pop_size, p.core_size, d.pan_size)
    with make(p) as sim:
        sim.upload(core, acc)
        sim.run_generations(0, 2)                      # recombination of generation 1 still pending
        path = str(tmp_path / "core.csv")
        n = sim.write_core_csv(path)
        assert n == 2 * p.pop_size * p.core_size       # 48 MB: two 32 MB chunks
        state = sim.download_core()
        text = open(path, "rb").read()
        assert text == sim.export_core_csv(0, p.pop_size)
    lut = np.zeros(9, np.uint8)
    lut[[1, 2, 4, 8]] = np.frombuffer(b"ACGT", np.uint8)
    want = np.empty((p.pop_size, p.core_size, 2), np.uint8)
    want[:, :, 0] = lut[state]
    want[:, :, 1] = ord(",")
    want[:, -1, 1] = ord("\n")
    assert text == want.tobytes()
