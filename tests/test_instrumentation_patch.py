"""integration/instrument_population.patch must apply to the reference tree (SURVEY.md 8f-3).

The patch is the route to real reference event dumps (PANSIM_EVENT_DUMP=<file> on a patched
`pansim` binary writes the PSEV records pansim_step_replay consumes). Without a Rust toolchain,
what can be checked is that the unified diff applies cleanly to a pristine copy of the reference
and that the hooks land on the lines the C ABI header cites. The reference (bacpop/Pansim) is not
part of this repository: set PANSIM_REFERENCE to the `pansim` crate directory of a checkout of it
to run that test; without it the test is skipped. The reference lines the patch itself records
(context and removed lines, at their line numbers) are checked without the reference."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATCH = os.path.join(ROOT, "integration", "instrument_population.patch")
REF = os.environ.get("PANSIM_REFERENCE", "")

needs_ref = pytest.mark.skipif(not os.path.isdir(REF),
                               reason="PANSIM_REFERENCE does not name a checkout of the reference's pansim crate")


def test_patch_touches_the_documented_files_only():
    text = open(PATCH).read()
    files = sorted(set(re.findall(r"^\+\+\+ b/(\S+)", text, flags=re.M)))
    assert files == ["pansim/src/event_dump.rs", "pansim/src/lib.rs", "pansim/src/main.rs", "pansim/src/population.rs"]
    # the new module in the patch is the committed source of integration/event_dump.rs
    added = [l[1:] for l in text.split("+++ b/pansim/src/event_dump.rs", 1)[1].split("\ndiff --git", 1)[0].splitlines()
             if l.startswith("+")]
    assert "\n".join(added).strip() == open(os.path.join(ROOT, "integration", "event_dump.rs")).read().strip()


def _hunk_images(text):
    """{path: (old {line: text}, new {line: text})} from the context, removed and added lines of each hunk."""
    images = {}
    for block in text.split("diff --git ")[1:]:
        path = re.search(r"^\+\+\+ b/(\S+)", block, flags=re.M).group(1)
        old, new = images.setdefault(path, ({}, {}))
        o = n = 0
        for line in block.splitlines():
            m = re.match(r"@@ -(\d+)(?:,\d+)? \+(\d+)(?:,\d+)? @@", line)
            if m:
                o, n = int(m.group(1)), int(m.group(2))
            elif o or n:
                if line.startswith((" ", "-")) or line == "":
                    old[o] = line[1:]
                    o += 1
                if line.startswith((" ", "+")) or line == "":
                    new[n] = line[1:]
                    n += 1
    return images


def test_patch_hooks_sit_on_the_reference_lines_it_records(tmp_path):
    """Without the reference tree: the context and removed lines of the patch are the reference's own lines
    at their line numbers. The stores the C ABI header cites sit on those lines, the hooks follow them in
    the documented order, and the patch applies to a tree rebuilt from those lines (hunk offsets and
    counts consistent)."""
    text = open(PATCH).read()
    images = _hunk_images(text)
    old, new = images["pansim/src/population.rs"]

    def at(image, needle):
        hits = [k for k, v in image.items() if needle in v]
        assert len(hits) >= 1, needle
        return hits

    assert at(old, "row[mutant_site] = new_allele;") == [508]           # include/pansim_b200.h: population.rs:508
    assert at(old, "row[mutant_site] = *new_allele;") == [537]          # :537, inside :525-538
    assert at(old, "self.pop[[row_idx, col_idx]] = value;") == [745]   # :745, inside :741-746
    assert 443 < at(new, "event_dump::set_parents(&sampled_indices);")[0] < 455
    a, = at(new, "event_dump::push_row_mutations(false, dump_row_idx, &dumped);")
    b, = at(new, "event_dump::push_row_mutations(true, dump_row_idx, &dumped);")
    c, = at(new, "event_dump::push_transfer(dump_is_core, pop_idx, row_idx, col_idx, value);")
    assert a < b < c
    assert new[c - 1].strip() == "self.pop[[row_idx, col_idx]] = value;"     # recorded right after the store
    removed = [l[1:].strip() for l in text.splitlines() if l.startswith("-") and not l.startswith("---")]
    assert removed == [".for_each(|mut row| {", ".for_each(|mut row| {"]

    # a pristine tree holding the recorded lines, unique filler elsewhere: the patch must apply to it and
    # leave every line it records on the line number it records
    for path, (old, new) in images.items():
        if not old:
            continue
        f = tmp_path / path
        f.parent.mkdir(parents=True, exist_ok=True)
        f.write_text("".join(old.get(k, f"// {path} line {k}") + "\n" for k in range(1, max(old) + 1)))
    subprocess.run(["git", "apply", "--check", PATCH], cwd=tmp_path, check=True)
    subprocess.run(["git", "apply", PATCH], cwd=tmp_path, check=True)
    for path, (_, new) in images.items():
        got = (tmp_path / path).read_text().splitlines()
        assert all(got[k - 1] == v for k, v in new.items()), path


@needs_ref
def test_patch_applies_to_the_reference(tmp_path):
    work = tmp_path / "ref"
    shutil.copytree(REF, work / "pansim")
    r = subprocess.run(["git", "apply", "--check", "--verbose", PATCH], cwd=work, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    subprocess.run(["git", "apply", PATCH], cwd=work, check=True)
    pop = (work / "pansim" / "src" / "population.rs").read_text().splitlines()
    main = (work / "pansim" / "src" / "main.rs").read_text()
    lib = (work / "pansim" / "src" / "lib.rs").read_text()
    assert "pub mod event_dump;" in lib
    assert "pansim::event_dump::init_from_env();" in main and "pansim::event_dump::finish_generation(j as u32);" in main

    def line_of(needle, nth=0):
        hits = [i + 1 for i, l in enumerate(pop) if needle in l]
        assert len(hits) > nth, needle
        return hits[nth]

    # hooks sit where include/pansim_b200.h and INTEGRATION.md say (line numbers of the patched file,
    # a handful of lines after the unpatched ones)
    orig = open(os.path.join(REF, "src", "population.rs")).read().splitlines()

    def orig_line(needle, nth=0):
        return [i + 1 for i, l in enumerate(orig) if needle in l][nth]

    assert orig_line("let sampled_indices: Vec<usize>") == 443
    assert 443 < line_of("event_dump::set_parents(&sampled_indices);") < 455
    assert 501 <= orig_line("row[mutant_site] = new_allele;") <= 509
    assert 525 <= orig_line("row[mutant_site] = *new_allele;") <= 538
    assert 741 <= orig_line("self.pop[[row_idx, col_idx]] = value;") <= 746
    a = line_of("event_dump::push_row_mutations(false, dump_row_idx, &dumped);")
    b = line_of("event_dump::push_row_mutations(true, dump_row_idx, &dumped);")
    c = line_of("event_dump::push_transfer(dump_is_core, pop_idx, row_idx, col_idx, value);")
    assert a < b < c
    assert pop[c - 2].strip() == "self.pop[[row_idx, col_idx]] = value;"       # recorded right after the store, in apply order
    # the patch only adds instrumentation: it removes exactly the two closure headers it re-writes
    removed = [l[1:].strip() for l in open(PATCH).read().splitlines() if l.startswith("-") and not l.startswith("---")]
    assert removed == [".for_each(|mut row| {", ".for_each(|mut row| {"]
