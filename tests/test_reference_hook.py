"""The hook that pins parity the day the reference source is available: `make -C oracle _ref REF=<dir>` compiles the
reference's own k-mer layer from <dir>/src/kmers (never copied into this repo).  Without those sources the target is
a no-op and the pinning test skips -- the oracle stays a spec-derived restatement ("parity unpinned", SURVEY.md 8c)."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ref_target_runs_and_reports(tmp_path):
    """`make _ref` on a copy of oracle/Makefile (so nothing lands in this tree): a reference directory without k-mer
    sources builds nothing and says so; with them (a stand-in source here) the library is compiled."""
    mk = tmp_path / "oracle"
    mk.mkdir()
    shutil.copy(os.path.join(ROOT, "oracle", "Makefile"), str(mk))
    src = tmp_path / "reference" / "src" / "kmers"
    src.mkdir(parents=True)

    def make_ref():
        out = subprocess.run(["make", "-C", str(mk), "-s", "_ref", "REF=%s" % (tmp_path / "reference")],
                             capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        return out.stdout

    assert "parity unpinned" in make_ref()
    assert not (mk / "_ref").exists()
    (src / "KmerSpectra.cc").write_text("int kmer_spectra_stand_in() { return 0; }\n")
    stdout = make_ref()
    assert (mk / "_ref" / "libref_kmers.so").exists(), stdout


def test_oracle_against_the_reference_build():
    so = os.path.join(ROOT, "oracle", "_ref", "libref_kmers.so")
    if not os.path.exists(so):
        pytest.skip("no reference build (the reference mount holds no source): parity unpinned")
    # The day this runs: drive the reference's KmerSpectrum / SortKmers entry points on the synthetic configs of
    # SURVEY.md section 8(d) and diff them with oracle_a.count / oracle_a.spectrum; until the signatures can be read
    # (Appendix A.2, questions 1-9) nothing can be asserted here.
    pytest.fail("a reference build exists: write the pinning comparison against its entry points (SURVEY.md Appendix A)")
