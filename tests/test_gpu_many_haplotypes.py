"""The CUDA path on windows with more distinct haplotype keys than a warp table (32) holds: the block histogram tier
(kernels/block_kernels.cu) behind the wide kernels and the serial replay, junctions with more than 255 merged records on
the device, and the 4096-key limit. Outputs must be the oracle's bytes."""
import os
import sys

import pytest

from conftest import GOLDEN, ROOT, materialize_reference, read_outputs, run_cli
from test_many_haplotypes_emu import LIMIT, LIMIT_MSG, LIMIT_REPLAY, MANYHAP, MANYHAP_PROFILES, SEEDS, make_input

sys.path.insert(0, ROOT)
sys.path.insert(0, GOLDEN)
import bailite  # noqa: E402
from microphaser_b200 import synth  # noqa: E402
from test_emu_parity import NORMAL, PROFILES, SOMATIC  # noqa: E402
from test_gpu_indexed import run_files  # noqa: E402

pytestmark = pytest.mark.gpu


def oracle_outputs(oracle_bin, d, out, mode):
    os.makedirs(out, exist_ok=True)
    r = run_cli(oracle_bin, d, out, subcommand=mode)
    assert r.returncode == 0, r.stderr.decode()[-300:]
    return read_outputs(out, mode)


def cli_outputs(product, d, out, mode):
    os.makedirs(out, exist_ok=True)
    r = run_cli(product[1], d, out, subcommand=mode)
    assert r.returncode == 0, r.stderr.decode()[-300:]
    return read_outputs(out, mode)


@pytest.mark.parametrize("force_wide", ["", "1", "2"])
@pytest.mark.parametrize("mode", ["somatic", "normal"])
@pytest.mark.parametrize("profile", list(MANYHAP_PROFILES))
@pytest.mark.parametrize("seed", SEEDS)
def test_cuda_cli_matches_oracle_with_many_keys(product, oracle_bin, profile, seed, mode, force_wide, tmp_path, monkeypatch):
    """manyhap_junction has splice junctions with more than 255 merged records on device-class transcripts."""
    d = make_input(tmp_path, profile, seed)
    want = oracle_outputs(oracle_bin, d, str(tmp_path / "o"), mode)
    if force_wide:
        monkeypatch.setenv("MPH_FORCE_WIDE", force_wide)
    else:
        monkeypatch.delenv("MPH_FORCE_WIDE", raising=False)
    assert cli_outputs(product, d, str(tmp_path / "p"), mode) == want


@pytest.mark.parametrize("case", SOMATIC + NORMAL)
def test_goldens_through_the_block_tier(product, case, tmp_path, monkeypatch):
    """MPH_FORCE_WIDE=2: every window with a key besides (0, 0) is spilled and folded by k_window_hist_block."""
    monkeypatch.setenv("MPH_FORCE_WIDE", "2")
    d = os.path.join(GOLDEN, case)
    fa = materialize_reference(d, str(tmp_path))
    r = run_cli(product[1], d, str(tmp_path), ref=fa, subcommand="normal" if case in NORMAL else "somatic")
    assert r.returncode == 0, r.stderr.decode()
    for name in sorted(os.listdir(os.path.join(d, "expected"))):
        assert open(tmp_path / name, "rb").read() == open(os.path.join(d, "expected", name), "rb").read(), name


@pytest.mark.parametrize("mode", ["somatic", "normal"])
@pytest.mark.parametrize("profile", list(PROFILES))
def test_profiles_through_the_block_tier(product, oracle_bin, profile, mode, tmp_path, monkeypatch):
    d = str(tmp_path / "in")
    synth.generate(d, synth.Params(seed=2024 + len(profile), n_genes=4, coverage=30.0, **PROFILES[profile]))
    want = oracle_outputs(oracle_bin, d, str(tmp_path / "o"), mode)
    monkeypatch.setenv("MPH_FORCE_WIDE", "2")
    assert cli_outputs(product, d, str(tmp_path / "p"), mode) == want


@pytest.mark.parametrize("mode", ["somatic", "normal"])
@pytest.mark.parametrize("profile", ["manyhap", "manyhap_junction"])
def test_contexts_and_shards_with_many_keys(product, oracle_bin, profile, mode, tmp_path, monkeypatch):
    """Two contexts, and the indexed driver in 8+ shards: the spill arenas and queues reused between calls hold no stale state."""
    d = make_input(tmp_path, profile, SEEDS[0])
    want = oracle_outputs(oracle_bin, d, str(tmp_path / "o"), mode)
    assert run_files(d, str(tmp_path / "multi"), mode, n_ctx=2) == want
    bailite.write(os.path.join(d, "reads.bam"))
    n_reads = len(bailite._records(os.path.join(d, "reads.bam"))[1])
    monkeypatch.setenv("MPH_SHARD_READS", str(max(1, n_reads // 10)))
    for n_ctx in (1, 2):
        assert run_files(d, str(tmp_path / ("idx%d" % n_ctx)), mode, n_ctx) == want, n_ctx


@pytest.mark.parametrize("force_wide", ["", "2"])
@pytest.mark.parametrize("mode", ["somatic", "normal"])
def test_spill_arena_grows(product, oracle_bin, mode, force_wide, tmp_path, monkeypatch):
    """One gene at 3000x. With MPH_FORCE_WIDE=2 its windows spill about 156 000 observations, twice the arena's first
    allocation: the stage reruns with a larger one."""
    d = str(tmp_path / "in")
    synth.generate(d, synth.Params(seed=3000, **dict(MANYHAP, n_genes=1, coverage=3000.0)))
    want = oracle_outputs(oracle_bin, d, str(tmp_path / "o"), mode)
    if force_wide:
        monkeypatch.setenv("MPH_FORCE_WIDE", force_wide)
    assert cli_outputs(product, d, str(tmp_path / "p"), mode) == want


@pytest.mark.parametrize("limit", ["closed_form", "replay"])
@pytest.mark.parametrize("mode", ["somatic", "normal"])
def test_more_than_4096_keys_is_unsupported(product, mode, limit, tmp_path):
    d = str(tmp_path / "in")
    synth.generate(d, synth.Params(seed=21, **(LIMIT if limit == "closed_form" else LIMIT_REPLAY)))
    p = tmp_path / "p"
    p.mkdir()
    r = run_cli(product[1], d, str(p), subcommand=mode)
    assert r.returncode == 3, r.stderr.decode()[-300:]
    assert LIMIT_MSG in r.stderr
