"""CPU checks of the streaming kernel's model (tests/k1_model.py) against the compiler's gram sets, and of the inputs the GPU
fast-path tests (tests/test_fast_path_gpu.py) rely on: that they reach every k_stream instantiation and every verification
kernel, and that most of them stay on the fast path."""

import random

import pytest

import fast_path_cases as fpc
from dfa_sim import CompiledDb, prefilter_flagged_chunks
from k1_model import K1Tables, has_newline_free_super_block, k1_candidates, super_block_bytes
from test_compiler import LITS, _factor_pattern


def _text(rng: random.Random, size: int) -> bytes:
    out = bytearray(rng.choice(b"abcAB _x1.\t\n\0") for _ in range(size))
    for _ in range(size // 24):
        at = rng.randrange(size)
        lit = rng.choice(LITS).encode()
        out[at:at + len(lit)] = lit
    return bytes(out[:size])


@pytest.mark.parametrize("seed", range(40))
def test_model_flags_the_chunks_of_the_exact_grams(seed, gpu_lib):
    """Exact mode flags exactly the chunks in which dfa_sim finds a sampled gram of the set; the bloom bitmap (with the
    multiplier that gpugrep_db_copy_prefilter reports) flags a superset of them.  Tuned and untuned tables, every length
    mod 16."""
    rng = random.Random(seed)
    k = rng.choice([1, 2, 4])
    db = CompiledDb(gpu_lib, [_factor_pattern(rng) for _ in range(k)], [rng.choice([14, 14, 15, 10])] * k, [0] * k)
    assert db.rc == 0
    if not db.info.prefilter:
        pytest.skip("no usable factor")
    data = _text(rng, rng.randint(1, 3000))
    if seed % 2:
        db.retune(_text(rng, 8192))
    tables = K1Tables(db)
    if db.info.prefilter_fold and int.from_bytes(b"    ", "little") in db.grams:
        pytest.skip("the folded zero padding past the end reads as a gram of the set")
    want = sorted(prefilter_flagged_chunks(db, data))
    newlines, exact = k1_candidates(data, tables, exact=True)
    assert exact.tolist() == want
    assert newlines == data.count(b"\n")
    _, bloom = k1_candidates(data, tables)
    assert set(exact.tolist()) <= set(bloom.tolist())
    # every gram of the set is in the bitmap under the reported multiplier
    assert tables.bloom_hit(tables.grams).all()


def test_copy_prefilter_reports_the_bloom_multiplier(gpu_lib):
    """A tuned table picks its bitmap multiplier among eight (prefilter.cpp finish_tables): the one whose bitmap the sample's
    other grams hit least.  The introspection entry point must report that one, not the multiplier of the exact table."""
    db = CompiledDb(gpu_lib, fpc.words(7, 200, 6), [15] * 200)
    rng = random.Random(3)
    muls = set()
    for _ in range(4):
        db.retune(bytes(rng.choice(b"abcdefghiklmnop rstuvwy\n") for _ in range(200000)))
        tables = K1Tables(db)
        assert tables.log2_bits == 20
        assert tables.bloom_hit(tables.grams).all()
        muls.add(tables.bloom_mul)
    assert muls - {0x9E3779B1}, "every sample kept the first multiplier"


def test_k1_configs_reach_every_instantiation(gpu_lib):
    """The pattern sets of the GPU K1 tests select all 14 fast-path instantiations of k_stream (MODE 1/2 x STRIDE 4/2/1 x
    FOLD, and the two mixed-sampling ones)."""
    reached = set()
    for name, pats, flags, env, inst in fpc.K1_CONFIGS:
        with fpc.environment(env):
            db = CompiledDb(gpu_lib, pats, flags)
            assert db.rc == 0 and db.info.simple and db.info.prefilter, name
            if "GPUGREP_NO_TUNE" not in env:
                db.retune(b"qjxz 0123 host=1 dur=2\n" * 1000)
            got = fpc.instantiation(K1Tables(db), env)
        assert got == inst, (name, got)
        reached.add(got)
    assert reached == fpc.ALL_INSTANTIATIONS, sorted(fpc.ALL_INSTANTIATIONS - reached)


N_FAST_CASES = 40


def test_random_fast_path_cases_cover_the_verification_kernels(gpu_lib):
    """The random cases of the GPU tests: most are built to stay on the fast path, and together (default run and switch run)
    they reach k_verify_smem, k_verify_local<false> with and without k_confirm and k_verify_local<true>, folded tables,
    mixed sampling and every super-block size."""
    variants, supers, fast, insts = set(), set(), 0, set()
    for seed in range(N_FAST_CASES):
        case = fpc.fast_case(seed)
        for switch in ("", case["switch"]):
            pats, flags, ids = fpc.tagged(case, switch) if switch else (case["patterns"], case["flags"], case["ids"])
            p = fpc.predict(gpu_lib, pats, flags, ids, fpc.switch_env(switch), case["data"], case["buffer_size"])
            if p["fast"]:
                variants.add(p["verify"])
                insts.add(p["inst"])
                fast += switch == "" and p["path"] == 1
        supers.add(super_block_bytes(case["buffer_size"]))
    assert {"smem", "local", "local+confirm", "local_nfa+confirm"} <= variants, variants
    assert fast >= 0.7 * N_FAST_CASES, fast
    assert {2048, 4096, 8192, 32768, 65536} <= supers
    assert any(i[2] for i in insts) and any(i[3] for i in insts), insts


def test_super_block_rule():
    """The long-line check of the fast path: super-block sizes per buffer_size, and which texts hold a newline-free one."""
    assert [super_block_bytes(b) for b in fpc.BUFFER_SIZES] == [2048, 2048, 2048, 4096, 8192, 32768, 65536, 65536, 65536]
    assert super_block_bytes(4095) == 0
    s = 2048
    assert not has_newline_free_super_block(b"x" * (s - 1) + b"\n", s)
    assert has_newline_free_super_block(b"x" * s + b"\n", s)
    assert not has_newline_free_super_block(b"y\n" + b"x" * s + b"\n", s)   # not aligned
    assert has_newline_free_super_block(b"y\n" + b"x" * (2 * s - 1) + b"\n", s)
    assert has_newline_free_super_block(b"y" * (s + 10), s)   # the zero padding of the last block counts
    assert not has_newline_free_super_block(b"y" * 10, s)
