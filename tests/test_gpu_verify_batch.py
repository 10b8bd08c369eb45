"""vgpu_verify_batch (verify_machines): many proofs checked in one call on the device.  Every verdict must be the one vgpu_verify
(verify_machine) gives the same proof alone — the first failed check in vgpu_verify's order — whatever else is in the batch."""
import ctypes as C
import random
import types

import cbor2
import pytest

import programs
from test_gpu_verify import TAMPERS, _flip

pytestmark = pytest.mark.gpu

P = 2013265921


def single(vb, cfg, proof, prep):
    try:
        vb.verify_machine(cfg, proof, prep)
        return 0
    except vb.VerificationError as e:
        return e.verdict


def tampered(proof, *whats):
    d = cbor2.loads(proof)
    for w in whats:
        (TAMPERS[w] if isinstance(w, str) else w)(d)
    return cbor2.dumps(d)


@pytest.fixture(scope="module")
def fib25(ctx, oracle):
    import valida_b200 as vb

    t = vb.run_program(vb.fib_program(25), initial_fp=0x1000)
    cfg = vb.StarkConfig(ctx, oracle.rc480)
    return vb, cfg, t, vb.prove_machine(cfg, t)


@pytest.fixture(scope="module")
def corpus(fib25, oracle):
    """(name, proof bytes, preprocessed pair) of programs with different ROMs and trace heights.  The traces objects stay in the
    fixture: their preprocessed arrays are views of memory the objects own."""
    vb, cfg, t25, p25 = fib25
    out, keep = [], []
    for n in (0, 3, 582, 9360):   # 9360: a 2^16-row CPU trace
        t = vb.run_program(vb.fib_program(n), initial_fp=0x1000)
        keep.append(t)
        out.append(("fib%d" % n, vb.prove_machine(cfg, t), t.preprocessed))
    out.append(("fib25", p25, t25.preprocessed))
    for name, prog in (("mixed", programs.mixed_program(100)), ("config5", programs.config5_program(60))):
        t = vb.run_program(prog, initial_fp=0x1000)
        keep.append(t)
        out.append((name, vb.prove_machine(cfg, t), t.preprocessed))
    prog, cells = programs.static_data_program()
    t = vb.run_program(prog, initial_fp=0x1000, static_data=cells)
    keep.append(t)
    out.append(("static_data", vb.prove_machine(cfg, t), t.preprocessed))
    out.append(("oracle_fib25", oracle.prove(t25.main, t25.preprocessed, debug_checks=False).cbor(), t25.preprocessed))
    yield out
    del keep


def test_accepts_a_mixed_corpus_in_one_call(fib25, corpus):
    vb, cfg, _, _ = fib25
    proofs = [p for _, p, _ in corpus]
    preps = [pp for _, _, pp in corpus]
    assert vb.verify_machines(cfg, proofs, preps) == [0] * len(corpus)
    order = list(range(len(corpus)))
    random.Random(7).shuffle(order)
    # shuffled, and several proofs sharing one program's traces
    proofs2 = [proofs[i] for i in order] + [proofs[4], proofs[4]]
    prog_of = [i for i in order] + [4, 4]
    assert vb.verify_machines(cfg, proofs2, preps, program_of=prog_of) == [0] * len(proofs2)


def test_tampered_proofs_interleaved_with_honest_ones(fib25):
    vb, cfg, t, proof = fib25
    batch, want = [], []
    for what in sorted(TAMPERS):
        bad = tampered(proof, what)
        batch += [proof, bad]
        want += [0, single(vb, cfg, bad, t.preprocessed)]
    assert all(w != 0 for w in want[1::2])
    got = vb.verify_machines(cfg, batch, [t.preprocessed], program_of=[0] * len(batch))
    assert got == want, [(w, g, n) for w, g, n in zip(want[1::2], got[1::2], sorted(TAMPERS)) if w != g]


def _input_path_q0(d):
    _flip(d["opening_proof"]["query_openings"][0][0]["opening_proof"][0][0])


@pytest.mark.parametrize("first,second,verdict", [
    ("input_path", "fri_path", -5),            # input path at query 7, FRI path at query 0: FRI_MERKLE
    ("input_row", "fri_sibling", -4),          # input row at query 3, FRI sibling at query 5: INPUT_MERKLE
    # an opened value of a one-row chip (not observed by the transcript; bound only by the final check of every query)
    ("one_row_chip_trace", _input_path_q0, -4),   # with the input path at query 0: INPUT_MERKLE
    ("one_row_chip_trace", "input_path", -6),     # with the input path at query 7: FRI_FINAL (query 0 fails first)
])
def test_order_of_checks(fib25, first, second, verdict):
    vb, cfg, t, proof = fib25
    bad = tampered(proof, first, second)
    assert single(vb, cfg, bad, t.preprocessed) == verdict
    assert vb.verify_machines(cfg, [proof, bad, proof], [t.preprocessed], program_of=[0, 0, 0]) == [0, verdict, 0]


def test_altered_witness_reaches_the_constraint_stage_like_vgpu_verify(fib25):
    vb, cfg, t, proof = fib25
    bad = vb.run_program(vb.fib_program(25), initial_fp=0x1000)
    row = next(i for i in range(bad.main[0].shape[0]) if bad.main[0][i, 22] == 1)
    bad.main[0][row, 22] = 0
    try:
        p = vb.prove_machine(cfg, bad)
    except vb.VgpuError:
        pytest.skip("prover refused the witness")
    want = single(vb, cfg, p, bad.preprocessed)
    assert vb.verify_machines(cfg, [proof, p], [t.preprocessed, bad.preprocessed], program_of=[0, 1]) == [0, want]


def test_malformed_and_wrong_inputs(fib25, corpus):
    vb, cfg, t, proof = fib25
    d = cbor2.loads(proof)
    d["commitments"]["main_trace"][0]["value"] = P
    malformed = [proof[:-3], b"", proof + b"\x00", cbor2.dumps(d)]
    dropped = tampered(proof, "drop_query")
    other = next(pp for name, _, pp in corpus if name == "fib582")
    batch = [proof] + malformed + [dropped, proof, proof]
    preps = [t.preprocessed, other]
    prog_of = [0] * (len(batch) - 2) + [1, 0]
    want = [0, -1, -1, -1, -1, single(vb, cfg, dropped, t.preprocessed), single(vb, cfg, proof, other), 0]
    assert want[6] != 0
    assert vb.verify_machines(cfg, batch, preps, program_of=prog_of) == want


def test_api_edges(fib25, ctx):
    import valida_b200 as vb
    from valida_b200.api import lib

    _, cfg, t, proof = fib25
    assert vb.verify_machines(cfg, [], []) == []
    L = lib()
    verdicts = (C.c_int32 * 1)()
    ptrs = (C.c_char_p * 1)(proof)
    lens = (C.c_uint64 * 1)(len(proof))
    prog = (C.c_uint32 * 1)(0)
    assert L.vgpu_verify_batch(ctx._h, None, lens, 1, None, 1, prog, 0, verdicts) != 0
    assert b"null" in L.vgpu_last_error(ctx._h)
    with pytest.raises(vb.VgpuError, match="program_of"):
        vb.verify_machines(cfg, [proof], [t.preprocessed], program_of=[1])
    fresh = vb.Context(0)   # vgpu_set_challenger never called on it
    with pytest.raises(vb.VgpuError, match="challenger"):
        vb.verify_machines(types.SimpleNamespace(ctx=fresh), [proof], [t.preprocessed])


def test_batch_of_256_matches_vgpu_verify_and_repeats(fib25):
    vb, cfg, t, proof = fib25
    rng = random.Random(2024)
    names = sorted(TAMPERS)
    batch = []
    for i in range(256):
        batch.append(tampered(proof, rng.choice(names)) if rng.random() < 0.1 else proof)
    want = [single(vb, cfg, p, t.preprocessed) for p in batch]
    assert sum(w != 0 for w in want) >= 10
    got = vb.verify_machines(cfg, batch, [t.preprocessed], program_of=[0] * 256)
    assert got == want
    assert vb.verify_machines(cfg, batch, [t.preprocessed], program_of=[0] * 256) == got
    phases = dict(vb.last_verify_batch_phases(cfg.ctx))
    assert "device checks (wall)" in phases, phases
    # vgpu_verify keeps its verdicts after batch calls on the same context
    assert single(vb, cfg, proof, t.preprocessed) == 0
    assert single(vb, cfg, tampered(proof, "fri_path"), t.preprocessed) == -5
