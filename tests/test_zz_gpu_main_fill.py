"""GPU run of MasterMainTable::new + pad from the AET (master_table.rs:881-974; csrc/main_fill.cu): the device tables against
the oracle's table fill, the RAM table's Bezout coefficient polynomials (ram.rs:162-214) against the oracle and — at sizes
where the two-pass transforms are reached — against their defining identity, and tvm_prove_aet against tvm_prove_tables on
the oracle's tables (identical proof words).  The same stage bodies are checked on the host by tests/test_main_fill_host.py;
this file sorts last: its kernels are the newest."""
import numpy as np
import pytest

import tvm_b200
from oracle import tracegen as tg

import test_vm_programs as tvp
from test_main_fill_host import _program, _ev, host  # noqa: F401 - `host` is the fixture that builds the host harness

pytestmark = pytest.mark.gpu
P = tg.P


@pytest.mark.parametrize("m", [1, 2, 3, 33, 100])
def test_device_bezout_coefficients_match_the_oracle(backend, m):
    rng = np.random.default_rng(7000 + m)
    roots = list(dict.fromkeys([0, 1, P - 1][:min(m, 3)] + [int(x) for x in rng.integers(0, P, size=max(0, m - 3), dtype=np.uint64)]))
    a, b = backend.bezout_coefficients(roots)
    want_a, want_b = tg.bezout_coefficients(roots)
    assert [int(v) for v in a] == want_a and [int(v) for v in b] == want_b


@pytest.mark.parametrize("m", [5000, 70001, 300000])
def test_device_bezout_identity(backend, m):
    """a rp + b rp' = 1, deg a < m - 1: sizes whose transforms span one pass (<= 2^13) and two passes"""
    rng = np.random.default_rng(m)
    roots = np.unique(np.concatenate([np.arange(1 << 20, (1 << 20) + m // 2, dtype=np.uint64),       # an array in RAM
                                      rng.integers(0, P, size=m - m // 2, dtype=np.uint64)]))
    rng.shuffle(roots)
    a, b = backend.bezout_coefficients(roots)
    assert int(a[-1]) == 0
    al, bl, rl = [int(v) for v in a], [int(v) for v in b], [int(v) for v in roots]
    for z in (3, P - 2):
        rp, fd = 1, 0
        for r in rl:
            fd = (fd * (z - r) + rp) % P
            rp = rp * (z - r) % P
        assert (_ev(al, z) * rp + _ev(bl, z) * fd) % P == 1


@pytest.mark.parametrize("name,extra", [("halt", 0), ("fib_100", 0), ("fib_100", 1), ("spin_9", 0), ("u32_mix", 0), ("verifier_3", 0),
                                        ("verifier_40", 0)])
def test_device_tables_from_the_aet_match_the_oracle(backend, name, extra):
    program, inp, ram = _program(name)
    ex = tg.execute(list(program), inp, (), ram)
    n = max(256, tg.padded_height(list(program), inp, (), ram)) << extra
    want, _, _ = tg.main_table(list(program), inp, n, (), ram)
    got, lengths = backend.main_table_from_aet(tg.aet_arrays(list(program), ex), n)
    bad = [c for c in range(379) if not np.array_equal(got[c], want[c])]
    assert not bad, [tg.column_name(True, c) for c in bad[:8]]
    heights = tg.table_heights(list(program), ex)
    assert lengths == [heights[k] for k in ("program", "processor", "op_stack", "ram", "jump_stack", "hash", "cascade", "lookup", "u32")]


@pytest.mark.parametrize("name,ldt", [("fib_100", "fri"), ("verifier_3", "stir"), ("verifier_40", "fri")])
def test_prove_from_the_aet_equals_prove_from_the_tables(backend, name, ldt):
    src, inp, ram = tvp._workload(name)
    inst = tvp.program_instance(src, inp, 8, ldt, ram=ram)
    words = tg.assemble(src)
    ex = tg.execute(words, inp, (), ram)
    claim = inst["claim"]
    args = (inst["main_rand"], inst["aux_rand"], inst["randomizer_column"], inst["quot_rand"])
    kw = dict(security_level=8, log2_expansion=2, padded_height=inst["padded_height"],
              ldt_choice=tvm_b200.LDT_FRI if ldt == "fri" else tvm_b200.LDT_STIR)
    c = (claim.program_digest, claim.input, claim.output)
    from_tables = backend.prove_tables(c, inst["main"], *args, **kw)
    from_aet = backend.prove_aet(c, tg.aet_arrays(words, ex), *args, **kw)
    assert np.array_equal(from_tables, from_aet)
    assert tvm_b200.verify(c, from_aet, 8, 2, ldt_choice=kw["ldt_choice"]) == (True, "")      # incl. the AIR


def test_aet_with_a_table_above_the_height_is_rejected(backend):
    program, inp, ram = _program("fib_100")
    ex = tg.execute(list(program), inp, (), ram)
    with pytest.raises(tvm_b200.TvmError):
        backend.main_table_from_aet(tg.aet_arrays(list(program), ex), 256)


def test_plain_c_aet_client_proves_halt_on_the_gpu(tmp_path):
    """examples/prove_aet.c: same proof words as examples/prove_tables.c on the same randomness (the tables of `halt`)"""
    import subprocess
    from test_native_verifier import _build_example, _write_prove_tables_dir, _write_aet_files
    digest = _write_prove_tables_dir(tmp_path)
    _write_aet_files(tmp_path)
    for name in ("prove_aet", "prove_tables"):
        r = subprocess.run([_build_example(tmp_path, name), str(tmp_path)], capture_output=True, text=True)
        assert r.returncode == 0 and "verified" in r.stdout, r.stderr
    from_aet = np.fromfile(str(tmp_path / "proof_aet.u64"), dtype="<u8")
    assert np.array_equal(from_aet, np.fromfile(str(tmp_path / "proof.u64"), dtype="<u8"))
    assert tvm_b200.verify((digest, [], []), from_aet, 8, 2, ldt_choice=tvm_b200.LDT_FRI) == (True, "")


@pytest.mark.parametrize("k", [13, 16, 18])
def test_device_fill_equals_the_host_executor_on_a_synthetic_aet(backend, host, k):
    """Sizes no program of the test suite reaches (2^16 rows: 2^15 RAM rows over 2^14 unique pointers -> subproduct tree of 14
    levels with the transform paths, radix sorts of 2^16 keys, 44 000 u32 rows): the CUDA executor against the sequential
    host executor running the same stage bodies (tests/host/main_fill_host.cu, itself checked against the oracle on real
    programs by tests/test_main_fill_host.py)."""
    import os
    from test_main_fill_host import host_main_table
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "tools", "fill_time.py")).read().split("b = tvm_b200.Backend(0)")[0]
    ns = {"__file__": os.path.join(root, "tools", "fill_time.py")}
    exec(compile(src, "fill_time", "exec"), ns)
    aet = ns["synthetic_aet"](k, np.random.default_rng(k))
    want, want_lengths = host_main_table(host, aet, 1 << k)
    got, lengths = backend.main_table_from_aet(aet, 1 << k)
    assert lengths == want_lengths
    bad = [c for c in range(149) if not np.array_equal(got[c], want[c])]
    assert not bad, [tg.column_name(True, c) for c in bad[:8]]
