"""Differential tests on drawn blocks (hypothesis): three implementations that share no code for the trie mutations.

  model    the final state as the GENERATOR tracked it (plain dicts), hashed as the canonical Merkle-Patricia trie of its
           items by a recursive pure-Python builder (trie_model.py): no insert, no delete, no collapse rule — a trie's shape is a function
           of its key set, so whatever sequence of inserts / deletes (with branch collapse, extension merge) led there must
           hash to the same root;
  oracle   the CPU restatement of the reference (insert / delete on pointer tries, per-txn subsets);
  product  the library through the C ABI: the txn loop on the device (path copies on the arena), and its host loop.

The model pins the oracle's mutation semantics for witnesses that carry the whole state (virtual_depth = 0); the product
is compared with the oracle on those and on witnesses whose siblings are hashed out (deletes next to Hash nodes)."""
import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

from proof_protocol_decoder_b200 import flat, synth
from trie_model import trie_root

EMPTY_CODE_HASH = synth.keccak256(b"")


def model_state_root(blk):
    state = {}
    for acc in blk.final_accounts:
        if not acc["alive"]:
            continue  # self-destructed: deleted from the state trie (decoding.rs:271-282)
        storage = {hk: synth.rlp_int(v) for (hk, v) in acc["slots"].values()}
        code_hash = acc.get("code_hash") if acc["contract"] else None
        state[acc["haddr"]] = synth.rlp_list([synth.rlp_int(acc["nonce"]), synth.rlp_int(acc["balance"]), synth.rlp_str(trie_root(storage)),
                                              synth.rlp_str(code_hash or EMPTY_CODE_HASH)])
    return trie_root(state)


block_params = st.fixed_dictionaries(
    {
        "seed": st.integers(0, 1 << 30),
        "n_accounts": st.integers(2, 40),
        "n_txns": st.integers(2, 10),
        "contract_frac": st.floats(0.2, 1.0),
        "slots_hi": st.integers(1, 24),
        "apt_hi": st.integers(2, 12),
        "writes_hi": st.integers(1, 12),
        "zero_write_frac": st.floats(0.0, 0.9),  # deletes: branches collapse, extensions merge, tries empty out
        "new_accounts": st.booleans(),
    }
)


def _gen(p, virtual_depth=0):
    return synth.gen_block(
        p["seed"], n_accounts=p["n_accounts"], n_txns=p["n_txns"], contract_frac=p["contract_frac"], slots_hi=p["slots_hi"],
        accounts_per_txn=(1, p["apt_hi"]), slot_reads=(0, 4), slot_writes=(0, p["writes_hi"]), zero_write_frac=p["zero_write_frac"],
        virtual_depth=virtual_depth, allow_new_accounts=p["new_accounts"] and virtual_depth == 0, allow_self_destruct=True, inline_code_frac=0.5,
    )


def test_model_trie_root_known_answers(goldens):
    # the builder itself, against the reference's constant and a one-leaf trie hashed by hand
    assert trie_root({}).hex() == "56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421"
    key = bytes(range(32))
    raw = synth.rlp_list([synth.rlp_str(b"\x20" + key), synth.rlp_str(b"\x2a")])
    assert trie_root({key: b"\x2a"}) == synth.keccak256(raw)


@settings(max_examples=30, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])
@given(p=block_params)
def test_oracle_final_state_root_is_the_canonical_trie_of_the_final_state(oracle, p):
    blk = _gen(p)
    irs = flat.parse_ir_dump(oracle.block_decode(blk.flat))
    assert len(irs) == p["n_txns"]
    assert irs[-1]["trie_roots_after"]["state_root"] == model_state_root(blk)


@pytest.mark.gpu
@settings(max_examples=25, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])
@given(p=block_params, vd=st.integers(0, 3))
def test_device_loop_and_host_loop_match_oracle_on_drawn_blocks(oracle, p, vd):
    import os

    from ppd_oracle_lib import OracleError
    from proof_protocol_decoder_b200.lib import Context, PpdError

    blk = _gen(p, virtual_depth=vd)
    try:
        want = oracle.block_decode(blk.flat)
    except OracleError as e:
        want = e.code
    ctx = _ctx()
    for host_txn in (False, True):
        saved = os.environ.pop("PPD_HOST_TXN", None)
        if host_txn:
            os.environ["PPD_HOST_TXN"] = "1"
        try:
            try:
                got = ctx.block_decode(blk.flat)
            except PpdError as e:
                got = e.code
            loops = ctx.stats()["txn_loops_on_gpu"]
        finally:
            os.environ.pop("PPD_HOST_TXN", None)
            if saved is not None:
                os.environ["PPD_HOST_TXN"] = saved
        assert got == want, f"{'host' if host_txn else 'device'} txn loop differs from the oracle"
        if not host_txn and not isinstance(want, int):
            assert loops == 1
    if vd == 0 and not isinstance(want, int):
        assert flat.parse_ir_dump(want)[-1]["trie_roots_after"]["state_root"] == model_state_root(blk)


_CTX = []


def _ctx():
    if not _CTX:
        from proof_protocol_decoder_b200.lib import Context

        _CTX.append(Context(0))
    return _CTX[0]
