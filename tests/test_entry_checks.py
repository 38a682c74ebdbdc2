"""What the entry points share: the one check of a many-block list (u64 offsets, so that no sum wraps) and the per-call
bookkeeping behind dark_bwt_stats."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def torch():
    import torch as t
    if not t.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    return t


@pytest.fixture(scope="module")
def saca():
    from dark_b200 import saca as s
    return s


# 0xFFFFFFFE + 2 wraps to 0 in u32: offsets that a u32 check `starts[k + 1] < starts[k] + 2` lets through
WRAPPED = {"wrap_to_zero": [0, 0xFFFFFFFE, 0], "wrap_then_block": [0, 0xFFFFFFFE, 0, 10]}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(WRAPPED))
def test_wrapped_offsets_are_refused_by_every_device_many_entry(saca, oracle, torch, name):
    """The three device many-block entries read the same offsets back and refuse them alike (DARK_BWT_E_INVALID_N), and the
    context then transforms a valid list."""
    from dark_b200 import _ffi
    starts = WRAPPED[name]
    count = len(starts) - 1
    cap = 1 << 16
    with saca.Constructor(cap, flags=_ffi.F_DEVICE_ONLY) as con:
        data = torch.zeros(cap, dtype=torch.uint8, device="cuda")
        out = torch.zeros(cap, dtype=torch.uint8, device="cuda")
        ds = torch.from_numpy(np.array(starts, np.uint32).view(np.int32)).cuda()  # int32 -2 is 0xFFFFFFFE
        do = torch.zeros(count, dtype=torch.int64, device="cuda")
        calls = {
            "forward_many_device": lambda: con.bwt_many_device(data.data_ptr(), ds.data_ptr(), count, out.data_ptr(), do.data_ptr()),
            "inverse_many_device": lambda: con.inverse_many_device(data.data_ptr(), ds.data_ptr(), do.data_ptr(), count, out.data_ptr()),
            "dc_encode_many_device": lambda: con.dc_encode_many_device(data.data_ptr(), ds.data_ptr(), count),
        }
        codes = {}
        for entry, call in calls.items():
            with pytest.raises(_ffi.DarkBwtError) as e:
                call()
            codes[entry] = e.value.code
        assert codes == {entry: _ffi.E_INVALID_N for entry in calls}

        blocks = [b"abracadabra", b"banana", b"mississippi"]
        good = np.concatenate([[0], np.cumsum([len(b) for b in blocks])]).astype(np.uint32)
        dt = torch.frombuffer(bytearray(b"".join(blocks)), dtype=torch.uint8).cuda()
        ds = torch.from_numpy(good.view(np.int32)).cuda()
        do = torch.zeros(len(blocks), dtype=torch.int64, device="cuda")
        con.bwt_many_device(dt.data_ptr(), ds.data_ptr(), len(blocks), out.data_ptr(), do.data_ptr())
        hb, ho = out[:int(good[-1])].cpu().numpy(), do.cpu().numpy()
    for k, b in enumerate(blocks):
        bwt_o, origin_o = oracle.bwt_forward(np.frombuffer(b, np.uint8))
        assert np.array_equal(hb[good[k]:good[k + 1]], bwt_o) and int(ho[k]) == origin_o, k


@pytest.mark.gpu
def test_forward_many_host_syncs_do_not_depend_on_earlier_calls(saca, oracle, torch):
    """dark_bwt_forward_many reports the round trips of its own call: the same on a fresh context, after a single-block
    forward and after an inverse on the same context, and at least one per round plus the alphabet scan and the end."""
    from dark_b200 import synth
    blocks = [synth.generate("text", 40 + k, 3000 + 500 * k) for k in range(6)]
    big = synth.generate("mixed", 7, 200_000)

    def many(con):
        outs = con.bwt_many(blocks)
        st = con.stats.as_dict()
        return outs, st["host_syncs"], st["rounds"]

    with saca.Constructor(1 << 18) as con:
        runs = [many(con)]
        bwt, origin = con.bwt(big)
        runs.append(many(con))
        assert np.array_equal(con.inverse(bwt, origin), big)
        runs.append(many(con))
    syncs = [s for _, s, _ in runs]
    rounds = runs[0][2]
    assert rounds >= 1 and all(r == rounds for _, _, r in runs)
    assert syncs[0] == syncs[1] == syncs[2], syncs
    assert syncs[0] >= rounds + 2, (syncs[0], rounds)
    for outs, _, _ in runs:
        for (b, o), t in zip(outs, blocks):
            bwt_o, origin_o = oracle.bwt_forward(t)
            assert o == origin_o and np.array_equal(b, bwt_o)
