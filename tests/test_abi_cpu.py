"""CPU-side checks of the C-ABI library: it loads and exports every symbol that
include/*.h declares.  No compute call is made (there is no GPU here)."""
import ctypes

from parelag_b200 import capi


def test_library_exports_every_declared_symbol():
    lib = capi.lib()
    names = capi.declared_symbols()
    assert len(names) > 30
    assert "pe_api_solver_replay_mode" in names
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, "declared in include/*.h but not exported: %s" % missing


def test_no_cpu_fallback_without_device():
    import torch
    if torch.cuda.is_available():
        return
    try:
        capi.Ctx()
    except capi.PEError as e:
        assert "no CUDA device" in str(e) or "CUDA" in str(e)
    else:
        raise AssertionError("context creation must fail loudly without a CUDA device")


def _header_enum(first, last):
    """name -> value of an enum in include/parelag_b200.h, from `first` to `last`"""
    import re
    text = open(capi.HEADER_PATHS[1]).read()
    body = text[text.index(first):text.index(last)]
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"PE_(?:VARIANT|TUNE)_(\w+)\s*=\s*(\d+)", body)}


def test_variant_counter_slots_match_the_header():
    """capi's slot constants are the header's enum; the counters are host integers, readable and resettable without a
    device"""
    slots = _header_enum("PE_VARIANT_SPMV_SELL", "int pe_variant_counts")
    assert slots.pop("COUNT") == len(capi.VARIANT_SLOTS)
    assert slots == {name: getattr(capi, name) for name in capi.VARIANT_SLOTS}
    assert [slots[n] for n in capi.VARIANT_SLOTS] == list(range(len(capi.VARIANT_SLOTS)))
    # the SELL entry-group slots: one per (kernel, G, single) choice, in the order sell_group_slot (pe_sell.cu) indexes
    for kernel in ("gs", "spmv"):
        for G in (4, 8, 12):
            for single in (True, False):
                name = "SELL_%s_G%d_%s" % (kernel.upper(), G, "SINGLE" if single else "PIPE")
                assert capi.sell_group_slot(kernel, G, single) == slots[name], name
    capi.variant_counts(reset=True)
    assert not capi.variant_counts().any()
    tune = _header_enum("PE_TUNE_SELL_MIN_ROWS", "int pe_set_tuning")
    assert tune["LOCAL_SMEM_BYTES"] == capi.TUNE_LOCAL_SMEM_BYTES and tune["COUNT"] == capi.TUNE_LOCAL_SMEM_BYTES + 1
    assert capi.get_tuning(capi.TUNE_LOCAL_SMEM_BYTES) == 0


def test_replay_mode_values_match_the_header():
    """the mode names api.Solver.replay_mode() returns are keyed by the header's PE_REPLAY_* values"""
    import re
    text = open(capi.HEADER_PATHS[2]).read()
    vals = {m.group(1): int(m.group(2)) for m in re.finditer(r"PE_REPLAY_(\w+)\s*=\s*(\d+)", text)}
    assert vals == {"DIRECT": capi.REPLAY_DIRECT, "GRAPH": capi.REPLAY_GRAPH, "PROGRAM": capi.REPLAY_PROGRAM}
    assert sorted(capi.REPLAY_MODE_NAMES) == sorted(vals.values())
