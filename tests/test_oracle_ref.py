"""CPU: the oracle and the graph reader against what the reference's own object code produced,
stored in tests/golden/ref_checks.json (struct layout, answers to seeded random searches, graphs its
CLI wrote under the committed seeds with their DOT conversions) and tests/golden/sboxes/ (its S-box
tables).  oracle/gen_golden.py regenerates both from the reference."""
import json
import os
import re
import tempfile

import pytest

import _support as S
from sboxgates_b200 import graph as G

SBOXES = os.path.join(S.GOLDEN, "sboxes")


@pytest.fixture(scope="module")
def ref():
    return json.load(open(os.path.join(S.GOLDEN, "ref_checks.json")))


def _graphs(ref, key):
    return next(g for g in ref["graphs"] if g["key"] == key)


def test_struct_layout_the_shim_assumes(ref):
    lay = ref["layout"]
    assert (lay["ttable"], lay["gate"], lay["state"], lay["state_gates_offset"]) == \
        (32, 64, 32032, 32)   # state.h:64-88
    # the node-level shim (lut_search) also reads three fields of `options` (sboxgates.h:49-66)
    assert (lay["options_randomize_offset"], lay["options_lut_graph_offset"],
            lay["options_verbosity_offset"], lay["options"], lay["boolfunc"]) == \
        (2019, 2018, 9756, 9760, 24)


def test_oracle_equals_reference_on_random_cases(ref):
    want = ref["searches"]
    cases = list(S.random_ref_cases())
    assert len(cases) == len(want) == 60
    for i, ((which, tabs, tgt, mask, inb, seed), w) in enumerate(zip(cases, want)):
        assert which == w["which"]
        a = S.OrcRng.from_seed(seed)
        found_o, ret_o, _ = S.oracle_search(which, tabs, tgt, mask, inb, a)
        assert (found_o, ret_o) == (bool(w["found"]), w["ret"]), (i // 2, which)
        assert a.draws == w["draws"] and a.words() == [int(x) for x in w["rng_after"]]
        assert a.p == w["rng_p"]


def test_reference_cli_reproduces_golden_file_names(ref):
    names = json.load(open(os.path.join(S.GOLDEN, "xml_names.json")))
    for key in ("crypto1_fa.txt -l seed1", "crypto1_fc.txt -l seed2"):
        run = _graphs(ref, key)
        assert run["names"] == names[key]
        # the stored files are those the run wrote, and each is a correct circuit for its S-box
        assert [f["name"] for f in run["files"]] == run["names"]
        sbox, _ = G.load_sbox(os.path.join(SBOXES, key.split()[0]))
        for f in run["files"]:
            g = _load_text(f["xml"])
            assert G.verify_graph(g, sbox, require_bits=[0]) == [0]
            assert g.num_luts == int(f["name"].split("-")[1])


def test_rijndael_table_is_the_aes_sbox():
    txt = open(os.path.join(SBOXES, "rijndael.txt")).read().split()
    assert [int(x, 16) for x in txt] == S.rijndael_sbox()


def _load_text(xml):
    with tempfile.NamedTemporaryFile("w", suffix=".xml", delete=False) as fp:
        fp.write(xml)
    try:
        return G.load_graph(fp.name)
    finally:
        os.unlink(fp.name)


def _dot_topology(dot):
    """(labels by gate, inputs by gate in edge order, outputs) of the reference's -d output."""
    labels = {int(m.group(1)): m.group(2) for m in re.finditer(r'gt(\d+) \[label="([^"]*)"\];', dot)}
    inputs = {g: [] for g in labels}
    outputs = {}
    for m in re.finditer(r"gt(\d+) -> (gt|out)(\d+);", dot):
        if m.group(2) == "out":
            outputs[int(m.group(3))] = int(m.group(1))
        else:
            inputs[int(m.group(3))].append(int(m.group(1)))
    return labels, inputs, outputs


def _label(gate, index):
    if gate.type == "IN":
        return "IN %d" % index
    return "0x%02x" % gate.function if gate.type == "LUT" else gate.type


def test_saved_graph_loads_back_and_converts(ref):
    """The XML the reference writes, read by the Python loader (sboxgates_b200/graph.py), gives the
    topology the reference's own loader gives (its DOT conversion, -d) and a correct circuit -- for
    a LUT graph (--lut) and a 2-input-gate graph."""
    for key, sbox_file in (("crypto1_fc.txt -l seed1", "crypto1_fc.txt"),
                           ("des_s1.txt -o 0 seed1", "des_s1.txt")):
        f = _graphs(ref, key)["files"][-1]
        assert "digraph sbox" in f["dot"] and "-> gt" in f["dot"]
        g = _load_text(f["xml"])
        labels, inputs, outputs = _dot_topology(f["dot"])
        assert len(labels) == len(g.gates)
        for i, gate in enumerate(g.gates):
            assert (labels[i], inputs[i]) == (_label(gate, i), gate.inputs), (key, i)
        assert outputs == g.outputs
        sbox, _ = G.load_sbox(os.path.join(SBOXES, sbox_file))
        assert G.verify_graph(g, sbox, require_bits=[0]) == [0]
        if "-l" in key.split():
            assert g.num_luts == int(f["name"].split("-")[1])
