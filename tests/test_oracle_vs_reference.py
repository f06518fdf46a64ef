"""Differential test: the C oracle against what the UNMODIFIED reference modules computed for the same seeded
scenarios, frozen in tests/golden/frozen/oracle_vs_reference.json (tests/golden/make_frozen_golden.py).  This is
the pin that makes the oracle trustworthy; fuller frozen copies of such runs are tests/golden/*.json."""
import pytest

from tests import helpers, ref_compare, scenarios

FLAVORS = ['mixed', 'wild', 'vf', 'big']


def flavor_scenarios(flavor):
    for seed in range(30):
        yield seed, scenarios.random_scenario(seed * 7 + {'mixed': 1, 'wild': 2, 'vf': 3, 'big': 4}[flavor] * 100003,
                                              n_nodes=6, n_pods=30, flavor=flavor)


def limit_scenarios():
    for seed in range(3):
        scn = scenarios.huge_scenario(81000 + seed, min_busy_secs=30.0 if seed % 3 else 0.0)
        scn['nodes'], scn['pods'], scn['now'] = scn['nodes'][:5], scn['pods'][:14], scn['now'][:14]
        yield seed, scn


def label_scenarios():
    for seed in range(40):
        yield seed, scenarios.random_scenario(4242 + seed, n_nodes=5, n_pods=1, flavor='wild' if seed % 2 else 'vf')


def node_view(x):
    """What ParseLabels made of a node's labels, as plain data."""
    return [[(c.core, c.socket, c.sibling, c.used) for c in x.cores],
            [(g.device_id, g.numa_node, g.pciesw, g.gtype.value) for g in x.gpus],
            [(n.ifname, n.mac, n.speed, n.numa_node, n.pciesw, n.idx, n.card, n.port) for n in x.nics],
            (x.groups, x.maintenance, x.data_vlan, x.gwip, x.mem.free_hugepages_gb, x.reserved_cores,
             x.sockets, x.numa_nodes, x.smt_enabled, x.cores_per_proc)]


def _check_stream(oracle_lib, scn, want, tag):
    """want: the reference's outcome per pod (ref_compare.freeze_outcomes) and digests of its initial and final
    packed records."""
    recs, pods, now, layout = ref_compare.pack_scenario(scn)
    # the packer gives identical records from the reference's Node objects and from the mirrors
    assert helpers.digest(recs) == want['init'], tag
    b, orecs = oracle_lib.solve(recs, layout.speed_table(), pods, now, min_busy_secs=scn['min_busy_secs'])
    errs = ref_compare.diff_frozen_outcomes(want['outcomes'], b)
    assert not errs, (tag, errs)
    assert helpers.digest(orecs) == want['final'], tag
    return len(b), want['outcomes'][0].count('p')


@pytest.mark.parametrize('flavor', FLAVORS)
def test_oracle_matches_live_reference(oracle_lib, flavor):
    frozen = helpers.frozen('oracle_vs_reference')['flavors'][flavor]
    attempts = placed = 0
    for (seed, scn), want in zip(flavor_scenarios(flavor), frozen, strict=True):
        a, p = _check_stream(oracle_lib, scn, want, (flavor, seed))
        attempts += a
        placed += p
    assert attempts == 900 and placed > 150


def test_mirror_node_ingest_matches_reference_labels():
    """nhd_b200.Node.ParseLabels builds the same node as nhd.Node.ParseLabels (Node.py:312-487)."""
    import nhd_b200.Node as mirror
    frozen = helpers.frozen('oracle_vs_reference')['labels']
    n = 0
    for (seed, scn), want in zip(label_scenarios(), frozen, strict=True):
        got = {name: helpers.digest(node_view(x)) for name, x in scenarios.build_nodes(scn, mirror).items()}
        assert got == want, seed
        n += len(got)
    assert n == 200


def test_oracle_matches_live_reference_near_the_limits(oracle_lib):
    """Nodes with up to 256 logical cores / 16 GPUs / 32 NICs / 4 NUMA nodes and pods with up to 72 cores: the
    reference itself is slow here (seconds per pod), so a few short streams."""
    frozen = helpers.frozen('oracle_vs_reference')['limits']
    attempts = placed = 0
    for (seed, scn), want in zip(limit_scenarios(), frozen, strict=True):
        a, p = _check_stream(oracle_lib, scn, want, seed)
        attempts += a
        placed += p
    assert attempts == 42 and placed > 20
