"""SURVEY 8f row 2 — the request codec: a pod's libconfig text <-> ``CfgTopology``
(``nhd_b200.TriadCfgParser`` on ``nhd_b200.libconfig``) against the UNMODIFIED reference class
``nhd.TriadCfgParser`` (build container; it runs on stand-ins for the absent third-party ``libconf`` /
``magicattr`` under ``oracle/_shim`` — parity of the libconfig *text layout* with the real package is
therefore unpinned, see DESIGN 8.4; parity of everything the reference class itself computes is pinned).

* generated: random Triad configs (``tests/triad_cfg.py``) — parsed topology, rewritten config text
  after a placement, GPU-map annotation, re-parse with the network section; broken configs — against
  digests of the reference's outcomes (``tests/golden/frozen/codec.json``, ``make_frozen_golden.py``);
* frozen: ``tests/golden/codec/cases.json`` made from the reference by ``make_codec_golden.py``;
* properties of the libconfig reader / writer on their own (round trip, number forms, escapes, paths).
"""
import json
import os

import numpy as np
import pytest

from nhd_b200 import libconfig
from nhd_b200.TriadCfgParser import TriadCfgParser
from tests import helpers
from tests import triad_cfg as T

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden', 'codec', 'cases.json')


def run_case(cls, text, parse_net, seed, exc_types=(Exception,)):
    """One config through one parser class -> plain-data outcome."""
    try:
        p = cls(text, False)
        top = p.CfgToTopology(parse_net)
    except exc_types as e:
        return {'raises': type(e).__name__}
    if top is None:
        return {'topology': None}
    out = {'topology': T.topo_dump(top)}
    if not parse_net and all(pg.vlan is not None for pg in top.proc_groups):
        T.assign_fake_ids(top, seed)
        out['cfg'] = p.TopologyToCfg()
        out['gpu_map'] = p.TopologyToGpuMap()
    return json.loads(json.dumps(out))


def broken_variants(text, rng):
    """Configs the reference refuses (returns None) or trips over (raises)."""
    cuts = ['cpu_arch = "ANY";', 'ext_cores_smt', 'kni_vlan = "ctrl.vlan";', 'map_type', 'Hugepages_GB',
            'helper_cores_smt', 'gpu_map', 'proc_cores_smt', 'tx_speeds', 'rx_cores', 'core0 = -1;', 'mod_defs']
    out = []
    for c in cuts:
        if c in text:
            i = text.index(c)
            j = text.index(';', i) + 1
            out.append(text[:i] + text[j:])
    out.append(text.replace('cpu_arch = "ANY"', 'cpu_arch = "Z80"'))
    out.append(text.replace('TopologyCfg', 'TopoCfg'))
    out.append(text.replace('Mod0 ', 'ModX ', 1) if 'Mod0 ' in text else text)
    out.append(text.replace('dp = ( {', 'dp = ( { rx_cores = []; }, {', 1))      # two NUMA nodes in a dp group
    out.append(text.replace('"txs", ', '', 1))                                     # nic_cores with 4 entries
    return [t for t in out if t != text]


def test_libconfig_reads_the_grammar():
    cfg = libconfig.loads('''
        a = 1; b : -2; c = 0x1F; d = 5000000000L; e = 1.5; f = -2e3; g = .5; t = TRUE; u = false;
        s = "x\\ty" "z\\x41\\"";  // adjacent literals
        grp = { inner = { deep = [1, 2, 3]; }; lst = ( 1, "two", { three = 3; }, [4.0, 5.0], () ); };
        /* block
           comment */ # hash
        last = []
    ''')
    assert (cfg.a, cfg.b, cfg.c, cfg.d, cfg.e, cfg.f, cfg.g, cfg.t, cfg.u) == (1, -2, 31, 5000000000, 1.5, -2000.0, .5, True, False)
    assert cfg.s == 'x\tyzA"'
    assert cfg.grp.inner.deep == [1, 2, 3] and isinstance(cfg.grp.lst, tuple) and cfg.grp.lst[2].three == 3
    assert cfg.grp.lst[4] == () and cfg.last == []
    assert libconfig.path_get(cfg, 'grp.lst[2].three') == 3 and libconfig.path_get(cfg, 'grp.inner.deep[-1]') == 3
    libconfig.path_set(cfg, 'grp.inner.deep[1]', 9)
    assert cfg.grp.inner.deep == [1, 9, 3]
    libconfig.path_set(cfg, 'grp.inner.fresh', 1)                # setattr on a group creates no setting
    assert 'fresh' not in cfg.grp.inner
    with pytest.raises(TypeError):
        libconfig.path_set(cfg, 'grp.lst[0]', 7)                 # lists are tuples
    with pytest.raises(AttributeError):
        libconfig.path_get(cfg, 'grp.missing')
    for bad in ('a = ;', 'a = [1, {b=2;}];', 'a = "open', 'a = 1 b', '= 3;', 'a = (1, 2;'):
        with pytest.raises(libconfig.ConfigParseError):
            libconfig.loads(bad)


def test_libconfig_round_trips():
    rng = np.random.default_rng(5)
    for seed in range(40):
        text = T.pod_to_cfg(T.codec_pod(rng, 'wild' if seed % 2 else 'mixed'), rng)
        cfg = libconfig.loads(text)
        again = libconfig.loads(libconfig.dumps(cfg))
        assert again == cfg and libconfig.dumps(again) == libconfig.dumps(cfg)
    doc = {'i': 7, 'big': 2 ** 40, 'neg': -2 ** 31, 'f': 3.0, 'e': 1e-9, 's': 'q"\\\n\x01', 'b': True,
           'l': (1, 'x', {'k': [1, 2]}, ()), 'a': [1.5, 2.5], 'empty': {}, 'strs': ['a', 'b']}
    text = libconfig.dumps(doc)
    assert 'big = 1099511627776L;' in text and 'neg = -2147483648;' in text and 'f = 3.0;' in text
    assert libconfig.loads(text) == doc
    with pytest.raises(libconfig.ConfigSerializeError):
        libconfig.dumps({'a': [1, 'x']})
    with pytest.raises(libconfig.ConfigSerializeError):
        libconfig.dumps({'a': [(1, 2)]})
    with pytest.raises(libconfig.ConfigSerializeError):
        libconfig.dumps({'a': None})


def test_codec_request_equals_directly_built_topology():
    """A generated config asks for exactly what scenarios.build_top builds for the same pod."""
    import nhd_b200.CfgTopology as cfg_mod
    from tests import scenarios
    rng = np.random.default_rng(11)
    for seed in range(60):
        pod = T.codec_pod(rng, 'mixed')
        top = TriadCfgParser(T.pod_to_cfg(pod, rng), False).CfgToTopology(False)
        want = scenarios.build_top(pod, cfg_mod)
        assert top.GetTotalGpusRequested() == want.GetTotalGpusRequested()
        assert top.GetTotalCpusRequested() == want.GetTotalCpusRequested()
        assert top.GetTotalNICsRequested() == want.GetTotalNICsRequested()
        assert (top.map_type, top.hugepages_gb, len(top.nic_core_pairing)) == \
               (want.map_type, want.hugepages_gb, len(want.nic_core_pairing))


def test_codec_reproduces_golden():
    with open(GOLDEN) as f:
        cases = json.load(f)
    assert len(cases) >= 150
    kinds = {'topology': 0, 'none': 0, 'raises': 0}
    for i, c in enumerate(cases):
        got = run_case(TriadCfgParser, c['text'], c['parse_net'], c['seed'])
        assert got == c['expected'], (i, c['note'])
        kinds['raises' if 'raises' in got else 'none' if got['topology'] is None else 'topology'] += 1
    assert kinds['topology'] > 80 and kinds['none'] > 20 and kinds['raises'] > 5, kinds


def generated_cases():
    """(seed, config text, broken variants of it) in the order the frozen outcomes follow."""
    rng = np.random.default_rng(77)
    for seed in range(120):
        pod = T.codec_pod(rng, 'wild' if seed % 2 else 'mixed')
        text = T.pod_to_cfg(pod, rng, gpu_type=[None, 'V100', 'bogus'][seed % 3])
        yield seed, text, broken_variants(text, rng) if seed % 4 == 0 else []


def test_codec_matches_live_reference():
    """Generated configs against digests (``tests.helpers.digest``) of the reference's outcomes, frozen by
    ``tests/golden/make_frozen_golden.py``: the parsed config, the rewritten config read back with its network
    section (a deployed pod after a restart), and broken variants."""
    frozen = helpers.frozen('codec')
    n = texts = 0
    for (seed, text, broken), want in zip(generated_cases(), frozen, strict=True):
        got = run_case(TriadCfgParser, text, False, seed)
        assert helpers.digest(got) == want['parsed'], (seed, got)
        assert got['topology'] is not None
        texts += 1
        got2 = run_case(TriadCfgParser, got['cfg'], True, seed)
        assert helpers.digest(got2) == want['reparsed'] and got2['topology'] is not None, (seed, got2)
        ids = [c[4] for g in got2['topology']['groups'] for c in g['proc'] + g['helpers']]
        assert all(x > 0 for x in ids)                           # physical ids survived the trip
        assert [helpers.digest(run_case(TriadCfgParser, bad, False, seed)) for bad in broken] == want['broken'], seed
        n += len(broken)
    assert texts == 120 and n > 200
