"""Host-side checks of ppn_parse_proposals and ppn_parse_proposals_workspace_bytes without a GPU.

Every rejection happens before anything touches a device, so the pointers are aligned fakes that are never
dereferenced; a B = 0 call with valid arguments is a no-op.
"""
import ctypes as C

import pytest

FAKE = 1 << 20                                                       # 256-byte aligned, never dereferenced


@pytest.fixture(scope="module")
def abi():
    from pytorch_pose_proposal_network_b200 import _lib
    return _lib, _lib.lib()


def cconfig(cfg):
    from pytorch_pose_proposal_network_b200.parser import _CConfig
    return _CConfig(cfg)


def humans(_lib, R=8, **moved):
    f = dict(count=FAKE, root_cell=FAKE, part_cell=FAKE, part_score=FAKE, part_box=FAKE)
    f.update(moved)
    return _lib.PPNHumans(f["count"], f["root_cell"], f["part_cell"], f["part_score"], f["part_box"], R)


def test_workspace_bytes(abi):
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    _lib, lib = abi
    cfg = PPNConfig.reference_native()
    c = cconfig(cfg)
    need = C.c_size_t()
    assert lib.ppn_parse_proposals_workspace_bytes(C.byref(c.shape(64)), C.byref(c.params), C.byref(need)) == 0
    assert need.value >= 64 * cfg.K * (cfg.HW + 1) * 4 and need.value % 256 == 0
    assert lib.ppn_parse_proposals_workspace_bytes(C.byref(c.shape(64)), C.byref(c.params), None) == -1
    assert lib.ppn_parse_proposals_workspace_bytes(None, C.byref(c.params), C.byref(need)) == -1
    assert lib.ppn_parse_proposals_workspace_bytes(C.byref(c.shape(64)), None, C.byref(need)) == -1
    p = c.params_for(0)
    p.n_nms_parts = 0                                                # not read by this entry
    assert lib.ppn_parse_proposals_workspace_bytes(C.byref(c.shape(64)), C.byref(p), C.byref(need)) == 0


def test_parse_checks(abi):
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    _lib, lib = abi
    cfg = PPNConfig.mpii16()
    c = cconfig(cfg)
    B = 4
    need = C.c_size_t()
    assert lib.ppn_parse_proposals_workspace_bytes(C.byref(c.shape(B)), C.byref(c.params), C.byref(need)) == 0

    def call(shape=None, params=None, h=None, head=FAKE, ws=FAKE, n=need.value, null=()):
        args = {"shape": C.byref(shape or c.shape(B)), "params": C.byref(params or c.params), "h": C.byref(h or humans(_lib))}
        for k in null:
            args[k] = None
        return lib.ppn_parse_proposals(head, args["shape"], args["params"], args["h"], ws, n, None)

    assert call(shape=c.shape(0)) == 0                               # B = 0: checked, nothing to do
    for k in ("shape", "params", "h"):
        assert call(null=(k,)) == -1
    assert call(head=None) == -1 and call(ws=None) == -1
    assert call(ws=FAKE + 16) == -1                                  # workspace: 256-byte aligned
    assert call(h=humans(_lib, part_box=FAKE + 4)) == -1             # boxes are written as float4
    for name in ("count", "root_cell", "part_cell", "part_score"):
        assert call(h=humans(_lib, **{name: 0})) == -1
    assert call(h=humans(_lib, R=0)) == -1
    assert call(n=need.value - 1) == -3
    assert call(shape=c.shape(B), head=FAKE + 2) == -1               # an fp32 head needs 4-byte alignment
    bad = c.shape(B)
    bad.head_dtype = 7
    assert call(shape=bad) == -1


@pytest.mark.parametrize("graphs,code", [
    ((((0, 1), (1, 0)),), -4),                                       # leads back to part 0
    ((((0,), (1,)), ((1,), (1,))), -4),                              # part 1 reached by two limbs
    ((((0, 1), (1, 2)), ((0,), (2,))), -4),                          # part 2 reached from two predecessors
])
def test_non_tree_chains_rejected(abi, graphs, code):
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    _lib, lib = abi
    c = cconfig(PPNConfig.mpii16().with_(directed_graphs=graphs))
    need = C.c_size_t()
    assert lib.ppn_parse_proposals_workspace_bytes(C.byref(c.shape(2)), C.byref(c.params), C.byref(need)) == code
    assert lib.ppn_parse_proposals(FAKE, C.byref(c.shape(2)), C.byref(c.params), C.byref(humans(_lib)), FAKE, 1 << 30,
                                   None) == code


def test_limits(abi):
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    _lib, lib = abi
    need = C.c_size_t()
    for K, rc in ((64, 0), (65, -2)):
        c = cconfig(PPNConfig(K=K, E=1, outsize=(4, 4), local_grid_size=(3, 3), directed_graphs=(((0,), (1,)),)))
        assert lib.ppn_parse_proposals_workspace_bytes(C.byref(c.shape(2)), C.byref(c.params), C.byref(need)) == rc, K
    for grid, rc in (((32, 32), 0), ((33, 32), -2)):
        c = cconfig(PPNConfig.mpii16(outsize=grid, insize=(grid[0] * 16, grid[1] * 16)))
        assert lib.ppn_parse_proposals_workspace_bytes(C.byref(c.shape(2)), C.byref(c.params), C.byref(need)) == rc, grid
    c = cconfig(PPNConfig.mpii16(outsize=(33, 32), insize=(528, 512)))
    assert lib.ppn_parse_proposals(FAKE, C.byref(c.shape(2)), C.byref(c.params), C.byref(humans(_lib)), FAKE, 1 << 30,
                                   None) == -2


def test_python_checks_without_a_call(abi):
    """PoseParser.parse_proposals shares parse's head checks (device, dtype, shape) — exercised via _check_head."""
    import torch
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    cfg = PPNConfig.mpii16()
    p = PoseParser.__new__(PoseParser)
    p.cfg = cfg
    assert p._check_head(torch.zeros(3, cfg.C, cfg.H, cfg.W)) == 3
    for bad in (torch.zeros(3, cfg.C, cfg.H, cfg.W, dtype=torch.float64), torch.zeros(3, cfg.C + 1, cfg.H, cfg.W),
                torch.zeros(cfg.C, cfg.H, cfg.W)):
        with pytest.raises(ValueError):
            p._check_head(bad)
