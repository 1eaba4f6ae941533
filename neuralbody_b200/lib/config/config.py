"""Config surface of the render hot path.

Mirrors the keys the reference reads inside the path (lib/config/config.py:9-129 +
the yaml-only keys of configs/snapshot_exp/snapshot_f3c.yaml:55-78):
  N_samples, perturb, raw_noise_std, white_bkgd   if_clight_renderer.py:13,16,82
  voxel_size                                      latent_xyzc.py:54
  xyz_res, view_res                               embedder.py:53-54
  num_train_frame                                 latent_xyzc.py:16
  H, W, ratio, N_rand, chunk
  mesh_th                                         if_mesh_renderer.py:47
  network_module/path, renderer_module/path       make_network.py / make_renderer.py
Same yaml format (`parent_cfg` inheritance, config.py:149-152) and the same trailing
`KEY VALUE` override form (config.py:153).  Unlike upstream nothing is parsed from
sys.argv at import time and open3d is not imported.
"""
import ast
import copy
import os

import yaml

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


class CfgNode(dict):
    """Attribute-style dict; nested dicts become CfgNodes (a minimal stand-in for yacs)."""

    def __init__(self, init=None):
        super().__init__()
        for k, v in (init or {}).items():
            self[k] = CfgNode(v) if isinstance(v, dict) and not isinstance(v, CfgNode) else v

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError:
            raise AttributeError(name)

    def __setattr__(self, name, value):
        self[name] = CfgNode(value) if isinstance(value, dict) and not isinstance(value, CfgNode) else value

    def clone(self):
        return copy.deepcopy(self)

    def merge_from_other_cfg(self, other):
        for k, v in other.items():
            if isinstance(v, dict) and isinstance(self.get(k), dict):
                self[k].merge_from_other_cfg(v)
            else:
                self[k] = CfgNode(v) if isinstance(v, dict) and not isinstance(v, CfgNode) else copy.deepcopy(v)

    def merge_from_file(self, path):
        with open(path, "r") as f:
            cur = yaml.safe_load(f) or {}
        if "parent_cfg" in cur:
            parent = cur["parent_cfg"]
            if not os.path.isabs(parent) and not os.path.exists(parent):
                parent = os.path.join(os.path.dirname(path), os.path.basename(parent))
            self.merge_from_file(parent)
        self.merge_from_other_cfg(cur)

    def merge_from_list(self, opts):
        opts = list(opts or [])
        if len(opts) % 2:
            raise ValueError("override list must be KEY VALUE pairs, got %r" % (opts,))
        for key, val in zip(opts[0::2], opts[1::2]):
            node = self
            parts = key.split(".")
            for p in parts[:-1]:
                node = node.setdefault(p, CfgNode())
            if isinstance(val, str):
                try:
                    val = ast.literal_eval(val)
                except (ValueError, SyntaxError):
                    pass
            node[parts[-1]] = val


def _defaults():
    c = CfgNode()
    c.task = "if_nerf"
    c.exp_name = "synth_313"
    c.gpus = [0]
    # plugin selection (make_network.py:5-9 / make_renderer.py:5-9)
    c.network_module = "neuralbody_b200.lib.networks.latent_xyzc"
    c.network_path = os.path.join(_PKG_ROOT, "lib/networks/latent_xyzc.py")
    c.renderer_module = "neuralbody_b200.lib.networks.renderer.if_nerf_renderer"
    c.renderer_path = os.path.join(_PKG_ROOT, "lib/networks/renderer/if_nerf_renderer.py")
    # rendering options (snapshot_f3c.yaml:55-66)
    c.xyz_res = 10
    c.view_res = 4
    c.raw_noise_std = 0
    c.N_samples = 64
    c.N_importance = 128
    c.N_rand = 1024
    c.perturb = 1
    c.white_bkgd = False
    c.num_render_views = 50
    # data options (config.py:14-36, latent_xyzc_313.yaml:74-79)
    c.H = 1024
    c.W = 1024
    c.ratio = 0.5
    c.num_train_frame = 60
    c.voxel_size = [0.005, 0.005, 0.005]
    c.big_box = False
    # mesh extraction (config.py:44-45; the 313 / snapshot yamls set 5 in mesh_cfg)
    c.mesh_th = 50
    # B200 renderer options (new)
    c.render_precision = "tc_fp16x3"    # "fp32" exact FFMA kernel | "tc_fp16x3" tcgen05, 3-pass hi/lo density path
                                        # (meets the 1e-3 parity gate) | "tc_fp16" tcgen05 1-pass (fastest, ~4e-3 on depth)
    c.render_volume_dtype = "auto"      # "auto": fp16 volume for tc_fp16, fp32 otherwise
    c.render_skip_empty = True          # tensor-core modes: exact empty-sample skipping (bit-identical outputs)
    c.render_return_weights = True      # 'weights' (B,n,S) is unused downstream; may be skipped
    c.render_train_precision = 'tc_tf32x3'   # calls autograd records: 'tc_tf32x3' (tcgen05 TF32 GEMM chains over the sample list) | 'fp32' (exact FFMA kernels)
    c.render_importance = 0             # f-4: > 0 adds a fine pass with this many importance samples (upstream's N_importance is a dead key for Neural Body, so the default stays single-pass)
    c.chunk = 0                         # 0 = all rays of the call in one launch
    return c


cfg = _defaults()


def make_cfg(cfg_file=None, opts=None, target=None):
    """Build (in place) a config from defaults + yaml (+ parent_cfg) + KEY VALUE overrides."""
    c = target if target is not None else cfg
    if cfg_file:
        c.merge_from_file(cfg_file)
    c.merge_from_list(opts)
    return c


def get_active_cfg():
    """When running inside the reference process (its `lib.config` already imported, e.g. the
    renderer was selected through the reference's own make_renderer), read the reference's
    singleton so yaml/CLI overrides made there are honoured; otherwise use ours."""
    import sys
    mod = sys.modules.get("lib.config")
    if mod is not None and hasattr(mod, "cfg"):
        return mod.cfg
    return cfg
