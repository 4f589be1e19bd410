"""Drop-in `MapAnything` for the feed-forward inference path of etola/map-anything, running on the sm_100a kernels.

Boundary mirrored (reference mapanything/models/mapanything/model.py):
  class MapAnything(nn.Module, PyTorchModelHubMixin)  :87     same constructor kwargs (:90-104), the ctor mutates the
                                                              passed config dicts the same way (:153-193, :260-265, :338-366)
  forward(views, memory_efficient_inference=False)    :1477   same inputs / per-view output dicts (:1727-1741, :1874-1907)
  infer(views, ...)                                   :1964   same kwargs, validation errors, in-place device move of the
                                                              caller's view dicts, temporary geometric_input_config mutation
  device / dtype properties                           :216-222
  state_dict key prefixes                             :157-202, :299, :374-388 (dense_head.{0,1} aliases included)
Only the released configuration is implemented (alternating attention + intermediate features, "dpt+pose" heads,
"raydirs+depth+pose+confidence+mask" adaptor); anything else raises ValueError at construction like the reference does
for unknown types.
"""
from __future__ import annotations

from functools import partial
from typing import Any, Callable, Dict, List, Type, Union

import torch
import torch.nn as nn

from . import ops
from . import params as P
from .engine import DPT_CHUNK, Engine
from .inference import (
    postprocess_model_outputs_for_inference,
    validate_input_views_for_inference,
)

try:  # the reference mixes in huggingface_hub's PyTorchModelHubMixin (from_pretrained / config.json + model.safetensors)
    from huggingface_hub import PyTorchModelHubMixin
except Exception:  # pragma: no cover

    class PyTorchModelHubMixin:  # type: ignore
        pass


class MapAnything(nn.Module, PyTorchModelHubMixin):
    "B200-native MapAnything (images + optional geometric inputs -> pointmaps, poses, masks, confidence, metric scale)."

    def __init__(
        self,
        name: str,
        encoder_config: Dict,
        info_sharing_config: Dict,
        pred_head_config: Dict,
        geometric_input_config: Dict,
        fusion_norm_layer: Union[Type[nn.Module], Callable[..., nn.Module]] = partial(nn.LayerNorm, eps=1e-6),
        pretrained_checkpoint_path: str = None,
        load_specific_pretrained_submodules: bool = False,
        specific_pretrained_submodules: list = None,
        torch_hub_force_reload: bool = False,
    ):
        super().__init__()
        self.name = name
        self.encoder_config = encoder_config
        self.info_sharing_config = info_sharing_config
        self.pred_head_config = pred_head_config
        self.geometric_input_config = geometric_input_config
        self.pretrained_checkpoint_path = pretrained_checkpoint_path
        self.load_specific_pretrained_submodules = load_specific_pretrained_submodules
        self.specific_pretrained_submodules = specific_pretrained_submodules
        self.torch_hub_force_reload = torch_hub_force_reload
        self.class_init_args = {
            "name": name, "encoder_config": encoder_config, "info_sharing_config": info_sharing_config,
            "pred_head_config": pred_head_config, "geometric_input_config": geometric_input_config,
            "pretrained_checkpoint_path": pretrained_checkpoint_path,
            "load_specific_pretrained_submodules": load_specific_pretrained_submodules,
            "specific_pretrained_submodules": specific_pretrained_submodules,
            "torch_hub_force_reload": torch_hub_force_reload,
        }
        self.info_sharing_type = info_sharing_config["model_type"]
        self.info_sharing_return_type = info_sharing_config["model_return_type"]
        self.pred_head_type = pred_head_config["type"]

        if self.encoder_config.get("uses_torch_hub", False):
            self.encoder_config["torch_hub_force_reload"] = torch_hub_force_reload
        enc_cfg = self.encoder_config.copy()
        enc_cfg.pop("uses_torch_hub", None)
        self.encoder = P.encoder_factory(**enc_cfg)
        c = self.encoder.enc_embed_dim

        g = self.geometric_input_config
        for key in ("ray_dirs_encoder_config", "depth_encoder_config"):
            g[key]["enc_embed_dim"] = c
            g[key]["patch_size"] = self.encoder.patch_size
        for key in ("scale_encoder_config", "cam_rot_encoder_config", "cam_trans_encoder_config"):
            g[key]["enc_embed_dim"] = c
        self.ray_dirs_encoder = P.encoder_factory(**g["ray_dirs_encoder_config"])
        self.depth_encoder = P.encoder_factory(**g["depth_encoder_config"])
        self.depth_scale_encoder = P.encoder_factory(**g["scale_encoder_config"])
        self.cam_rot_encoder = P.encoder_factory(**g["cam_rot_encoder_config"])
        self.cam_trans_encoder = P.encoder_factory(**g["cam_trans_encoder_config"])
        self.cam_trans_scale_encoder = P.encoder_factory(**g["scale_encoder_config"])
        self.fusion_norm_layer = fusion_norm_layer(c)
        self.scale_token = nn.Parameter(torch.zeros(c))
        torch.nn.init.trunc_normal_(self.scale_token, std=0.02)

        self._initialize_info_sharing(info_sharing_config)
        self._initialize_prediction_heads(pred_head_config)
        self._initialize_adaptors(pred_head_config)
        self._load_pretrained_weights()
        self._engine = None
        self._shard_comm = None
        self._shard_counts = None
        self._graphs = None   # enable_cuda_graphs(): {(views, batch, H, W): captured forward}

    # ------------------------------------------------------------------------------------------ construction
    def _initialize_info_sharing(self, cfg):
        if cfg["custom_positional_encoding"] is not None:
            raise ValueError(
                f"Invalid custom_positional_encoding: {cfg['custom_positional_encoding']}. None implemented."
            )
        self.custom_positional_encoding = None
        cfg["module_args"]["input_embed_dim"] = self.encoder.enc_embed_dim
        cfg["module_args"]["custom_positional_encoding"] = None
        if self.info_sharing_type == "cross_attention":
            raise ValueError(
                "info_sharing model_type 'cross_attention' (the two-view CroCo / DUSt3R decoder) is not implemented: the only "
                "reference YAML that selects it (configs/model/info_sharing/cat_ifr_dust3r.yaml) sets a string "
                "custom_positional_encoding, which the reference's MapAnything class rejects as well (model.py:244-250)")
        if self.info_sharing_type not in ("alternating_attention", "global_attention"):
            raise ValueError(
                f"Invalid info_sharing_type: {self.info_sharing_type}. Valid options: ['cross_attention', 'global_attention', 'alternating_attention']"
            )
        if self.info_sharing_return_type not in ("no_intermediate_features", "intermediate_features"):
            raise ValueError(
                f"Invalid info_sharing_return_type: {self.info_sharing_return_type}. Valid options: ['no_intermediate_features', 'intermediate_features']"
            )
        if self.info_sharing_type == "global_attention":   # reference model.py:271-284, gat_ifr_24_layers.yaml
            cfg["module_args"].setdefault("attention_pattern", "global")
        if self.info_sharing_return_type == "no_intermediate_features":
            # reference model.py:266-285: only the normalised last-layer features come back, which only the linear head can
            # consume (the DPT branches of forward read intermediate features the module does not return)
            if self.pred_head_type != "linear":
                raise ValueError("model_return_type 'no_intermediate_features' feeds pred_head_type 'linear' only "
                                 "(the DPT heads need the intermediate features)")
            cfg["module_args"].pop("indices", None)
            self.info_sharing = P.AlternatingAttentionIFR(indices=(), **cfg["module_args"])
            return
        self.info_sharing = P.AlternatingAttentionIFR(**cfg["module_args"])
        # reference model.py:304-313: 2 taps -> the DPT also takes the (fused) encoder features; 3 taps -> it does not
        if len(self.info_sharing.indices) == 2:
            self.use_encoder_features_for_dpt = True
        elif len(self.info_sharing.indices) == 3:
            self.use_encoder_features_for_dpt = False
        else:
            raise ValueError(
                "Invalid number of indices provided for info sharing feature returner. Please provide 2 or 3 indices."
            )

    def _initialize_prediction_heads(self, cfg):
        """reference model.py:320-388: "linear" (one 1x1 conv + pixel shuffle on the final features), "dpt" (DPT + regressor),
        "dpt+pose" (+ pose head); the scale head always."""
        cfg["feature_head"]["patch_size"] = self.encoder.patch_size
        if self.pred_head_type == "linear":
            cfg["feature_head"]["input_feature_dim"] = self.info_sharing.dim
        elif "dpt" in self.pred_head_type:
            if self.use_encoder_features_for_dpt:
                cfg["feature_head"]["input_feature_dims"] = [self.encoder.enc_embed_dim] + [self.info_sharing.dim] * 3
            else:
                cfg["feature_head"]["input_feature_dims"] = [self.info_sharing.dim] * 4
            cfg["regressor_head"]["input_feature_dim"] = cfg["feature_head"]["feature_dim"]
            if "pose" in self.pred_head_type:
                cfg["pose_head"]["patch_size"] = self.encoder.patch_size
                cfg["pose_head"]["input_feature_dim"] = self.info_sharing.dim
        else:
            raise ValueError(
                f"Invalid pred_head_type: {self.pred_head_type}. Valid options: ['linear', 'dpt', 'dpt+pose']"
            )
        cfg["scale_head"]["input_feature_dim"] = self.info_sharing.dim
        if self.pred_head_type == "linear":
            self.dense_head = P.LinearFeature(**cfg["feature_head"])
        else:
            self.dpt_feature_head = P.DPTFeature(**cfg["feature_head"])
            self.dpt_regressor_head = P.DPTRegressionProcessor(**cfg["regressor_head"])
            self.dense_head = nn.Sequential(self.dpt_feature_head, self.dpt_regressor_head)
            if "pose" in self.pred_head_type:
                self.pose_head = P.PoseHead(**cfg["pose_head"])
        self.scale_head = P.MLPHead(**cfg["scale_head"])

    # scene representation -> channels of the dense head it consumes (before the optional confidence / mask channels)
    _SCENE_REP_CHANNELS = {"pointmap": 3, "raymap+depth": 7, "raydirs+depth+pose": 4, "campointmap+pose": 3,
                           "pointmap+raydirs+depth+pose": 7}

    def _initialize_adaptors(self, cfg):
        """reference model.py:390-588: the 20 adaptor types = 5 scene representations x {-, confidence} x {-, mask}.  The
        adaptors are parameter-free; here they are the selectors of the fused decode kernels (ma_decode_dense for the
        released representation, ma_decode_scene for the others), which implement the parameter values of the reference's
        adaptor YAMLs (configs/model/pred_head/adaptor_config/*.yaml) -- anything else raises instead of decoding differently."""
        adaptor_type = cfg["adaptor_type"]
        parts = adaptor_type.split("+")
        has_mask = parts[-1] == "mask"
        parts = parts[:-1] if has_mask else parts
        has_conf = parts[-1] == "confidence"
        parts = parts[:-1] if has_conf else parts
        rep = "+".join(parts)
        if rep not in self._SCENE_REP_CHANNELS:
            raise ValueError(
                f"Invalid adaptor_type: {adaptor_type}. Valid options: ['pointmap', 'raymap+depth', 'raydirs+depth+pose', "
                f"'campointmap+pose', 'pointmap+raydirs+depth+pose'], each optionally followed by '+confidence', '+mask' or "
                f"'+confidence+mask'")
        posed = "pose" in rep
        if posed:
            assert self.pred_head_type == "dpt+pose", (
                f"{rep} can only be used as scene representation with dpt + pose head."
            )
        inf = float("inf")
        a = cfg.get("dpt_adaptor" if posed else "adaptor", {})

        def unbounded(prefix):
            return a.get(f"{prefix}_vmin", -inf) == -inf and a.get(f"{prefix}_vmax", inf) == inf

        ok = True
        self._point_mode = "exp"
        if rep in ("pointmap", "campointmap+pose", "pointmap+raydirs+depth+pose"):
            self._point_mode = a.get("pointmap_mode", "exp")
            ok = ok and self._point_mode in ("linear", "exp", "z_exp") and unbounded("pointmap")
        if rep != "pointmap" and rep != "campointmap+pose":
            ok = (ok and a.get("ray_directions_mode", "linear") == "linear"
                  and a.get("ray_directions_normalize_to_unit_sphere", True)
                  and not a.get("ray_directions_normalize_to_unit_image_plane", False)
                  and not a.get("ray_directions_clamp_min_of_z_dir", False) and unbounded("ray_directions")
                  and a.get("depth_mode", "exp") == "exp" and float(a.get("depth_vmin", 0)) == 0.0
                  and a.get("depth_vmax", inf) == inf)
            if rep == "raymap+depth":
                ok = ok and a.get("ray_origins_mode", "linear") == "linear" and unbounded("ray_origins")
        if has_conf:
            ok = ok and a.get("confidence_type", "exp") == "exp" and a.get("confidence_vmax", inf) == inf
        if not ok:
            raise ValueError("the fused decode kernels implement the dense adaptor parameters of the reference's adaptor YAMLs "
                             "only (linear unit-sphere rays, exp depth, exp confidence, linear / exp / z_exp points, no clamping)")
        self._conf_vmin = float(a.get("confidence_vmin", 1))
        if posed:
            # the kernels hard-code the pose adaptor (linear translation, linear + normalised quaternion)
            pa = cfg.get("pose_adaptor", {})
            ok = (pa.get("cam_trans_mode", "linear") == "linear" and pa.get("quaternions_mode", "linear") == "linear"
                  and pa.get("quaternions_normalize", True) and pa.get("cam_trans_vmin", -inf) == -inf
                  and pa.get("cam_trans_vmax", inf) == inf and pa.get("quaternions_vmin", -inf) == -inf
                  and pa.get("quaternions_vmax", inf) == inf)
            if not ok:
                raise ValueError("the fused decode kernel implements the released pose adaptor parameters only "
                                 "(linear translation, linear normalised quaternion, no clamping)")
        sa = cfg.get("scale_adaptor", {})
        ok = (sa.get("mode", "exp") == "exp" and abs(float(sa.get("vmin", 1e-8)) - 1e-8) < 1e-12
              and sa.get("vmax", inf) == inf)
        if not ok:
            raise ValueError("the fused decode kernel implements the released scale adaptor parameters only (exp, vmin 1e-8)")
        head_dim = (cfg["feature_head"] if self.pred_head_type == "linear" else cfg["regressor_head"])["output_dim"]
        need = self._SCENE_REP_CHANNELS[rep] + int(has_conf) + int(has_mask)
        if head_dim != need:
            raise ValueError(f"adaptor_type {adaptor_type!r} consumes {need} channels, the dense head produces {head_dim}")
        self.scene_rep_type = adaptor_type
        self._scene_rep, self._has_conf, self._has_mask = rep, has_conf, has_mask
        self._released_decode = (adaptor_type == "raydirs+depth+pose+confidence+mask" and self._conf_vmin == 1.0)

    def _load_pretrained_weights(self):
        if self.pretrained_checkpoint_path is None:
            return
        ckpt = torch.load(self.pretrained_checkpoint_path, weights_only=False)
        if not self.load_specific_pretrained_submodules:
            print(f"Loading pretrained MapAnything weights from {self.pretrained_checkpoint_path} ...")
            print(self.load_state_dict(ckpt["model"]))
        else:
            print(
                f"Loading pretrained MapAnything weights from {self.pretrained_checkpoint_path} for specific submodules: "
                f"{self.specific_pretrained_submodules} ..."
            )
            filtered = {k: v for k, v in ckpt["model"].items()
                        if any(k.startswith(s) for s in self.specific_pretrained_submodules)}
            print(self.load_state_dict(filtered, strict=False))

    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    @property
    def dtype(self) -> torch.dtype:
        return next(self.parameters()).dtype

    # ------------------------------------------------------------------------------------------ engine plumbing
    def load_state_dict(self, *a, **k):
        self._engine = None
        self._drop_graphs()
        return super().load_state_dict(*a, **k)

    def _apply(self, fn, *a, **k):
        self._engine = None
        self._drop_graphs()
        return super()._apply(fn, *a, **k)

    def _drop_graphs(self):
        if getattr(self, "_graphs", None):   # captured graphs hold pointers to the packed weights of the old engine
            self._graphs = {}

    def enable_cuda_graphs(self, enabled: bool = True) -> None:
        """Replay forward() / infer() as ONE captured CUDA graph per input signature (number of views, per-view batch, image
        size) instead of ~400 kernel launches from Python.  The step of a small scene is partly launch-bound (2 views: 7.85 ms
        kernel by kernel, 7.43 ms replayed); a graph removes the host from it.  Applies to image-only scenes on one GPU without
        memory_efficient_inference; every other call runs the normal path.  The first call of a signature runs the step
        eagerly once (lazy initialisation), captures it and keeps the captured activations alive (one private memory pool
        per signature); inputs are copied into the graph's static image buffers, outputs are copied out, so the returned
        tensors are the caller's.  The kernels, their order and therefore the results are those of the normal path.  No
        reference counterpart (its model.py:1477-1909 launches through the PyTorch dispatcher)."""
        self._graphs = {} if enabled else None

    def engine(self) -> Engine:
        """Packs the parameters for the kernels (once per weight/device change)."""
        if self._engine is None or self._engine.device != self.device:
            with torch.cuda.device(self.device):  # weight packing launches kernels: on the module's device, not the current one
                self._engine = Engine(self)
        return self._engine

    # ------------------------------------------------------------------------------------------ multi-GPU
    def enable_view_sharding(self, group=None, views_per_rank=None):
        """Shard ONE scene by view over the ranks of `group` (default: the world group), one process per GPU
        (SURVEY.md 8e).  Afterwards every rank calls forward()/infer() with ITS OWN contiguous range of the scene's
        views, in rank order (rank 0 holds view 0, the reference view), and gets the predictions of those views back;
        all ranks must call together.  `views_per_rank` (list of ints) skips the per-call exchange of view counts."""
        from .sharding import ViewShardComm

        self._shard_comm = ViewShardComm(group)
        self._shard_counts = list(views_per_rank) if views_per_rank is not None else None
        return self

    def disable_view_sharding(self):
        self._shard_comm = None
        self._shard_counts = None
        return self

    def _sample_geometric_gates(self, views, comm=None) -> Dict[str, Any]:
        """The random input masks of reference model.py:1155-1201 for one batch item, drawn on the host:
          overall_prob (per batch item), 1 - dropout_prob (per view), ray_dirs_prob / depth_prob / cam_prob (per batch item),
          sparse_depth_prob (one coin), depth_scale_norm_all_prob / pose_scale_norm_all_prob (per view).
        With probabilities in {0, 1} -- always the case inside infer() -- nothing is random and a modality is fused iff a
        view provides it.  When nothing is active the reference still runs all five encoders on zeros and multiplies by 0
        (SURVEY F8); the result is exactly LayerNorm(encoder features), which is what this path computes directly.

        View-sharded (comm with world > 1): the per-batch-item coins are drawn on rank 0 and broadcast (one coin per scene,
        as in the reference), and "does ANY view of the scene use the modality" is an all-reduce of three flags -- the
        fusion path contains a collective (the pose all-gather), so every rank must take the same branch even when only
        some shards carry geometric inputs."""
        g = self.geometric_input_config
        V = len(views)
        sharded = comm is not None and comm.world > 1

        def coin(p: float, u: float) -> bool:
            return u < float(p)   # p = 1 -> always, p = 0 -> never (u in [0, 1))

        names = ("overall_prob", "ray_dirs_prob", "depth_prob", "cam_prob", "sparse_depth_prob")
        if all(float(g.get(n, 0.0)) in (0.0, 1.0) for n in names):
            u = [0.0] * len(names)
        else:
            ut = torch.rand(len(names))
            if sharded:
                ut = comm.broadcast(ut.to(self.device), src=0).cpu()
            u = ut.tolist()
        overall, ray_b, depth_b, cam_b, sparse = (coin(g.get(n, 0.0), x) for n, x in zip(names, u))

        def per_view(p: float) -> List[bool]:
            p = float(p)
            if p in (0.0, 1.0):
                return [p == 1.0] * V
            return [bool(x) for x in (torch.rand(V) < p).tolist()]

        keep = [overall and k for k in per_view(1.0 - float(g["dropout_prob"]))]
        gates = {
            "ray": [keep[i] and ray_b and "ray_directions_cam" in v for i, v in enumerate(views)],
            "depth": [keep[i] and depth_b and "depth_along_ray" in v for i, v in enumerate(views)],
            "cam": [keep[i] and cam_b and "camera_pose_quats" in v and "camera_pose_trans" in v for i, v in enumerate(views)],
            "cam_enabled": overall and cam_b,
            "sparse_depth": sparse,
            "depth_norm_all": per_view(g["depth_scale_norm_all_prob"]),
            "pose_norm_all": per_view(g["pose_scale_norm_all_prob"]),
        }
        flags = [any(gates["ray"]), any(gates["depth"]), any(gates["cam"])]
        if sharded:
            flags = comm.any_flags(flags, self.device)
        gates["active"] = any(flags)
        return gates

    def _fuse_geometric_inputs(self, eng, feat, views, b, N, plan, comm, gates=None):
        """Rows a7-a11 of SURVEY 8a for batch item b.  `gates` = _sample_geometric_gates(): which view uses which modality
        (with probabilities in {0,1}: "the view provides it").  Encodes ray directions, depth (+ its metric scale) and the
        camera poses relative to view 0 (+ their metric scale) and adds them to the encoder features in place."""
        g = self.geometric_input_config
        V = len(views)
        dev = self.device
        if gates is None:
            gates = self._sample_geometric_gates(views, comm)

        def metric_flag(view):
            return bool(view["is_metric_scale"][b]) if "is_metric_scale" in view else False

        ray = depth = pose = None
        ids = [i for i in range(V) if gates["ray"][i]]
        if ids:
            ray = (ids, torch.cat([views[i]["ray_directions_cam"][b:b + 1] for i in ids], 0).to(dev, torch.float32))
        ids = [i for i in range(V) if gates["depth"][i]]
        if ids:
            d = torch.cat([views[i]["depth_along_ray"][b:b + 1] for i in ids], 0).to(dev, torch.float32)
            if gates["sparse_depth"]:
                d = self._sparsify_depth(d, float(g.get("sparsification_removal_percent", 0.0)))
            depth = (ids, d, [0.0 if gates["depth_norm_all"][i] else float(metric_flag(views[i])) for i in ids])
        sharded = plan is not None and plan.world > 1
        if any(gates["cam"]) or (sharded and gates["cam_enabled"]):
            # view 0's pose is the reference frame whenever it is PROVIDED, even if view 0's own pose features are dropped
            # (reference model.py:689-703 reads views[0]["camera_pose_*"] under the other view's mask)
            has_data = [("camera_pose_quats" in v and "camera_pose_trans" in v) for v in views]
            q = torch.zeros(V, 4, device=dev)
            t = torch.zeros(V, 3, device=dev)
            for i, v in enumerate(views):
                if has_data[i]:
                    q[i] = v["camera_pose_quats"][b].to(dev, torch.float32)
                    t[i] = v["camera_pose_trans"][b].to(dev, torch.float32)
            use = list(gates["cam"])
            first_is_ref = (not sharded) or plan.rank == 0
            if first_is_ref and has_data[0]:
                use[0] = True     # relative pose of view 0 to itself = identity, zero translation: inert in the normaliser
            hp_ = torch.tensor(use, dtype=torch.uint8, device=dev)
            lo, n_loc = 0, V
            if sharded:  # the pose of view 0 and the translation norms of all views are needed on every rank
                packed = torch.cat([q, t, hp_.float().unsqueeze(1)], dim=1)           # [V_local, 8]
                allp = comm.all_gather_rows(packed, plan.counts)                      # [V_total, 8]
                q, t, hp_ = allp[:, :4].contiguous(), allp[:, 4:7].contiguous(), allp[:, 7].to(torch.uint8).contiguous()
                lo = plan.view_offset
                has_any = bool(hp_.any())  # one host sync; only with pose inputs in sharded mode
            else:
                has_any = True
            if has_any:
                if not bool(hp_[0]):
                    raise ValueError("camera pose inputs need the pose of view 0 (the reference view)")
                q8, t8, s8 = ops.pose_inputs(q, t, hp_)
                pose = (q8[lo:lo + n_loc].contiguous(), t8[lo:lo + n_loc].contiguous(), s8[lo:lo + n_loc].contiguous(),
                        [float(x) for x in gates["cam"]],
                        [0.0 if gates["pose_norm_all"][i] else float(metric_flag(v)) for i, v in enumerate(views)])
        eng.fuse_geometric(feat, V, N, ray=ray, depth=depth, pose=pose)

    @staticmethod
    def _sparsify_depth(d: torch.Tensor, removal: float) -> torch.Tensor:
        """Training-time augmentation of reference model.py:902-933: zero a random `removal` share of the valid (> 0)
        pixels of every depth map.  Host-orchestrated torch indexing: not part of the inference hot path (infer() sets
        sparse_depth_prob = 0)."""
        d = d.clone()
        for i in range(d.shape[0]):
            valid = (d[i] > 0).nonzero(as_tuple=True)
            n = valid[0].numel()
            k = int(n * removal)
            if k > 0:
                sel = torch.randperm(n, device=d.device)[:k]
                d[i][tuple(ix[sel] for ix in valid)] = 0
        return d

    # ------------------------------------------------------------------------------------------ forward
    def forward(self, views: List[Dict[str, Any]], memory_efficient_inference: bool = False) -> List[Dict[str, torch.Tensor]]:
        """Same contract as the reference forward (model.py:1477-1909). Runs under no_grad: this is an inference engine.
        Kernels, side streams and scratch allocations follow the MODULE's device (model.to("cuda:1") works whatever the
        caller's current device is)."""
        if self.device.type != "cuda":
            raise RuntimeError("mapanything_b200 has no CPU path: move the module to a CUDA (sm_100a) device first")
        with torch.cuda.device(self.device):
            return self._forward(views, memory_efficient_inference)

    def _forward(self, views: List[Dict[str, Any]], memory_efficient_inference: bool = False) -> List[Dict[str, torch.Tensor]]:
        per_scene, _ = self._forward_scenes(views, memory_efficient_inference)
        num_views = len(views)
        res = []
        for i in range(num_views):
            d = {}
            for key in ("pts3d", "pts3d_cam", "ray_origins", "ray_directions", "depth_along_ray", "cam_trans", "cam_quats",
                        "conf", "non_ambiguous_mask", "non_ambiguous_mask_logits"):
                if key not in per_scene[0]:   # keys follow the scene representation (reference model.py:1618-1907)
                    continue
                parts = [s[key][i:i + 1] for s in per_scene]
                d[key] = parts[0] if len(parts) == 1 else torch.cat(parts, dim=0)
            scales = [s["metric_scaling_factor"] for s in per_scene]
            d["metric_scaling_factor"] = scales[0] if len(scales) == 1 else torch.cat(scales, dim=0)
            res.append(d)
        return res

    def _compute_adaptive_minibatch_size(self, memory_safety_factor: float = 0.95) -> int:
        """Views per dense-head pass under memory_efficient_inference, by the reference's rule (model.py:1263-1300): free
        device memory x safety factor / 680 MB per 518 x 518 sample, at least 1.  Memory torch's caching allocator holds
        but does not use counts as free (the reference empties the cache first; this avoids the synchronising call).  The
        result is further capped by the engine's normal chunk (8 views), which is what runs when memory is plentiful."""
        free, _ = torch.cuda.mem_get_info(self.device)
        free += torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        return max(1, int(free * memory_safety_factor / (680 * 1024 * 1024)))

    def _forward_scenes(self, views: List[Dict[str, Any]], memory_efficient_inference: bool = False):
        """-> (one dict of [V, ...] output tensors per batch item, the (V,3,H,W) image tensor of each batch item)."""
        if self._graphs is not None and self._graph_eligible(views, memory_efficient_inference):
            return self._forward_scenes_graphed(views)
        return self._forward_scenes_eager(views, memory_efficient_inference)

    _GEOMETRIC_KEYS = ("ray_directions_cam", "depth_along_ray", "camera_pose_quats", "camera_pose_trans")

    def _graph_eligible(self, views, memory_efficient_inference: bool) -> bool:
        """Static launch sequence: image-only views (a modality is fused only when a view provides it), one GPU, the normal
        dense-head chunking."""
        if memory_efficient_inference or (self._shard_comm is not None and self._shard_comm.world > 1):
            return False
        if any(k in v for v in views for k in self._GEOMETRIC_KEYS):
            return False
        shape = views[0]["img"].shape
        return all(torch.is_tensor(v["img"]) and v["img"].shape == shape for v in views)

    def _forward_scenes_graphed(self, views):
        batch, _, height, width = views[0]["img"].shape
        key = (len(views), int(batch), int(height), int(width), views[0]["data_norm_type"][0])
        entry = self._graphs.get(key)
        copy_in = None
        if entry is None:
            static = [torch.empty(batch, 3, height, width, device=self.device, dtype=torch.float32) for _ in views]
            sviews = [{"img": s, "data_norm_type": list(v["data_norm_type"])} for s, v in zip(static, views)]

            def copy_in(vs):
                for s, v in zip(static, vs):
                    s.copy_(v["img"], non_blocking=True)

            copy_in(views)
            # one eager step on a side stream first: engine packing, kernel attribute configuration, positional-embedding
            # cache, allocator warm-up -- nothing of that may happen inside the capture
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._forward_scenes_eager(sviews, False)
            torch.cuda.current_stream().wait_stream(side)
            before = ops.LAUNCHES
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = self._forward_scenes_eager(sviews, False)
            entry = (graph, copy_in, out, ops.LAUNCHES - before)
            self._graphs[key] = entry
        graph, copy_in, (per_scene, scene_imgs), launches = entry
        copy_in(views)
        graph.replay()
        ops._count(launches)   # the captured kernels do run: keep the launch count honest
        # the captured outputs are overwritten by the next replay: hand out copies (13 MB per view)
        return [{k: t.clone() for k, t in s.items()} for s in per_scene], scene_imgs

    def _forward_scenes_eager(self, views: List[Dict[str, Any]], memory_efficient_inference: bool = False):
        batch_size_per_view, _, height, width = views[0]["img"].shape
        num_views = len(views)
        data_norm_type = views[0]["data_norm_type"][0]
        if data_norm_type != self.encoder.data_norm_type:
            raise AssertionError(
                f"Input data_norm_type {data_norm_type} does not match the encoder's {self.encoder.data_norm_type}"
            )
        p = self.encoder.patch_size
        if height % p or width % p:
            raise AssertionError(f"Input image size ({height}, {width}) must be a multiple of the patch size {p}")
        eng = self.engine()
        eng.dpt_chunk = min(self._compute_adaptive_minibatch_size(), DPT_CHUNK) if memory_efficient_inference else DPT_CHUNK
        hp, wp = height // p, width // p
        N = hp * wp
        plan, comm = None, self._shard_comm
        if comm is not None and comm.world > 1:
            from .sharding import ViewShardPlan

            counts = self._shard_counts or comm.exchange_counts(num_views, self.device)
            if counts[comm.rank] != num_views:
                raise ValueError(f"rank {comm.rank} was given {num_views} views, views_per_rank says {counts[comm.rank]}")
            plan = ViewShardPlan(counts, comm.rank, N)
        per_scene, scene_imgs = [], []
        with torch.no_grad():
            for b in range(batch_size_per_view):
                imgs = torch.cat([v["img"][b:b + 1] for v in views], dim=0).to(self.device, torch.float32)
                scene_imgs.append(imgs)
                feat = eng.encode(imgs)                       # fp32 [V*N][C]   DINOv2 x_norm_patchtokens
                gates = self._sample_geometric_gates(views, comm)
                if gates["active"]:
                    self._fuse_geometric_inputs(eng, feat, views, b, N, plan, comm, gates)
                fused = eng.fuse_norm(feat)                   # bf16 [V*N][C]   fusion LayerNorm (DPT tap 0)
                taps, final, final32 = eng.info_sharing(fused, num_views, N, plan=plan, comm=comm)
                if self.pred_head_type == "linear":   # reference model.py:1541-1545: the final features only
                    dpt_in = [final]
                else:
                    dpt_in = [fused, taps[0], taps[1], final] if self.use_encoder_features_for_dpt else [*taps, final]
                raw, pose_raw = eng.dpt_and_pose(dpt_in, num_views, hp, wp, height, width, final32=final32[:num_views * N])
                if plan is None:
                    scale_raw = eng.scale_head(final32[num_views * N:])
                else:  # the scale token lives on rank 0: one float travels to the other ranks
                    scale_raw = eng.scale_head(final32[num_views * N:]) if plan.rank == 0 else \
                        torch.empty(1, device=self.device, dtype=torch.float32)
                    comm.broadcast(scale_raw, src=0)
                per_scene.append(self._decode(raw, pose_raw, scale_raw, num_views, height, width))
        return per_scene, scene_imgs

    def _decode(self, raw, pose_raw, scale_raw, num_views, height, width):
        """dense / pose / scale adaptors + the scene-representation branch of reference model.py:1618-1907, one launch."""
        if self._released_decode:
            return ops.decode_dense(raw, pose_raw, scale_raw, num_views, height, width)
        use_factored = False
        if self._scene_rep == "pointmap+raydirs+depth+pose":   # reference model.py:1822-1833
            use_factored = bool(self.pred_head_config["adaptor_config"]["use_factored_predictions_for_global_pointmaps"])
        return ops.decode_scene(raw, pose_raw, scale_raw, num_views, height, width, rep=self._scene_rep,
                                has_conf=self._has_conf, has_mask=self._has_mask, point_mode=self._point_mode,
                                use_factored=use_factored, conf_vmin=self._conf_vmin)

    # ------------------------------------------------------------------------------------------ infer
    def _configure_geometric_input_config(self, use_calibration: bool, use_depth: bool, use_pose: bool,
                                          use_depth_scale: bool, use_pose_scale: bool):
        if not hasattr(self, "_original_geometric_config"):
            self._original_geometric_config = dict(self.geometric_input_config)
        if not (use_calibration or use_depth or use_pose):
            self.geometric_input_config.update({
                "overall_prob": 0.0, "dropout_prob": 1.0, "ray_dirs_prob": 0.0, "depth_prob": 0.0, "cam_prob": 0.0,
                "sparse_depth_prob": 0.0, "depth_scale_norm_all_prob": 0.0, "pose_scale_norm_all_prob": 0.0,
            })
        else:
            self.geometric_input_config.update({
                "overall_prob": 1.0, "dropout_prob": 0.0, "ray_dirs_prob": 1.0 if use_calibration else 0.0,
                "depth_prob": 1.0 if use_depth else 0.0, "cam_prob": 1.0 if use_pose else 0.0, "sparse_depth_prob": 0.0,
                "depth_scale_norm_all_prob": 0.0 if use_depth_scale else 1.0,
                "pose_scale_norm_all_prob": 0.0 if use_pose_scale else 1.0,
            })

    def _restore_original_geometric_input_config(self):
        if hasattr(self, "_original_geometric_config"):
            self.geometric_input_config.update(self._original_geometric_config)

    @torch.inference_mode()
    def infer(
        self,
        views: List[Dict[str, Any]],
        memory_efficient_inference: bool = False,
        use_amp: bool = True,
        amp_dtype: str = "bf16",
        apply_mask: bool = True,
        mask_edges: bool = True,
        edge_normal_threshold: float = 5.0,
        edge_depth_threshold: float = 0.03,
        apply_confidence_mask: bool = False,
        confidence_percentile: float = 10,
        ignore_calibration_inputs: bool = False,
        ignore_depth_inputs: bool = False,
        ignore_pose_inputs: bool = False,
        ignore_depth_scale_inputs: bool = False,
        ignore_pose_scale_inputs: bool = False,
    ) -> List[Dict[str, torch.Tensor]]:
        """Same surface as the reference infer (model.py:1964-2112).  The kernels always compute with bf16 tensor-core
        operands, fp32 accumulation and fp32 residual streams -- the reference's `use_amp=True, amp_dtype="bf16"` mode;
        `use_amp=False` / other amp_dtype values raise (there is no fp32 / fp16 path to fall back to)."""
        if self.device.type != "cuda":
            raise RuntimeError("mapanything_b200 has no CPU path: move the module to a CUDA (sm_100a) device first")
        with torch.cuda.device(self.device):
            return self._infer(views, memory_efficient_inference, use_amp, amp_dtype, apply_mask, mask_edges,
                               edge_normal_threshold, edge_depth_threshold, apply_confidence_mask, confidence_percentile,
                               ignore_calibration_inputs, ignore_depth_inputs, ignore_pose_inputs, ignore_depth_scale_inputs,
                               ignore_pose_scale_inputs)

    def _infer(self, views, memory_efficient_inference, use_amp, amp_dtype, apply_mask, mask_edges, edge_normal_threshold,
               edge_depth_threshold, apply_confidence_mask, confidence_percentile, ignore_calibration_inputs,
               ignore_depth_inputs, ignore_pose_inputs, ignore_depth_scale_inputs, ignore_pose_scale_inputs):
        if not use_amp or amp_dtype != "bf16":
            raise ValueError(
                f"mapanything_b200 computes with bf16 tensor-core operands (fp32 accumulate / residual streams) only: "
                f"use_amp={use_amp!r}, amp_dtype={amp_dtype!r} is not available (reference model.py:2044-2059 would run "
                f"fp32 / fp16 autocast)")
        # view-sharded: only rank 0's first view is the scene's reference view; the scene-wide "view 0 has a pose" rule is
        # enforced on the gathered flags in _fuse_geometric_inputs (identically on every rank)
        sharded = self._shard_comm is not None and self._shard_comm.world > 1
        validated = validate_input_views_for_inference(
            views, first_view_is_reference=(not sharded) or self._shard_comm.rank == 0)
        ignore_keys = {"instance", "idx", "true_shape", "data_norm_type"}
        for view in validated:
            for key in view.keys():
                if key in ignore_keys:
                    continue
                view[key] = view[key].to(self.device, non_blocking=True)
        from .preprocess import preprocess_input_views_for_inference

        processed = preprocess_input_views_for_inference(validated)
        self._configure_geometric_input_config(
            use_calibration=not ignore_calibration_inputs, use_depth=not ignore_depth_inputs,
            use_pose=not ignore_pose_inputs, use_depth_scale=not ignore_depth_scale_inputs,
            use_pose_scale=not ignore_pose_scale_inputs,
        )
        scene = None
        try:
            one_norm = all(v["data_norm_type"][0] == processed[0]["data_norm_type"][0] for v in processed)
            if processed[0]["img"].shape[0] == 1 and one_norm:   # one scene: post-process all views with one launch set
                scene = self._forward_scenes(processed, memory_efficient_inference)
            else:
                preds = self.forward(processed, memory_efficient_inference=memory_efficient_inference)
        finally:
            self._restore_original_geometric_input_config()
        if scene is not None:
            from .inference import postprocess_scene

            return postprocess_scene(
                scene[0][0], scene[1][0], processed[0]["data_norm_type"][0], apply_mask=apply_mask, mask_edges=mask_edges,
                edge_normal_threshold=edge_normal_threshold, edge_depth_threshold=edge_depth_threshold,
                apply_confidence_mask=apply_confidence_mask, confidence_percentile=confidence_percentile)
        return postprocess_model_outputs_for_inference(
            raw_outputs=preds, input_views=processed, apply_mask=apply_mask, mask_edges=mask_edges,
            edge_normal_threshold=edge_normal_threshold, edge_depth_threshold=edge_depth_threshold,
            apply_confidence_mask=apply_confidence_mask, confidence_percentile=confidence_percentile,
        )
