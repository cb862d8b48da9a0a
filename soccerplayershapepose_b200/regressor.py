"""Regressor head + multi-task loss around the SMPL layer (SURVEY.md section 8f.2; BASELINE.json configs[4]).

Mirrors the reference's training step (PlayerReconstruction/PyTorch3DTest.py:1046-1106):

    features -> IEFModule (models/ief_module.py:8-64) -> (cam, pose 6D, shape)
             -> rot6d_to_rotmat (utils/rigid_transform_utils.py:27-41)           [C-ABI kernel]
             -> SMPL(body_pose, global_orient, betas, pose2rot=False)            [C-ABI kernels]
             -> orthographic projection of the joints, COCO map, pixels          [fused C-ABI kernel]
             -> (silhouette term: the predicted bodies' soft silhouettes, PyTorch3DTest.py:1084-1087)
             -> HomoscedasticUncertaintyWeightedMultiTaskLoss (losses/multi_task_loss.py:92-144)
             -> backward -> (data-parallel: NCCL all-reduce of the head's gradients) -> Adam

The CNN encoder in front is the caller's (BASELINE.json: "CNN features -> SMPL head"); the head's three linear
layers are plain library GEMMs (torch.nn.Linear).  The SMPL layer has no parameters, so under
DistributedDataParallel only the head (and the loss's log-variances) are all-reduced: ~1.9 M floats for the
reference sizes (fc 1024/1024, 512 input features, 157 outputs).  The SMPL layer and the fused loss need a CUDA
device; the head and `MultiTaskLoss` themselves are device-agnostic (the CPU tests run them with the oracle).
"""
from __future__ import annotations

from typing import Callable, Dict, NamedTuple, Optional, Sequence, Tuple, Union

import numpy as np
import torch
import torch.nn as nn

from . import config

NUM_OUTPUT_PARAMS = 3 + 24 * 6 + 10


def default_mean_params() -> torch.Tensor:
    """models/ief_module.py:36-48 with the SMPL mean parameters file absent: camera [0.9, 0, 0], identity
    rotations in the 6D representation (columns (1,0,0),(0,1,0) -> x.view(3,2) = [[1,0],[0,1],[0,0]]), zero shape."""
    p = np.zeros(NUM_OUTPUT_PARAMS, np.float32)
    p[0] = 0.9
    p[3:3 + 24 * 6] = np.tile(np.array([1, 0, 0, 1, 0, 0], np.float32), 24)
    return torch.from_numpy(p)


class IEFModule(nn.Module):
    """Iterative error feedback head (models/ief_module.py:8-64): same layers, same zero-bias init, same loop."""

    def __init__(self, fc_layers_neurons: Sequence[int] = (1024, 1024), in_features: int = 512,
                 num_output_params: int = NUM_OUTPUT_PARAMS, iterations: int = 3,
                 mean_params: Optional[torch.Tensor] = None):
        super().__init__()
        self.fc1 = nn.Linear(in_features + num_output_params, fc_layers_neurons[0])
        self.fc2 = nn.Linear(fc_layers_neurons[0], fc_layers_neurons[1])
        self.fc3 = nn.Linear(fc_layers_neurons[1], num_output_params)
        self.relu = nn.ReLU(inplace=True)
        for fc in (self.fc1, self.fc2, self.fc3):
            torch.nn.init.zeros_(fc.bias)
        self.ief_layers = nn.Sequential(self.fc1, self.relu, self.fc2, self.relu, self.fc3)
        self.iterations = iterations
        # a plain (non-persistent) buffer: the reference keeps it as an attribute (models/ief_module.py:30), so its
        # checkpoints carry fc1/fc2/fc3 and ief_layers.* keys only and state_dicts interchange in both directions
        self.register_buffer("initial_params_estimate",
                             default_mean_params() if mean_params is None else mean_params.float().clone(),
                             persistent=False)

    def forward(self, img_features: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        params = self.initial_params_estimate.repeat([img_features.size(0), 1])
        state = torch.cat([img_features, params], dim=1)
        for _ in range(self.iterations):
            params = params + self.ief_layers(state)
            state = torch.cat([img_features, params], dim=1)
        return params[:, :3], params[:, 3:3 + 24 * 6], params[:, 3 + 24 * 6:]


class MultiTaskLoss(nn.Module):
    """HomoscedasticUncertaintyWeightedMultiTaskLoss (losses/multi_task_loss.py:16-152): MSE(mean) per task *
    exp(-log_var) + log_var, log_var0 = -log(w + 1e-6), log-variances trainable.

    "silhouette" (losses/multi_task_loss.py:132-144): L = batch mean of the per-body mean over the S^2 pixels of
    (alpha - target)^2, alpha the soft silhouette of the predicted body and target = labels["silhouette"] (B,S,S)
    (floating point >= 0.5 or non-zero is inside).  The form of the reference's silhouette loss could not be read;
    this squared error is the fitter's stated definition (DESIGN.md section 11).  The camera is
    `SMPL.render_silhouettes`': t = [tx, ty, 2 f / (proj_wh s + 1e-9)] from the head's weak-perspective cam, f =
    config.FOCAL_LENGTH, rendered at S = `silhouette_wh` with focal length f S / proj_wh and blur `silhouette_sigma`.
    `faces` (F,3) are required with the term and kept as a non-persistent buffer (state_dicts gain only
    `silhouette_log_var`)."""

    TASKS = ("verts", "joints2D", "joints3D", "shape_params", "pose_params", "silhouette")

    def __init__(self, losses_on: Sequence[str], init_loss_weights: Optional[Dict[str, float]] = None, eps: float = 1e-6,
                 faces=None, silhouette_sigma: float = 1.0, silhouette_wh: int = config.REGRESSOR_IMG_WH,
                 proj_wh: float = 512.0):
        super().__init__()
        self.losses_on = tuple(losses_on)
        for t in self.losses_on:
            if t not in self.TASKS:
                raise ValueError("unsupported loss term: " + t)
            w = None if init_loss_weights is None else init_loss_weights.get(t)
            lv = 0.0 if w is None else float(-np.log(w + eps))
            setattr(self, t + "_log_var", nn.Parameter(torch.tensor(lv).float()))
        if "silhouette" in self.losses_on:
            if faces is None:
                raise ValueError("the silhouette term needs the mesh faces (faces=...)")
            faces = torch.as_tensor(faces)
            if faces.dim() != 2 or faces.shape[1] != 3 or faces.dtype.is_floating_point:
                raise ValueError("faces must be an integer (F, 3) array")
            self.register_buffer("silhouette_faces", faces.to(torch.int32).contiguous(), persistent=False)
            self.silhouette_sigma = float(silhouette_sigma)
            self.silhouette_wh = int(silhouette_wh)
            self.proj_wh = float(proj_wh)

    def _silhouette_target(self, labels: Dict[str, torch.Tensor], B: int) -> torch.Tensor:
        tgt = labels["silhouette"]
        S = self.silhouette_wh
        if tuple(tgt.shape) != (B, S, S):
            raise ValueError("labels['silhouette'] has shape {}, expected {}".format(tuple(tgt.shape), (B, S, S)))
        return tgt

    def silhouette_camera(self, cam: torch.Tensor) -> Tuple[torch.Tensor, float]:
        """Camera translation (B,3) from the head's weak-perspective cam (differentiable) and the render focal length."""
        from .cam_utils import convert_weak_perspective_to_camera_translation_torch
        t = convert_weak_perspective_to_camera_translation_torch(cam, config.FOCAL_LENGTH, self.proj_wh)
        return t.contiguous(), config.FOCAL_LENGTH * self.silhouette_wh / self.proj_wh

    def forward(self, labels: Dict[str, torch.Tensor], outputs: Dict[str, torch.Tensor]):
        total, parts = 0.0, {}

        def add(name, value):
            nonlocal total
            lv = getattr(self, name + "_log_var")
            total = total + value * torch.exp(-lv) + lv
            parts[name] = value * torch.exp(-lv)

        if "verts" in self.losses_on:
            add("verts", torch.mean((outputs["verts"] - labels["verts"]) ** 2))
        if "joints2D" in self.losses_on:
            lab, pred = labels["joints2D"], outputs["joints2D"]
            if "vis" in labels:
                lab, pred = lab[labels["vis"], :], pred[labels["vis"], :]
            lab = (2.0 * lab) / config.REGRESSOR_IMG_WH - 1.0
            pred = (2.0 * pred) / config.REGRESSOR_IMG_WH - 1.0
            add("joints2D", torch.mean((pred - lab) ** 2))
        if "joints3D" in self.losses_on:
            add("joints3D", torch.mean((outputs["joints3D"] - labels["joints3D"]) ** 2))
        if "shape_params" in self.losses_on:
            add("shape_params", torch.mean((outputs["shape_params"] - labels["shape_params"]) ** 2))
        if "pose_params" in self.losses_on:
            add("pose_params", torch.mean((outputs["pose_params_rot_matrices"] - labels["pose_params_rot_matrices"]) ** 2))
        if "silhouette" in self.losses_on:
            if outputs.get("silhouettes") is None:
                raise ValueError("the silhouette term needs outputs['silhouettes']: pass render_silhouettes to predict")
            alpha = outputs["silhouettes"]
            tgt = self._silhouette_target(labels, alpha.shape[0])
            mask = tgt >= 0.5 if tgt.dtype.is_floating_point else tgt != 0
            add("silhouette", torch.mean((alpha - mask.to(alpha.dtype)) ** 2))
        return total, parts


    def forward_fused(self, labels: Dict[str, torch.Tensor], outputs: Dict[str, torch.Tensor]):
        """The same loss through ONE fused reduction + ONE fused gradient kernel (`ops.multitask_loss`,
        csrc/loss.cu) instead of ~40 eager PyTorch kernels: needs CUDA tensors and the raw `joints` (B,90,3) / `cam`
        of `predict` (the projection, both joint gathers and the pixel normalisation happen inside the kernel)."""
        from . import ops
        on = self.losses_on
        dev = outputs["joints"].device
        zero = torch.zeros((), dtype=torch.float32, device=dev)
        lv = torch.stack([getattr(self, t + "_log_var") if t in on else zero
                          for t in ("verts", "joints2D", "joints3D", "shape_params", "pose_params")])
        kw = {}
        if "verts" in on:
            kw.update(verts=outputs["verts"], verts_label=labels["verts"])
        if "joints2D" in on:
            kw.update(map2d=_index32("SMPL_TO_KPRCNN_MAP", dev), label2d=labels["joints2D"], vis=labels.get("vis"))
        if "joints3D" in on:
            kw.update(map3d=_index32("ALL_JOINTS_TO_COCO_MAP", dev), label3d=labels["joints3D"])
        if "shape_params" in on:
            kw.update(shape=outputs["shape_params"], shape_label=labels["shape_params"])
        if "pose_params" in on:
            kw.update(pose=outputs["pose_params_rot_matrices"], pose_label=labels["pose_params_rot_matrices"])
        loss, parts = ops.multitask_loss(lv, joints=outputs["joints"], cam=outputs["cam"], proj_wh=512.0,
                                         norm_wh=float(config.REGRESSOR_IMG_WH), **kw)
        names = ("verts", "joints2D", "joints3D", "shape_params", "pose_params")
        parts = {n: parts[i] for i, n in enumerate(names) if n in on}
        if "silhouette" in on:
            verts = outputs["verts"]
            t, f = self.silhouette_camera(outputs["cam"])
            L = ops.silhouette_term(verts, self.silhouette_faces, t, self._silhouette_target(labels, verts.shape[0]),
                                    self.silhouette_wh, f, self.silhouette_sigma)
            lv = self.silhouette_log_var
            parts["silhouette"] = L * torch.exp(-lv)
            loss = loss + parts["silhouette"] + lv
        return loss, parts


_INDEX_CACHE: Dict[Tuple[str, str], torch.Tensor] = {}


def _index32(name: str, device: torch.device) -> torch.Tensor:
    key = (name + ":i32", str(device))
    if key not in _INDEX_CACHE:
        _INDEX_CACHE[key] = torch.tensor(getattr(config, name), dtype=torch.int32, device=device)
    return _INDEX_CACHE[key]


def _index(name: str, device: torch.device) -> torch.Tensor:
    """config joint maps as device index tensors, built once per device (a Python list index would upload the
    indices on every call, which a CUDA graph capture cannot contain)."""
    key = (name, str(device))
    if key not in _INDEX_CACHE:
        _INDEX_CACHE[key] = torch.tensor(getattr(config, name), dtype=torch.long, device=device)
    return _INDEX_CACHE[key]


def predict(head: nn.Module, smpl: Callable, features: torch.Tensor, rot6d_to_rotmat: Callable,
            project_pixels: Optional[Callable], need_verts: bool = True,
            render_silhouettes: Optional[Callable] = None) -> Dict[str, torch.Tensor]:
    """PyTorch3DTest.py:1046-1071: head -> rotation matrices -> SMPL -> COCO joints in 3D and in pixels.
    `smpl`, `rot6d_to_rotmat` and `project_pixels(joints, cam) -> (B,90,2) pixels` are injected so that the same
    code runs on the C-ABI kernels (GPU) and on the oracle (CPU tests).  `render_silhouettes(verts, cam) -> (B,S,S)`
    soft alpha (PyTorch3DTest.py:1084-1087; `gpu_silhouette_renderer` on the GPU) fills "silhouettes"."""
    cam, pose6d, shape = head(features)
    rotmats = rot6d_to_rotmat(pose6d.contiguous()).view(-1, 24, 3, 3)
    out = smpl(body_pose=rotmats[:, 1:], global_orient=rotmats[:, 0].unsqueeze(1), betas=shape, pose2rot=False,
               return_verts=need_verts)
    dev = out.joints.device
    res = {"verts": out.vertices if need_verts else None, "shape_params": shape, "pose_params_rot_matrices": rotmats,
           "cam": cam, "joints": out.joints}
    if project_pixels is not None:       # None: the fused loss projects / gathers inside its kernel
        res["joints2D"] = project_pixels(out.joints, cam).index_select(1, _index("SMPL_TO_KPRCNN_MAP", dev))
        res["joints3D"] = out.joints.index_select(1, _index("ALL_JOINTS_TO_COCO_MAP", dev))
    if render_silhouettes is not None:
        res["silhouettes"] = render_silhouettes(out.vertices, cam)
    return res


def train_step(head: nn.Module, criterion: MultiTaskLoss, optimiser: torch.optim.Optimizer, smpl: Callable,
               features: torch.Tensor, labels: Dict[str, torch.Tensor], rot6d_to_rotmat: Callable,
               project_pixels: Optional[Callable], fused_loss: bool = False,
               render_silhouettes: Optional[Callable] = None) -> torch.Tensor:
    """One optimisation step (PyTorch3DTest.py:1097-1102).  When `head` / `criterion` are wrapped in
    DistributedDataParallel the backward all-reduces their gradients (NCCL on the GPUs).  `fused_loss`: evaluate
    the loss with the fused kernels (CUDA only).  `render_silhouettes`: see `predict` (the eager silhouette term;
    the fused one renders inside its kernel)."""
    optimiser.zero_grad(set_to_none=True)
    outputs = predict(head, smpl, features, rot6d_to_rotmat, None if fused_loss else project_pixels,
                      need_verts=_needs_verts(criterion), render_silhouettes=_renderer(criterion, fused_loss,
                                                                                       render_silhouettes))
    crit = getattr(criterion, "module", criterion)
    loss, _ = crit.forward_fused(labels, outputs) if fused_loss else criterion(labels, outputs)
    loss.backward()
    optimiser.step()
    return loss.detach()


def validation_step(head: nn.Module, criterion: MultiTaskLoss, smpl: Callable, features: torch.Tensor,
                    labels: Dict[str, torch.Tensor], rot6d_to_rotmat: Callable, project_pixels: Optional[Callable],
                    fused_loss: bool = False,
                    render_silhouettes: Optional[Callable] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """One validation batch (the reference's `is_train = False` pass, PyTorch3DTest.py:947-1118) -> (loss, errors).
    Under torch.no_grad: `predict` (forward-only SMPL calls), the criterion as `train_step` evaluates it (eager or
    `fused_loss`; the fused silhouette term then only evaluates its value), the target bodies from
    labels["pose_params_rot_matrices"] and labels["shape_params"] (PyTorch3DTest.py:1036-1042), and one T-pose forward
    (zero pose, zero translation) of the predicted and target shapes.  errors (B, 7) float32 on the device: pve,
    pve_sc, pve_pa, mpjpe, mpjpe_sc, mpjpe_pa (`ops.reconstruction_errors` on the vertices and the LSP-14 joints,
    config.ALL_JOINTS_TO_J14_MAP) and pve_t_sc (pve_sc of the T-pose meshes), in the SMPL model's units.  It never
    synchronises with the host (after the first call, which checks the joint map once) and touches no gradient or
    optimiser state.  Per-epoch sums stay on the device: `sums += errors.sum(0)`."""
    from . import ops
    with torch.no_grad():
        outputs = predict(head, smpl, features, rot6d_to_rotmat, None if fused_loss else project_pixels,
                          need_verts=True, render_silhouettes=_renderer(criterion, fused_loss, render_silhouettes))
        crit = getattr(criterion, "module", criterion)
        loss, _ = crit.forward_fused(labels, outputs) if fused_loss else criterion(labels, outputs)
        rot, shape = labels["pose_params_rot_matrices"], labels["shape_params"]
        target = smpl(body_pose=rot[:, 1:], global_orient=rot[:, 0].unsqueeze(1), betas=shape, pose2rot=False)
        pred_shape = outputs["shape_params"]
        B, dev = pred_shape.shape[0], pred_shape.device
        eye = torch.eye(3, dtype=torch.float32, device=dev).expand(2 * B, 24, 3, 3)
        tpose = smpl(body_pose=eye[:, 1:], global_orient=eye[:, :1], betas=torch.cat([pred_shape, shape]),
                     transl=torch.zeros((2 * B, 3), dtype=torch.float32, device=dev), pose2rot=False).vertices
        errors = ops.reconstruction_errors(outputs["verts"], target.vertices, outputs["joints"], target.joints,
                                           _index32("ALL_JOINTS_TO_J14_MAP", dev))
        t_sc = ops.reconstruction_errors(tpose[:B], tpose[B:])[:, 1:2]
        return loss.detach(), torch.cat([errors, t_sc], dim=1)


def _tasks(criterion) -> Sequence[str]:
    return getattr(criterion, "module", criterion).losses_on


def _needs_verts(criterion) -> bool:
    tasks = _tasks(criterion)
    return "verts" in tasks or "silhouette" in tasks


def _renderer(criterion, fused_loss: bool, render_silhouettes: Optional[Callable]) -> Optional[Callable]:
    """The renderer `predict` runs: only for the eager loss of a criterion with the silhouette term."""
    return render_silhouettes if ("silhouette" in _tasks(criterion) and not fused_loss) else None


class _BasicBlock(nn.Module):
    """torchvision BasicBlock as restated in models/resnet.py:35-74 (attribute names kept for state_dict parity)."""
    expansion = 1

    def __init__(self, inplanes: int, planes: int, stride: int = 1, downsample: Optional[nn.Module] = None):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = nn.Conv2d(planes, planes, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = downsample

    def forward(self, x):
        out = self.bn2(self.conv2(self.relu(self.bn1(self.conv1(x)))))
        return self.relu(out + (x if self.downsample is None else self.downsample(x)))


class ResNet18Encoder(nn.Module):
    """The reference's image encoder (models/resnet.py:124-217 with BasicBlock [2,2,2,2], no final FC): the CALLER's
    side of BASELINE.json configs[4] ("CNN features -> SMPL head").  Plain library convolutions (cuDNN) -- it is here
    so that the data-parallel step all-reduces the reference's real 11.9 M parameters (47.6 MB), not just the head;
    module / parameter names follow the reference so `image_encoder.*` checkpoints interchange."""

    def __init__(self, in_channels: int = 18):
        super().__init__()
        self.inplanes = 64
        self.conv1 = nn.Conv2d(in_channels, 64, 7, 2, 3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(3, 2, 1)
        self.layer1 = self._make_layer(64, 2, 1)
        self.layer2 = self._make_layer(128, 2, 2)
        self.layer3 = self._make_layer(256, 2, 2)
        self.layer4 = self._make_layer(512, 2, 2)
        self.avgpool = nn.AdaptiveAvgPool2d((1, 1))
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")

    def _make_layer(self, planes: int, blocks: int, stride: int) -> nn.Sequential:
        down = None
        if stride != 1 or self.inplanes != planes:
            down = nn.Sequential(nn.Conv2d(self.inplanes, planes, 1, stride, bias=False), nn.BatchNorm2d(planes))
        layers = [_BasicBlock(self.inplanes, planes, stride, down)]
        self.inplanes = planes
        layers += [_BasicBlock(planes, planes) for _ in range(1, blocks)]
        return nn.Sequential(*layers)

    def forward(self, x):
        x = self.maxpool(self.relu(self.bn1(self.conv1(x))))
        x = self.layer4(self.layer3(self.layer2(self.layer1(x))))
        return torch.flatten(self.avgpool(x), 1)


class SingleInputRegressor(nn.Module):
    """models/regressor.py:7-46 for resnet_layers=18: `image_encoder` (ResNet-18 over the 18-channel 256x256 proxy
    representation, PyTorch3DTest.py:241) + `ief_module` IEFModule([512, 512], 512, 157)."""

    def __init__(self, resnet_in_channels: int = 18, resnet_layers: int = 18, ief_iters: int = 3):
        super().__init__()
        if resnet_layers != 18:
            raise NotImplementedError("only the ResNet-18 configuration the reference trains is provided")
        self.image_encoder = ResNet18Encoder(resnet_in_channels)
        self.ief_module = IEFModule((512, 512), 512, NUM_OUTPUT_PARAMS, iterations=ief_iters)

    def forward(self, input):
        return self.ief_module(self.image_encoder(input))


def gpu_ops():
    """The C-ABI-backed implementations to inject on a CUDA device."""
    from . import ops
    return ops.rot6d_to_rotmat, (lambda joints, cam: ops.orthographic_project(joints, cam, 512.0))


def gpu_silhouette_renderer(faces, img_wh: int = config.REGRESSOR_IMG_WH, sigma: float = 1.0,
                            proj_wh: float = 512.0) -> Callable:
    """`render_silhouettes(verts, cam) -> (B, img_wh, img_wh)` soft alpha for `predict` on a CUDA device
    (ops.render_silhouettes with the camera of `SMPL.render_silhouettes` and of MultiTaskLoss's silhouette term)."""
    from . import ops
    from .cam_utils import convert_weak_perspective_to_camera_translation_torch
    f = config.FOCAL_LENGTH * float(img_wh) / float(proj_wh)

    def render(verts: torch.Tensor, cam: torch.Tensor) -> torch.Tensor:
        t = convert_weak_perspective_to_camera_translation_torch(cam, config.FOCAL_LENGTH, proj_wh)
        return ops.render_silhouettes(verts, faces, t.contiguous(), img_wh, focal_length=f, sigma=sigma)
    return render


class ProxyInputs(NamedTuple):
    """What a detector gives per crop, for `GraphedTrainStep` to build the proxy representation from inside its graph
    (`ops.proxy_representation`): masks (B, in_wh, in_wh) bool / uint8 / float, keypoints (B, K, 2) float32 pixels
    of the in_wh image, vis (B, K) or None; out_wh / std as in the op."""
    masks: torch.Tensor
    keypoints: torch.Tensor
    vis: Optional[torch.Tensor] = None
    out_wh: int = config.REGRESSOR_IMG_WH
    std: float = 4.0


def _channels_last(module: nn.Module) -> bool:
    """True when the module's first 4-D parameter (an encoder's first convolution) is in torch.channels_last."""
    for p in module.parameters():
        if p.dim() == 4:
            return p.is_contiguous(memory_format=torch.channels_last) and not p.is_contiguous()
    return False


class GraphedTrainStep:
    """The training step of `train_step` captured ONCE in a CUDA graph and replayed: (encoder +) head forward, SMPL
    layer, loss, backward, gradient all-reduce (NCCL) and a capturable Adam step.  The eager step is bound by ~100
    small PyTorch launches; a replay is one launch.

    All gradients live in one flat buffer (`p.grad` are views into it), laid out in the order the backward produces
    them (last layer first) and cut into buckets of ~`bucket_mb`: as soon as the backward has written the last
    gradient of a bucket, its all-reduce is issued on a side stream -- inside the captured graph this becomes a fork,
    so the NCCL kernels of the late layers overlap the encoder's backward, as DistributedDataParallel does eagerly.
    The SMPL layer has no parameters: the buckets are the head (+ encoder) and the loss's log-variances.  Inputs are
    copied into static buffers before each replay; `world_size > 1` requires an initialised NCCL process group.
    `features` may be a `ProxyInputs`: the static input buffers are then the masks, keypoints and vis, the captured
    step starts with the proxy kernel writing a static proxy buffer in the encoder's memory format, and a call copies
    only those raw inputs (pass a `ProxyInputs` of the same shapes, with vis given iff it was given here).
    `fused_loss`: the loss through the fused kernels of csrc/loss.cu instead of eager PyTorch ops (with the
    silhouette term, ops.silhouette_term); `render_silhouettes`: see `predict`, for the eager loss.  The silhouette
    label is one more static label buffer.
    """

    def __init__(self, head: nn.Module, criterion: MultiTaskLoss, smpl: Callable,
                 features: Union[torch.Tensor, ProxyInputs],
                 labels: Dict[str, torch.Tensor], rot6d_to_rotmat: Callable, project_pixels: Optional[Callable],
                 lr: float = 1e-4, world_size: int = 1, warmup: int = 3, fused_loss: bool = False,
                 bucket_mb: float = 8.0, overlap: bool = True, render_silhouettes: Optional[Callable] = None):
        from . import ops
        self.proxy = None
        if isinstance(features, ProxyInputs):
            self.proxy = ProxyInputs(features.masks.clone(), features.keypoints.clone(),
                                     None if features.vis is None else features.vis.clone(), int(features.out_wh),
                                     float(features.std))
            B, K, S = features.masks.shape[0], features.keypoints.shape[1], self.proxy.out_wh
            proxy_cl = _channels_last(head)
            features = torch.empty((B, 1 + K, S, S), dtype=torch.float32, device=features.masks.device,
                                   memory_format=torch.channels_last if proxy_cl else torch.contiguous_format)
        dev = features.device
        if dev.type != "cuda":
            raise RuntimeError("GraphedTrainStep needs CUDA tensors")
        self.head, self.criterion, self.world = head, criterion, int(world_size)
        self.params = [p for p in list(head.parameters()) + list(criterion.parameters()) if p.requires_grad]
        order = list(reversed(self.params))                       # the order the backward fills the gradients in
        self.flat_grad = torch.zeros(sum(p.numel() for p in order), dtype=torch.float32, device=dev)
        self.buckets = []                                          # (begin, end) element ranges of flat_grad
        bucket_of, off, b0, limit = {}, 0, 0, int(bucket_mb * (1 << 20) / 4)
        for p in order:
            p.grad = self.flat_grad[off:off + p.numel()].view_as(p)
            bucket_of[p] = len(self.buckets)
            off += p.numel()
            if off - b0 >= limit:
                self.buckets.append((b0, off))
                b0 = off
        if off > b0:
            self.buckets.append((b0, off))
        counts = [0] * len(self.buckets)
        for p in order:
            counts[bucket_of[p]] += 1
        self.optimiser = torch.optim.Adam(self.params, lr=lr, capturable=True)
        self.features = features if self.proxy is not None else features.clone()
        self.labels = {k: v.clone() for k, v in labels.items()}
        need_verts = _needs_verts(criterion)
        render = _renderer(criterion, fused_loss, render_silhouettes)
        comm = torch.cuda.Stream(device=dev) if (self.world > 1 and overlap) else None
        state = {"pending": list(counts), "sent": [False] * len(self.buckets)}

        def reduce_bucket(b):
            import torch.distributed as dist
            lo, hi = self.buckets[b]
            state["sent"][b] = True
            if comm is None:
                dist.all_reduce(self.flat_grad[lo:hi], op=dist.ReduceOp.AVG)
                return
            comm.wait_stream(torch.cuda.current_stream(dev))      # fork: the bucket's gradients are complete
            with torch.cuda.stream(comm):
                dist.all_reduce(self.flat_grad[lo:hi], op=dist.ReduceOp.AVG)

        if self.world > 1 and overlap:
            def make_hook(b):
                def hook(_p):
                    state["pending"][b] -= 1
                    if state["pending"][b] == 0:
                        reduce_bucket(b)
                return hook
            self._hooks = [p.register_post_accumulate_grad_hook(make_hook(bucket_of[p])) for p in order]

        def one_step():
            self.flat_grad.zero_()
            state["pending"], state["sent"] = list(counts), [False] * len(self.buckets)
            if self.proxy is not None:
                ops.proxy_representation(self.proxy.masks, self.proxy.keypoints, self.proxy.vis, self.proxy.out_wh,
                                         self.proxy.std, channels_last=proxy_cl, out=self.features)
            outputs = predict(head, smpl, self.features, rot6d_to_rotmat, None if fused_loss else project_pixels,
                              need_verts=need_verts, render_silhouettes=render)
            loss, _ = criterion.forward_fused(self.labels, outputs) if fused_loss else criterion(self.labels, outputs)
            loss.backward()
            if self.world > 1:
                for b in range(len(self.buckets)):                 # buckets no hook completed (unused parameters)
                    if not state["sent"][b]:
                        reduce_bucket(b)
                if comm is not None:
                    torch.cuda.current_stream(dev).wait_stream(comm)   # join before the optimiser reads the gradients
            self.optimiser.step()
            return loss.detach()

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):                   # eager: allocations, Adam state, NCCL communicator
                self.last_eager_loss = one_step()
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = one_step()

    def __call__(self, features: Union[torch.Tensor, ProxyInputs], labels: Dict[str, torch.Tensor]) -> torch.Tensor:
        if self.proxy is None:
            self.features.copy_(features, non_blocking=True)
        else:
            if not isinstance(features, ProxyInputs) or (features.vis is None) != (self.proxy.vis is None):
                raise TypeError("this step was captured from ProxyInputs{}: pass the same kind of inputs".format(
                    "" if self.proxy.vis is None else " with vis"))
            self.proxy.masks.copy_(features.masks, non_blocking=True)
            self.proxy.keypoints.copy_(features.keypoints, non_blocking=True)
            if features.vis is not None:
                self.proxy.vis.copy_(features.vis, non_blocking=True)
        for k, v in labels.items():
            self.labels[k].copy_(v, non_blocking=True)
        self.graph.replay()
        return self.loss
