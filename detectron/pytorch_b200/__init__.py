"""detectron.pytorch_b200 -- B200-native (sm_100a) RoIAlign / RoIPool / RoICrop / NMS for
Detectron.pytorch, behind the reference's own Python surface.

    from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.functions.roi_align import RoIAlignFunction
    from detectron.pytorch_b200.model.roi_pooling.functions.roi_pool import RoIPoolFunction
    from detectron.pytorch_b200.model.roi_crop.functions.roi_crop import RoICropFunction
    from detectron.pytorch_b200.model.nms.nms_gpu import nms_gpu

or, to make an unmodified checkout of the reference pick these up under ITS import paths
(`model.*`, `modeling.roi_xfrom.*`), call :func:`install_reference_aliases` before importing
`modeling.model_builder`.
"""
__version__ = "0.1.0"


def install_reference_aliases(overwrite=True, proposals=False, nms=False, segm=False):
    """Register this package's op modules in sys.modules under the reference's import paths.

    After this, `from modeling.roi_xfrom.roi_align.functions.roi_align import RoIAlignFunction`
    (lib/modeling/model_builder.py:13), `from model.roi_pooling.functions.roi_pool import
    RoIPoolFunction` (:11), `from model.roi_crop.functions.roi_crop import RoICropFunction` (:12) and
    `from model.nms.nms_gpu import nms_gpu` resolve to the sm_100a implementations.
    Parent packages that already exist (e.g. the reference's own `modeling`) are left alone; only the
    op sub-packages are injected.  `proposals=True` additionally routes `modeling.generate_proposals` (the RPN proposal
    layer, rpn_heads.py / FPN.py import it) and `modeling.collect_and_distribute_fpn_rpn_proposals` to the device
    implementations (SURVEY.md 8f N1); the latter only implements the inference path, hence opt-in.
    `nms=True` re-points the reference's `utils.boxes.nms` (lib/utils/boxes.py:320-324; called from
    generate_proposals.py:161 and core/test.py:764 with numpy arrays) at the device NMS (`utils/boxes.py` here); the
    reference's `utils.boxes` must be importable for that.
    `segm=True` re-points the reference's `core.test.segm_results` (lib/core/test.py:793-847, called by im_detect_all)
    at `core.test.segm_results` here, bound to the reference's `cfg`: the mask paste and RLE run on the device.  The
    reference's `core.test` and `core.config` must be importable for that.
    """
    import importlib
    import sys
    names = [
        "model.roi_align", "model.roi_align.functions", "model.roi_align.functions.roi_align",
        "model.roi_align.modules", "model.roi_align.modules.roi_align",
        "model.roi_pooling", "model.roi_pooling.functions", "model.roi_pooling.functions.roi_pool",
        "model.roi_pooling.modules", "model.roi_pooling.modules.roi_pool",
        "model.roi_crop", "model.roi_crop.functions", "model.roi_crop.functions.roi_crop",
        "model.roi_crop.modules", "model.roi_crop.modules.roi_crop",
        "model.roi_crop.functions.gridgen", "model.roi_crop.functions.crop_resize", "model.roi_crop.modules.gridgen",
        "model.nms", "model.nms.nms_gpu", "model.nms.nms_wrapper",
        "modeling.roi_xfrom", "modeling.roi_xfrom.roi_align", "modeling.roi_xfrom.roi_align.functions",
        "modeling.roi_xfrom.roi_align.functions.roi_align", "modeling.roi_xfrom.roi_align.modules",
        "modeling.roi_xfrom.roi_align.modules.roi_align", "modeling.roi_xfrom.roi_align.functions.roi_align_fpn",
    ]
    if proposals:
        names += ["modeling.generate_proposals", "modeling.collect_and_distribute_fpn_rpn_proposals"]
    installed = []
    for top in ("model", "modeling"):
        if top not in sys.modules:
            try:
                importlib.import_module(top)            # the reference's own package, if on sys.path
            except ImportError:
                sys.modules[top] = importlib.import_module(__name__ + "." + top)
                installed.append(top)
    for name in names:
        if name in sys.modules and not overwrite:
            continue
        mod = importlib.import_module(__name__ + "." + name)
        sys.modules[name] = mod
        parent, _, child = name.rpartition(".")
        if parent in sys.modules:
            setattr(sys.modules[parent], child, mod)
        installed.append(name)
    if nms:
        ref_boxes = importlib.import_module("utils.boxes")          # the reference's module
        ref_boxes.nms = importlib.import_module(__name__ + ".utils.boxes").nms
        installed.append("utils.boxes.nms")
    if segm:
        ref_test = importlib.import_module("core.test")             # the reference's module
        ref_cfg = importlib.import_module("core.config").cfg
        impl = importlib.import_module(__name__ + ".core.test").segm_results
        ref_test.segm_results = lambda cls_boxes, masks, ref_boxes, im_h, im_w: impl(cls_boxes, masks, ref_boxes, im_h, im_w, cfg=ref_cfg)
        installed.append("core.test.segm_results")
    return installed
