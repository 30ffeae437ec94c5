"""Case tables shared by the golden generator (tests/golden/make_golden.py) and the tests that re-create the inputs."""

PRE_CASES = [  # (source h, w, seed, letterbox kwargs)
    (60, 90, 1, dict(new_shape=(96, 128), auto=False)),
    (123, 77, 2, dict(new_shape=(96, 128), auto=False)),
    (200, 150, 3, dict(new_shape=(96, 128), auto=False)),          # down-scaling
    (48, 64, 4, dict(new_shape=(96, 128), auto=False)),            # exact 2x up-scaling
    (96, 128, 5, dict(new_shape=(96, 128), auto=False)),           # no resize at all
    (70, 101, 6, dict(new_shape=160, auto=True, stride=32)),       # minimum-rectangle padding
    (70, 101, 7, dict(new_shape=(96, 128), auto=False, scaleup=False)),
    (50, 120, 8, dict(new_shape=(64, 64), auto=False, scaleFill=True)),
]

SIGNATURE_SURFACE = [  # (module path in the reference == module under yolov5_b200, qualified name): the drop-in call signatures
    ("models.yolo", "DetectionModel.__init__"), ("models.yolo", "DetectionModel.forward"), ("models.yolo", "SegmentationModel.__init__"),
    ("models.yolo", "Detect.__init__"), ("models.yolo", "Segment.__init__"), ("models.yolo", "parse_model"),
    ("models.common", "Conv.__init__"), ("models.common", "Bottleneck.__init__"), ("models.common", "C3.__init__"),
    ("models.common", "SPPF.__init__"), ("models.common", "Concat.__init__"), ("models.common", "Proto.__init__"), ("models.common", "autopad"),
    ("models.experimental", "attempt_load"),
    ("utils.general", "non_max_suppression"), ("utils.general", "scale_boxes"), ("utils.general", "xyxy2xywh"),
    ("utils.loss", "ComputeLoss.__init__"), ("utils.loss", "ComputeLoss.__call__"), ("utils.loss", "ComputeLoss.build_targets"),
    ("utils.metrics", "process_batch"),
    ("utils.torch_utils", "fuse_conv_and_bn"), ("utils.torch_utils", "smart_DDP"), ("utils.torch_utils", "de_parallel"),
    ("utils.torch_utils", "ModelEMA.__init__"), ("utils.torch_utils", "ModelEMA.update"), ("utils.torch_utils", "ModelEMA.update_attr"),
    ("utils.torch_utils", "smart_optimizer"),
    ("utils.augmentations", "letterbox"),
    ("utils.segment.general", "crop_mask"), ("utils.segment.general", "process_mask"), ("utils.segment.general", "process_mask_native"),
]
