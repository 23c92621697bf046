"""face_detection_tflite_b200 — B200 (sm_100a) implementation of the face_detection_tflite
detection hot path behind the plugin's own API surface.

    from face_detection_tflite_b200 import FaceDetector, FaceDetectionModel, FaceDetectionMode
    det = FaceDetector.create(FaceDetectionModel.shortRange)
    faces = det.detectFacesFromMatBytes(bgr_bytes, width=1280, height=720, mode=FaceDetectionMode.fast)

Compute lives in csrc/ (hand-written CUDA behind the C ABI of include/fdt_api.h); this package is
only the host-side mirror of the reference's Dart interface."""
from .face_detector import FaceCropSpec, FaceDetector, FormatException, StateError
from .face_gates import applyDetectionGates, applyFaceGates, boxVisibleWidthFraction, validateFaceGates
from .face_types import (BoundingBox, Detection, Eye, EyePair, Face, FaceDetectionMode, FaceDetectionModel, FaceLandmarkType,
                         FaceMesh, Point, RectF, Size, irisCenterFromPoints)

__all__ = ["FaceDetector", "FaceCropSpec", "StateError", "FormatException", "BoundingBox", "Detection", "Face", "FaceDetectionMode",
           "FaceDetectionModel", "FaceLandmarkType", "FaceMesh", "Point", "RectF", "Size", "Eye", "EyePair",
           "irisCenterFromPoints", "applyDetectionGates", "applyFaceGates", "boxVisibleWidthFraction", "validateFaceGates"]
