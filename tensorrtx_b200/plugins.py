"""Host-side mirror of the reference's plugin / helper interface for the hot path.

Same names, argument meaning and error behaviour as the reference classes, so the parity tests read
like the reference's call sites:

  YoloLayerPlugin        yolov8/plugin/yololayer.h:7-85      (IPluginV2IOExt; "YoloLayer_TRT" v1)
  YoloLayerPluginV5      yolov5/plugin/yololayer.h:10-82
  YoloPluginCreator      yolov8/plugin/yololayer.h:87-109    (field "combinedInfo", block.cpp:264-296)
  DecodePlugin           retinaface/decode.h:22-83           ("Decode_TRT" v1)
  RpnDecodePlugin / RpnNmsPlugin / PredictorDecodePlugin / BatchedNmsPlugin   rcnn/*Plugin.h
  batch_nms / cuda_decode+cuda_nms / cuda_batch_preprocess   yolov8/include/postprocess.h, preprocess.h

All compute goes through the C ABI of libtrtx_hot.so (include/trtx_hot.h); torch is used only for
device memory and streams.  There is no CPU fallback: without the library these classes raise.
"""
from __future__ import annotations

import ctypes as C
import math
import struct
from typing import Sequence

import torch

from . import _lib as L


def _ptr(t) -> int:
    if isinstance(t, torch.Tensor):
        if not t.is_cuda:
            raise L.TrtxError("expected a CUDA tensor (device pointer); host buffers are not accepted here")
        if not t.is_contiguous():
            raise L.TrtxError("tensor must be contiguous (TensorFormat::kLINEAR)")
        return t.data_ptr()
    return int(t)


def _stream(stream=None) -> int:
    if stream is None:
        return torch.cuda.current_stream().cuda_stream
    if isinstance(stream, torch.cuda.Stream):
        return stream.cuda_stream
    return int(stream)


def _tune(params, slices: int = 0, rows: int = 0, tma: int = 0, stages: int = 0, box: int = 0, nms_threads: int = 0) -> None:
    """Per-plugin launch tuning of the scan kernel and of the fused NMS (trtx_yolo_params.tune_*; 0 = default).  Plain
    data inside the plugin's own parameter block -- nothing global, clones / other plugins are unaffected."""
    params.tune_class_slices, params.tune_rows_in_flight = int(slices), int(rows)
    params.tune_tma_pipeline, params.tune_tma_stages, params.tune_box_prefetch = int(tma), int(stages), int(box)
    params.tune_nms_threads = int(nms_threads)


def float_le_threshold(x: float) -> float:
    """Largest fp32 t with t <= x: `(double)conf <= x`  <=>  `conf <= t` in fp32 (retinaface 0.1 / 0.02 literals)."""
    t = struct.unpack("f", struct.pack("f", x))[0]
    if t > x:
        t = float(torch.nextafter(torch.tensor(t, dtype=torch.float32), torch.tensor(-math.inf)).item())
    return t


# --------------------------------------------------------------------------------------------------
# YoloLayer_TRT, anchor-free (yolov8 / yolo11 / yolov12 / yolov13 ...)
# --------------------------------------------------------------------------------------------------
class YoloLayerPlugin:
    PLUGIN_TYPE = "YoloLayer_TRT"
    PLUGIN_VERSION = "1"
    DET_FLOATS = 90  # sizeof(Detection)/4, yolov8/include/types.h:4-12

    def __init__(self, classCount: int, numberofpoints: int, confthreshkeypoints: float, netWidth: int,
                 netHeight: int, maxOut: int, is_segmentation: bool, is_pose: bool, is_obb: bool,
                 strides: Sequence[int], in_dtype: int = L.F32):
        self.mClassCount = int(classCount)
        self.mNumberofpoints = int(numberofpoints)
        self.mConfthreshkeypoints = float(confthreshkeypoints)
        self.mYoloV8NetWidth = int(netWidth)
        self.mYoloV8netHeight = int(netHeight)
        self.mMaxOutObject = int(maxOut)
        self.is_segmentation_ = bool(is_segmentation)
        self.is_pose_ = bool(is_pose)
        self.is_obb_ = bool(is_obb)
        self.mStrides = [int(s) for s in strides]
        self.mThreadCount = 256  # serialized by the reference (yololayer.cu:80); unused here
        self.mPluginNamespace = ""
        self.in_dtype = in_dtype
        self._lib = L.load()
        p = L.YoloParams()
        arr = (C.c_int * len(self.mStrides))(*self.mStrides)
        L.check(self._lib.trtx_yolo_params_init_v8(C.byref(p), self.mClassCount, self.mYoloV8NetWidth,
                                                  self.mYoloV8netHeight, self.mMaxOutObject, arr, len(self.mStrides)),
                "trtx_yolo_params_init_v8")
        p.det_floats = self.DET_FLOATS
        p.is_seg, p.is_pose, p.is_obb = int(self.is_segmentation_), int(self.is_pose_), int(self.is_obb_)
        p.num_kpts = self.mNumberofpoints
        p.kpt_thresh = self.mConfthreshkeypoints
        p.gate = 0.1  # literal of yololayer.cu:203
        p.in_dtype = in_dtype
        self.params = p

    # ---- IPluginV2 surface ----
    def tune(self, **kw) -> "YoloLayerPlugin":
        _tune(self.params, **kw)
        return self

    def getNbOutputs(self) -> int:
        return 1

    def getOutputDimensions(self, index=0, inputs=None, nbInputDims=0):
        total = self.mMaxOutObject * self.DET_FLOATS  # yololayer.cu:107-111
        return (total + 1, 1, 1)

    def output_elems(self) -> int:
        return 1 + self.mMaxOutObject * self.DET_FLOATS

    def initialize(self) -> int:
        return 0

    def terminate(self) -> None:
        pass

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return int(self._lib.trtx_yolo_workspace_size(C.byref(self.params), int(maxBatchSize)))

    def enqueue(self, batchSize: int, inputs, outputs, workspace, stream=None) -> int:
        """inputs: one device tensor per stride [B, C, g]; outputs[0]: [B, 1+maxOut*90] fp32; returns 0 on success."""
        ptrs = L.ptr_array([_ptr(t) for t in inputs])
        ws_bytes = workspace.numel() * workspace.element_size() if isinstance(workspace, torch.Tensor) else self.getWorkspaceSize(batchSize)
        return int(self._lib.trtx_yolo_decode_enqueue(C.byref(self.params), int(batchSize), ptrs, _ptr(outputs[0]),
                                                      _ptr(workspace), ws_bytes, _stream(stream)))

    def supportsFormatCombination(self, pos, inOut, nbInputs, nbOutputs) -> bool:
        fmt, dtype = inOut[pos]
        if pos < nbInputs:
            return fmt == "kLINEAR" and dtype in (("kFLOAT",) if self.in_dtype == L.F32 else ("kHALF",))
        return fmt == "kLINEAR" and dtype == "kFLOAT"

    def getPluginType(self) -> str:
        return self.PLUGIN_TYPE

    def getPluginVersion(self) -> str:
        return self.PLUGIN_VERSION

    def getOutputDataType(self, index, inputTypes, nbInputs) -> str:
        return "kFLOAT"

    def setPluginNamespace(self, ns: str) -> None:
        self.mPluginNamespace = ns

    def getPluginNamespace(self) -> str:
        return self.mPluginNamespace

    def destroy(self) -> None:
        pass

    def clone(self) -> "YoloLayerPlugin":
        p = YoloLayerPlugin(self.mClassCount, self.mNumberofpoints, self.mConfthreshkeypoints, self.mYoloV8NetWidth,
                            self.mYoloV8netHeight, self.mMaxOutObject, self.is_segmentation_, self.is_pose_,
                            self.is_obb_, self.mStrides, self.in_dtype)
        p.setPluginNamespace(self.mPluginNamespace)
        return p

    # ---- serialization: byte layout of yololayer.cu:75-101 ----
    def getSerializationSize(self) -> int:
        return 4 * 8 + 4 * len(self.mStrides) + 3

    def serialize(self) -> bytes:
        d = struct.pack("<iifiiiii", self.mClassCount, self.mNumberofpoints, self.mConfthreshkeypoints,
                        self.mThreadCount, self.mYoloV8NetWidth, self.mYoloV8netHeight, self.mMaxOutObject,
                        len(self.mStrides))
        d += struct.pack(f"<{len(self.mStrides)}i", *self.mStrides)
        d += struct.pack("<???", self.is_segmentation_, self.is_pose_, self.is_obb_)
        assert len(d) == self.getSerializationSize()
        return d

    @classmethod
    def deserialize(cls, data: bytes) -> "YoloLayerPlugin":
        cc, nk, kt, tc, w, h, mo, ns = struct.unpack_from("<iifiiiii", data, 0)
        strides = struct.unpack_from(f"<{ns}i", data, 32)
        seg, pose, obb = struct.unpack_from("<???", data, 32 + 4 * ns)
        if 32 + 4 * ns + 3 != len(data):
            raise L.TrtxError("YoloLayerPlugin.deserialize: length mismatch")  # assert(d == a + length)
        p = cls(cc, nk, kt, w, h, mo, seg, pose, obb, strides)
        p.mThreadCount = tc
        return p


class YoloPluginCreator:
    """yolov8/plugin/yololayer.cu:318-369."""

    def __init__(self):
        self.mNamespace = ""

    def getPluginName(self) -> str:
        return "YoloLayer_TRT"

    def getPluginVersion(self) -> str:
        return "1"

    def getFieldNames(self):
        return []

    def setPluginNamespace(self, ns: str) -> None:
        self.mNamespace = ns

    def getPluginNamespace(self) -> str:
        return self.mNamespace

    def createPlugin(self, name: str, fc: dict) -> YoloLayerPlugin:
        if len(fc) != 1 or "combinedInfo" not in fc:  # assert(fc->nbFields == 1), assert(strcmp(...)==0)
            raise L.TrtxError("YoloPluginCreator.createPlugin expects exactly one field 'combinedInfo'")
        ci = [int(v) for v in fc["combinedInfo"]]
        if len(ci) < 10:
            raise L.TrtxError("combinedInfo needs 9 net-info ints + at least one stride")
        obj = YoloLayerPlugin(ci[0], ci[1], float(ci[2]), ci[3], ci[4], ci[5], bool(ci[6]), bool(ci[7]), bool(ci[8]), ci[9:])
        obj.setPluginNamespace(self.mNamespace)
        return obj

    def deserializePlugin(self, name: str, data: bytes) -> YoloLayerPlugin:
        obj = YoloLayerPlugin.deserialize(data)
        obj.setPluginNamespace(self.mNamespace)
        return obj


# --------------------------------------------------------------------------------------------------
# YoloLayer_TRT, anchor-based (yolov5 / yolov7 ...)
# --------------------------------------------------------------------------------------------------
class YoloKernel:
    """yolov5/src/types.h:5-9."""

    def __init__(self, width: int, height: int, anchors: Sequence[float]):
        self.width, self.height = int(width), int(height)
        self.anchors = [float(a) for a in anchors]
        assert len(self.anchors) == 6


class YoloLayerPluginV5:
    PLUGIN_TYPE = "YoloLayer_TRT"
    PLUGIN_VERSION = "1"
    DET_FLOATS = 38  # yolov5/src/types.h:11-16

    def __init__(self, classCount: int, netWidth: int, netHeight: int, maxOut: int, is_segmentation: bool,
                 vYoloKernel: Sequence[YoloKernel], in_dtype: int = L.F32):
        self.mClassCount, self.mYoloV5NetWidth, self.mYoloV5NetHeight = int(classCount), int(netWidth), int(netHeight)
        self.mMaxOutObject = int(maxOut)
        self.is_segmentation_ = bool(is_segmentation)
        self.mYoloKernel = list(vYoloKernel)
        self.mKernelCount = len(self.mYoloKernel)
        self.mThreadCount = 256
        self.mPluginNamespace = ""
        self._lib = L.load()
        p = L.YoloParams()
        p.variant = L.YOLO_V5
        p.num_classes = self.mClassCount
        p.net_w, p.net_h = self.mYoloV5NetWidth, self.mYoloV5NetHeight
        p.max_out = self.mMaxOutObject
        p.det_floats = self.DET_FLOATS
        p.num_levels = self.mKernelCount
        for i, k in enumerate(self.mYoloKernel):
            p.grid_w[i], p.grid_h[i] = k.width, k.height
            for j in range(6):
                p.anchors[i][j] = k.anchors[j]
        p.is_seg = int(self.is_segmentation_)
        p.gate = 0.1  # kIgnoreThresh, yolov5/src/config.h:38
        p.in_dtype = in_dtype
        self.params = p

    def tune(self, **kw) -> "YoloLayerPlugin":
        _tune(self.params, **kw)
        return self

    def getNbOutputs(self) -> int:
        return 1

    def output_elems(self) -> int:
        return 1 + self.mMaxOutObject * self.DET_FLOATS

    def getOutputDimensions(self, index=0, inputs=None, nbInputDims=0):
        return (self.mMaxOutObject * self.DET_FLOATS + 1, 1, 1)

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return int(self._lib.trtx_yolo_workspace_size(C.byref(self.params), int(maxBatchSize)))

    def enqueue(self, batchSize: int, inputs, outputs, workspace, stream=None) -> int:
        ptrs = L.ptr_array([_ptr(t) for t in inputs])
        ws_bytes = workspace.numel() * workspace.element_size()
        return int(self._lib.trtx_yolo_decode_enqueue(C.byref(self.params), int(batchSize), ptrs, _ptr(outputs[0]),
                                                      _ptr(workspace), ws_bytes, _stream(stream)))

    def getPluginType(self) -> str:
        return self.PLUGIN_TYPE

    def getPluginVersion(self) -> str:
        return self.PLUGIN_VERSION

    def clone(self) -> "YoloLayerPluginV5":
        p = YoloLayerPluginV5(self.mClassCount, self.mYoloV5NetWidth, self.mYoloV5NetHeight, self.mMaxOutObject,
                              self.is_segmentation_, self.mYoloKernel, self.params.in_dtype)
        p.mPluginNamespace = self.mPluginNamespace
        return p

    # byte layout of yolov5/plugin/yololayer.cu:48-83
    def serialize(self) -> bytes:
        d = struct.pack("<iiiiii?", self.mClassCount, self.mThreadCount, self.mKernelCount, self.mYoloV5NetWidth,
                        self.mYoloV5NetHeight, self.mMaxOutObject, self.is_segmentation_)
        for k in self.mYoloKernel:
            d += struct.pack("<ii6f", k.width, k.height, *k.anchors)
        return d

    def getSerializationSize(self) -> int:
        return 25 + 32 * self.mKernelCount

    @classmethod
    def deserialize(cls, data: bytes) -> "YoloLayerPluginV5":
        cc, tc, kc, w, h, mo, seg = struct.unpack_from("<iiiiii?", data, 0)
        ks = []
        for i in range(kc):
            v = struct.unpack_from("<ii6f", data, 25 + 32 * i)
            ks.append(YoloKernel(v[0], v[1], v[2:]))
        if 25 + 32 * kc != len(data):
            raise L.TrtxError("YoloLayerPluginV5.deserialize: length mismatch")
        p = cls(cc, w, h, mo, seg, ks)
        p.mThreadCount = tc
        return p


class YoloLayerPluginV7(YoloLayerPluginV5):
    """yolov7/plugin/yololayer.h:9-73 (same kernel arithmetic as yolov5, yolov7/plugin/yololayer.cu:152-200, but
    Detection = 6 floats, yolov7/include/types.h:11-16; also yolov10 / yolov13 style rows).  No segmentation flag:
    ctor (classCount, netWidth, netHeight, maxOut, vYoloKernel), serialization without the bool."""
    DET_FLOATS = 6

    def __init__(self, classCount: int, netWidth: int, netHeight: int, maxOut: int, vYoloKernel: Sequence[YoloKernel],
                 in_dtype: int = L.F32):
        super().__init__(classCount, netWidth, netHeight, maxOut, False, vYoloKernel, in_dtype)

    def clone(self) -> "YoloLayerPluginV7":
        p = YoloLayerPluginV7(self.mClassCount, self.mYoloV5NetWidth, self.mYoloV5NetHeight, self.mMaxOutObject,
                              self.mYoloKernel, self.params.in_dtype)
        p.mPluginNamespace = self.mPluginNamespace
        return p

    def serialize(self) -> bytes:  # yolov7/plugin/yololayer.cu:62-77
        d = struct.pack("<iiiiii", self.mClassCount, self.mThreadCount, self.mKernelCount, self.mYoloV5NetWidth,
                        self.mYoloV5NetHeight, self.mMaxOutObject)
        for k in self.mYoloKernel:
            d += struct.pack("<ii6f", k.width, k.height, *k.anchors)
        return d

    def getSerializationSize(self) -> int:
        return 24 + 32 * self.mKernelCount

    @classmethod
    def deserialize(cls, data: bytes) -> "YoloLayerPluginV7":
        cc, tc, kc, w, h, mo = struct.unpack_from("<iiiiii", data, 0)
        if 24 + 32 * kc != len(data):
            raise L.TrtxError("YoloLayerPluginV7.deserialize: length mismatch")
        ks = []
        for i in range(kc):
            v = struct.unpack_from("<ii6f", data, 24 + 32 * i)
            ks.append(YoloKernel(v[0], v[1], v[2:]))
        p = cls(cc, w, h, mo, ks)
        p.mThreadCount = tc
        return p


class YoloKernelV3:
    """Yolo::YoloKernel of yolov3-spp/yololayer.h:20-26: width, height (dynamic, -1 until enqueue), stride, anchors."""

    def __init__(self, width: int, height: int, stride: int, anchors: Sequence[float]):
        self.width, self.height, self.stride = int(width), int(height), int(stride)
        self.anchors = [float(a) for a in anchors]
        assert len(self.anchors) == 6


# yolo1..3 of yolov3-spp/yololayer.h:27-44 (the plugin's level order: stride 32, 16, 8)
YOLOV3_KERNELS = (YoloKernelV3(-1, -1, 32, (116, 90, 156, 198, 373, 326)),
                  YoloKernelV3(-1, -1, 16, (30, 61, 62, 45, 59, 119)),
                  YoloKernelV3(-1, -1, 8, (10, 13, 16, 30, 33, 23)))


class YoloLayerPluginV3:
    """yolov3-spp/yololayer.h:58-121 (IPluginV2DynamicExt "YoloLayer_TRT" v1; yolov3 / yolov4 carry the same plugin).
    The reference compiles CLASS_NUM, the kernels and MAX_OUTPUT_BBOX_COUNT in; here they are constructor arguments with
    the reference's values as defaults.  enqueue() takes the grids from the input tensors like the reference
    (yololayer.cu:207-216)."""
    PLUGIN_TYPE = "YoloLayer_TRT"
    PLUGIN_VERSION = "1"
    DET_FLOATS = 7  # x,y,w,h, det_confidence, class_id, class_confidence (yololayer.h:47-53)

    def __init__(self, classCount: int = 80, kernels: Sequence[YoloKernelV3] = YOLOV3_KERNELS, maxOut: int = 1000,
                 in_dtype: int = L.F32):
        self.mClassCount, self.mYoloKernel, self.mMaxOutObject = int(classCount), list(kernels), int(maxOut)
        self.mKernelCount, self.mThreadCount, self.mPluginNamespace = len(self.mYoloKernel), 256, ""
        self._lib = L.load()
        p = L.YoloParams()
        p.variant = L.YOLO_V3
        p.num_classes, p.max_out, p.det_floats, p.num_levels = self.mClassCount, self.mMaxOutObject, self.DET_FLOATS, self.mKernelCount
        for i, k in enumerate(self.mYoloKernel):
            p.strides[i] = k.stride
            p.grid_w[i], p.grid_h[i] = max(k.width, 1), max(k.height, 1)
            for j in range(6):
                p.anchors[i][j] = k.anchors[j]
        p.gate = 0.1  # IGNORE_THRESH, yololayer.h:15
        p.in_dtype = in_dtype
        self.params = p

    def tune(self, **kw) -> "YoloLayerPluginV3":
        _tune(self.params, **kw)
        return self

    def getNbOutputs(self) -> int:
        return 1

    def output_elems(self) -> int:
        return 1 + self.mMaxOutObject * self.DET_FLOATS

    def configure(self, inputs) -> None:
        """grid = dims 2, 3 of every input tensor [B, 3*(5+nc), gh, gw] (yololayer.cu:209-212)."""
        for i, t in enumerate(inputs):
            self.params.grid_h[i], self.params.grid_w[i] = int(t.shape[2]), int(t.shape[3])

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return int(self._lib.trtx_yolo_workspace_size(C.byref(self.params), int(maxBatchSize)))

    def enqueue(self, inputs, outputs, workspace=None, stream=None) -> int:
        """IPluginV2DynamicExt::enqueue: batch = inputs[0].shape[0]."""
        self.configure(inputs)
        batch = int(inputs[0].shape[0])
        if workspace is None:
            workspace = torch.empty(self.getWorkspaceSize(batch), dtype=torch.uint8, device=inputs[0].device)
        ptrs = L.ptr_array([_ptr(t) for t in inputs])
        return int(self._lib.trtx_yolo_decode_enqueue(C.byref(self.params), batch, ptrs, _ptr(outputs[0]), _ptr(workspace),
                                                      workspace.numel() * workspace.element_size(), _stream(stream)))

    def getPluginType(self) -> str:
        return self.PLUGIN_TYPE

    def getPluginVersion(self) -> str:
        return self.PLUGIN_VERSION

    def clone(self) -> "YoloLayerPluginV3":
        p = YoloLayerPluginV3(self.mClassCount, self.mYoloKernel, self.mMaxOutObject, self.params.in_dtype)
        p.mPluginNamespace = self.mPluginNamespace
        return p

    # byte layout of yolov3-spp/yololayer.cu:36-71: classCount, threadCount, kernelCount, kernels {w, h, stride, anchors[6]}
    def serialize(self) -> bytes:
        d = struct.pack("<iii", self.mClassCount, self.mThreadCount, self.mKernelCount)
        for k in self.mYoloKernel:
            d += struct.pack("<iii6f", k.width, k.height, k.stride, *k.anchors)
        return d

    def getSerializationSize(self) -> int:
        return 12 + 36 * self.mKernelCount

    @classmethod
    def deserialize(cls, data: bytes) -> "YoloLayerPluginV3":
        cc, tc, kc = struct.unpack_from("<iii", data, 0)
        if 12 + 36 * kc != len(data):
            raise L.TrtxError("YoloLayerPluginV3.deserialize: length mismatch")
        ks = []
        for i in range(kc):
            v = struct.unpack_from("<iii6f", data, 12 + 36 * i)
            ks.append(YoloKernelV3(v[0], v[1], v[2], v[3:]))
        p = cls(cc, ks)
        p.mThreadCount = tc
        return p


class YoloLayerPlugin26:
    """yolo26/plugin/yololayer.h:10-77 ("YoloLayer_TRT" v1 of the NMS-free yolo26 heads): ctor (classCount, numberOfPoints,
    maxDetections, isDetection, isSegmentation, isPose, isObb, anchor_count); setPluginDeviceParams(confThreshold) of the
    reference is the `conf_thresh` argument here (no device global).  One input [B, anchor_count, 4+nc(+1)]."""
    PLUGIN_TYPE = "YoloLayer_TRT"
    PLUGIN_VERSION = "1"
    DET_FLOATS = 90  # yolo26/include/types.h

    def __init__(self, classCount: int, numberOfPoints: int, maxDetections: int, isDetection: bool, isSegmentation: bool,
                 isPose: bool, isObb: bool, anchor_count: int, conf_thresh: float = 0.4):
        self.mClassCount, self.mNumberOfPoints, self.mMaxDetections = int(classCount), int(numberOfPoints), int(maxDetections)
        self.mIsDetection, self.mIsSegmentation, self.mIsPose, self.mIsObb = bool(isDetection), bool(isSegmentation), bool(isPose), bool(isObb)
        self.mAnchorCount, self.mThreadCount, self.mPluginNamespace = int(anchor_count), 256, ""
        self._lib = L.load()
        p = L.YoloParams()
        p.variant = L.YOLO_V26
        p.num_classes, p.max_out, p.det_floats, p.num_levels = self.mClassCount, self.mMaxDetections, self.DET_FLOATS, 1
        p.grid_h[0], p.grid_w[0] = 1, self.mAnchorCount
        p.is_seg, p.is_pose, p.is_obb = int(self.mIsSegmentation), int(self.mIsPose), int(self.mIsObb)
        p.num_kpts = self.mNumberOfPoints
        p.gate = float(conf_thresh)  # d_confThreshold, yololayer.cu:9 / setPluginDeviceParams :31-33
        p.in_dtype = L.F32
        self.params = p

    def getNbOutputs(self) -> int:
        return 1

    def output_elems(self) -> int:
        return 1 + self.mMaxDetections * self.DET_FLOATS

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return int(self._lib.trtx_yolo_workspace_size(C.byref(self.params), int(maxBatchSize)))

    def enqueue(self, batchSize: int, inputs, outputs, workspace, stream=None) -> int:
        ptrs = L.ptr_array([_ptr(inputs[0])])
        return int(self._lib.trtx_yolo_decode_enqueue(C.byref(self.params), int(batchSize), ptrs, _ptr(outputs[0]), _ptr(workspace),
                                                      workspace.numel() * workspace.element_size(), _stream(stream)))

    def getPluginType(self) -> str:
        return self.PLUGIN_TYPE

    def getPluginVersion(self) -> str:
        return self.PLUGIN_VERSION

    def clone(self) -> "YoloLayerPlugin26":
        p = YoloLayerPlugin26(self.mClassCount, self.mNumberOfPoints, self.mMaxDetections, self.mIsDetection, self.mIsSegmentation,
                              self.mIsPose, self.mIsObb, self.mAnchorCount, self.params.gate)
        p.mPluginNamespace = self.mPluginNamespace
        return p

    # byte layout of yolo26/plugin/yololayer.cu:68-100 (4 ints, 4 bools, 1 int)
    def serialize(self) -> bytes:
        return struct.pack("<iiii????i", self.mClassCount, self.mNumberOfPoints, self.mThreadCount, self.mMaxDetections,
                           self.mIsDetection, self.mIsSegmentation, self.mIsPose, self.mIsObb, self.mAnchorCount)

    def getSerializationSize(self) -> int:
        return 24

    @classmethod
    def deserialize(cls, data: bytes, conf_thresh: float = 0.4) -> "YoloLayerPlugin26":
        if len(data) != 24:
            raise L.TrtxError("YoloLayerPlugin26.deserialize: length mismatch")
        cc, nk, tc, md, d, sg, po, ob, ac = struct.unpack("<iiii????i", data)
        p = cls(cc, nk, md, d, sg, po, ob, ac, conf_thresh)
        p.mThreadCount = tc
        return p


# --------------------------------------------------------------------------------------------------
# NMS helpers (postprocess.h)
# --------------------------------------------------------------------------------------------------
def nms_params(box_format=L.BOX_LTRB, mode=L.NMS_GREEDY, conf_thresh=0.5, nms_thresh=0.45, max_det=1000,
               class_aware=True, tie_break_x0=None, extra_floats=0, extra_offset=0) -> L.NmsParams:
    q = L.NmsParams()
    q.box_format, q.mode = box_format, mode
    q.conf_thresh, q.nms_thresh = conf_thresh, nms_thresh
    q.max_det = max_det
    q.class_aware = int(class_aware)
    q.tie_break_x0 = int(box_format in (L.BOX_LTRB, L.BOX_OBB) if tie_break_x0 is None else tie_break_x0)  # v8 cmp, postprocess.cpp:87-92
    q.extra_floats, q.extra_offset = extra_floats, extra_offset
    return q


def batch_nms(output: torch.Tensor, batch_size: int, output_size: int, conf_thresh: float, nms_thresh: float = 0.5,
              box_format: int = L.BOX_LTRB, det_floats: int = 90, max_det: int | None = None, mode: int = L.NMS_GREEDY,
              extra_floats: int = 0, extra_offset: int = 0, return_index: bool = False, stream=None):
    """GPU drop-in for batch_nms() (yolov8/src/postprocess.cpp:123-129): `output` is the plugin buffer
    [batch, output_size] on the device; returns the compact buffer [batch, 1 + max_det*(7+extra)]."""
    lib = L.load()
    max_rows = (output_size - 1) // det_floats
    max_det = max_det or max_rows
    q = nms_params(box_format, mode, conf_thresh, nms_thresh, max_det, box_format != L.BOX_RETINA,
                   extra_floats=extra_floats, extra_offset=extra_offset)
    R = 7 + extra_floats
    out = torch.empty((batch_size, 1 + max_det * R), dtype=torch.float32, device=output.device)
    idx = torch.empty((batch_size, max_det), dtype=torch.int32, device=output.device) if return_index else None
    ws_bytes = int(lib.trtx_nms_workspace_size(C.byref(q), batch_size, max_rows))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=output.device)
    L.check(lib.trtx_nms_enqueue(C.byref(q), batch_size, _ptr(output), max_rows, det_floats, _ptr(out),
                                 _ptr(idx) if idx is not None else None, _ptr(ws), ws_bytes, _stream(stream)),
            "trtx_nms_enqueue")
    return (out, idx) if return_index else out


def batch_nms_obb(output: torch.Tensor, batch_size: int, output_size: int, conf_thresh: float, nms_thresh: float = 0.5,
                  max_det: int | None = None, mode: int = L.NMS_GREEDY, return_index: bool = False, stream=None):
    """GPU drop-in for batch_nms_obb() (yolov8/src/postprocess.cpp:387-393; mode=NMS_ONESHOT: cuda_decode_obb +
    cuda_nms_obb, postprocess.cu:7-40,147-193): oriented boxes, ProbIoU.  Returns [batch, 1 + max_det*8] rows
    (cx, cy, w, h, conf, cls, keep, angle) -- the 8-float element decode_kernel_obb writes."""
    return batch_nms(output, batch_size, output_size, conf_thresh, nms_thresh, box_format=L.BOX_OBB, det_floats=90,
                     max_det=max_det, mode=mode, extra_floats=1, extra_offset=89, return_index=return_index, stream=stream)


def process_mask(proto: torch.Tensor, dets: torch.Tensor, max_rows: int, row_floats: int = 39, coeff_offset: int = 7,
                 max_masks: int = 100, net_w: int = 640, net_h: int = 640, variant: int = L.YOLO_V8, out=None, stream=None):
    """GPU drop-in for process_mask() (yolov8/yolov8_seg.cpp:36-60, yolov5/src/postprocess.cpp:106-125) for the whole
    batch: proto [B, 32, net_h/4, net_w/4]; dets [B, 1 + max_rows*row_floats] (count, rows; e.g. batch_nms(...,
    extra_floats=32, extra_offset=6) output) -> masks [B, max_masks, net_h, net_w]; slots >= count are not written."""
    lib = L.load()
    B, nm, mh, mw = proto.shape
    q = L.MaskParams(variant, net_w, net_h, mw, mh, nm, row_floats, coeff_offset, max_masks)
    if out is None:
        out = torch.zeros((B, max_masks, net_h, net_w), dtype=torch.float32, device=proto.device)
    L.check(lib.trtx_process_mask_enqueue(C.byref(q), B, _ptr(proto), _ptr(dets), max_rows, _ptr(out), _stream(stream)),
            "trtx_process_mask_enqueue")
    return out


class FusedYoloDecodeNms:
    """YoloLayer inputs -> compact detections in two launches (scan + NMS), no plugin-format round trip.
    Owns its workspace/output buffers (allocated once; enqueue itself allocates nothing)."""

    def __init__(self, plugin, max_batch: int, conf_thresh=0.5, nms_thresh=0.45, max_det=None, mode=L.NMS_GREEDY,
                 device="cuda", return_index=True):
        self.plugin = plugin
        self.max_batch = max_batch
        v5 = plugin.params.variant in (L.YOLO_V5, L.YOLO_V3)  # anchor-based rows are cx, cy, w, h
        self.max_det = max_det or plugin.mMaxOutObject
        self.q = nms_params(L.BOX_CXCYWH if v5 else L.BOX_LTRB, mode, conf_thresh, nms_thresh, self.max_det, True)
        self._lib = L.load()
        self.ws_bytes = plugin.getWorkspaceSize(max_batch)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=device)
        self.out = torch.empty((max_batch, 1 + self.max_det * 7), dtype=torch.float32, device=device)
        self.idx = torch.empty((max_batch, self.max_det), dtype=torch.int32, device=device) if return_index else None

    def enqueue(self, batch: int, inputs, stream=None, out=None, idx=None, gather=None):
        """gather: an L.Gather descriptor (pipeline.PeerGather.desc) -> the NMS kernel also stores its rows into every
        rank's gathered buffer (trtx_yolo_decode_nms_gather_enqueue)."""
        ptrs = L.ptr_array([_ptr(t) for t in inputs])
        out = self.out if out is None else out
        idx = self.idx if idx is None else idx
        if gather is not None:
            L.check(self._lib.trtx_yolo_decode_nms_gather_enqueue(C.byref(self.plugin.params), C.byref(self.q), int(batch), ptrs,
                                                                  _ptr(out), _ptr(idx) if idx is not None else None, _ptr(self.ws),
                                                                  self.ws_bytes, C.byref(gather), _stream(stream)),
                    "trtx_yolo_decode_nms_gather_enqueue")
            return out[:batch], (idx[:batch] if idx is not None else None)
        L.check(self._lib.trtx_yolo_decode_nms_enqueue(C.byref(self.plugin.params), C.byref(self.q), int(batch), ptrs,
                                                       _ptr(out), _ptr(idx) if idx is not None else None,
                                                       _ptr(self.ws), self.ws_bytes, _stream(stream)),
                "trtx_yolo_decode_nms_enqueue")
        return out[:batch], (idx[:batch] if idx is not None else None)

    def enqueue_scan(self, batch: int, inputs, stream=None) -> None:
        """Split form, first half: the HBM-bound scan kernel only."""
        ptrs = L.ptr_array([_ptr(t) for t in inputs])
        L.check(self._lib.trtx_yolo_scan_enqueue(C.byref(self.plugin.params), int(batch), ptrs, _ptr(self.ws),
                                                 self.ws_bytes, _stream(stream)), "trtx_yolo_scan_enqueue")

    def enqueue_nms(self, batch: int, inputs, stream=None, out=None):
        """Split form, second half: NMS over the tiles left by enqueue_scan (out: another [max_batch, 1 + max_det*7] buffer,
        e.g. the second of a double buffer whose first half is still being gathered)."""
        ptrs = L.ptr_array([_ptr(t) for t in inputs])
        out = self.out if out is None else out
        L.check(self._lib.trtx_yolo_nms_after_scan_enqueue(C.byref(self.plugin.params), C.byref(self.q), int(batch), ptrs,
                                                           _ptr(out), _ptr(self.idx) if self.idx is not None else None,
                                                           _ptr(self.ws), self.ws_bytes, _stream(stream)),
                "trtx_yolo_nms_after_scan_enqueue")
        return out[:batch], (self.idx[:batch] if self.idx is not None else None)


# --------------------------------------------------------------------------------------------------
# Decode_TRT (RetinaFace)
# --------------------------------------------------------------------------------------------------
class DecodePlugin:
    PLUGIN_TYPE = "Decode_TRT"
    PLUGIN_VERSION = "1"

    def __init__(self, input_h: int = 480, input_w: int = 640, anticov: bool = False):
        """anticov=True: the Decode_TRT of retinafaceAntiCov/decode.cu (38-channel inputs, 16-float rows, 640x640 there)."""
        self._lib = L.load()
        p = L.RetinaParams()
        p.in_h, p.in_w = int(input_h), int(input_w)
        p.gate = float_le_threshold(0.02)  # `conf2 <= 0.02` with a double literal (decode.cu:131)
        p.variant = L.RETINA_ANTICOV if anticov else L.RETINA_FACE
        self.params = p
        self.det_floats = 16 if anticov else 15
        self.total_priors = int(self._lib.trtx_retina_total_priors(C.byref(p)))

    def getNbOutputs(self) -> int:
        return 1

    def output_elems(self) -> int:
        return 1 + self.total_priors * self.det_floats

    def getOutputDimensions(self, index=0, inputs=None, nbInputDims=0):
        return (self.output_elems(), 1, 1)  # decode.cu:33-41

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return int(self._lib.trtx_retina_workspace_size(C.byref(self.params), int(maxBatchSize)))

    def enqueue(self, batchSize: int, inputs, outputs, workspace, stream=None) -> int:
        ptrs = L.ptr_array([_ptr(t) for t in inputs])
        return int(self._lib.trtx_retina_decode_enqueue(C.byref(self.params), int(batchSize), ptrs, _ptr(outputs[0]),
                                                        _ptr(workspace), workspace.numel() * workspace.element_size(),
                                                        _stream(stream)))

    def getPluginType(self) -> str:
        return self.PLUGIN_TYPE

    def getPluginVersion(self) -> str:
        return self.PLUGIN_VERSION

    def clone(self) -> "DecodePlugin":
        return DecodePlugin(self.params.in_h, self.params.in_w, self.params.variant == L.RETINA_ANTICOV)

    def serialize(self) -> bytes:  # the reference serializes nothing (decode.cu:23-31); the runtime size is new state
        return struct.pack("<ii", self.params.in_h, self.params.in_w)

    @classmethod
    def deserialize(cls, data: bytes) -> "DecodePlugin":
        if len(data) == 0:
            return cls()
        h, w = struct.unpack("<ii", data)
        return cls(h, w)


# --------------------------------------------------------------------------------------------------
# Faster R-CNN plugins (rcnn/*Plugin.h): "null workspace returns the size" idiom kept
# --------------------------------------------------------------------------------------------------
def _rc64(rc: int, what: str) -> int:
    if rc < 0:
        L.check(-rc, what)
    return rc


class RpnDecodePlugin:
    def __init__(self, top_n: int, anchors: Sequence[float], stride: float, image_height: int, image_width: int,
                 height: int = 0, width: int = 0):
        self._lib = L.load()
        self._top_n, self._anchors, self._stride = int(top_n), [float(a) for a in anchors], float(stride)
        self._image_height, self._image_width = int(image_height), int(image_width)
        self._height, self._width = int(height), int(width)
        self._anc = (C.c_float * len(self._anchors))(*self._anchors)

    def configurePlugin(self, inputDims):  # RpnDecodePlugin.h:148-157: height/width from the scores tensor dims
        self._height, self._width = int(inputDims[0][1]), int(inputDims[0][2])

    def getNbOutputs(self) -> int:
        return 2

    def getOutputDimensions(self, index):
        return (self._top_n, 4 if index == 1 else 1)

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return _rc64(self._lib.trtx_rpn_decode(maxBatchSize, None, None, None, None, self._height, self._width,
                                               self._image_height, self._image_width, self._stride, self._anc,
                                               len(self._anchors) // 4, self._top_n, None, 0, None), "trtx_rpn_decode(size)")

    def enqueue(self, batchSize, inputs, outputs, workspace, stream=None) -> int:
        rc = self._lib.trtx_rpn_decode(batchSize, _ptr(inputs[0]), _ptr(inputs[1]), _ptr(outputs[0]), _ptr(outputs[1]),
                                       self._height, self._width, self._image_height, self._image_width, self._stride,
                                       self._anc, len(self._anchors) // 4, self._top_n, _ptr(workspace),
                                       workspace.numel() * workspace.element_size(), _stream(stream))
        return int(-rc if rc < 0 else 0)


class RpnNmsPlugin:
    def __init__(self, nms_thresh: float, post_nms_topk: int, pre_nms_topk: int = 1):
        self._lib = L.load()
        self._nms_thresh, self._post_nms_topk, self._pre_nms_topk = float(nms_thresh), int(post_nms_topk), int(pre_nms_topk)

    def configurePlugin(self, inputDims):
        self._pre_nms_topk = int(inputDims[0][0])

    def getNbOutputs(self) -> int:
        return 1

    def getOutputDimensions(self, index=0):
        return (self._post_nms_topk, 4)

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return _rc64(self._lib.trtx_rpn_nms(maxBatchSize, None, None, None, self._pre_nms_topk, self._post_nms_topk,
                                            self._nms_thresh, None, 0, None), "trtx_rpn_nms(size)")

    def enqueue(self, batchSize, inputs, outputs, workspace, stream=None) -> int:
        rc = self._lib.trtx_rpn_nms(batchSize, _ptr(inputs[0]), _ptr(inputs[1]), _ptr(outputs[0]), self._pre_nms_topk,
                                    self._post_nms_topk, self._nms_thresh, _ptr(workspace),
                                    workspace.numel() * workspace.element_size(), _stream(stream))
        return int(-rc if rc < 0 else 0)


class PredictorDecodePlugin:
    def __init__(self, num_boxes: int, image_height: int, image_width: int, bbox_reg_weights: Sequence[float],
                 num_classes: int = 0):
        self._lib = L.load()
        self._num_boxes, self._num_classes = int(num_boxes), int(num_classes)
        self._image_height, self._image_width = int(image_height), int(image_width)
        self._w = (C.c_float * 4)(*[float(x) for x in bbox_reg_weights])

    def configurePlugin(self, inputDims):
        self._num_classes = int(inputDims[0][1])

    def getNbOutputs(self) -> int:
        return 3

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return _rc64(self._lib.trtx_predictor_decode(maxBatchSize, None, None, None, None, None, None, self._num_boxes,
                                                     self._num_classes, self._image_height, self._image_width, self._w,
                                                     None, 0, None), "trtx_predictor_decode(size)")

    def enqueue(self, batchSize, inputs, outputs, workspace, stream=None) -> int:
        rc = self._lib.trtx_predictor_decode(batchSize, _ptr(inputs[0]), _ptr(inputs[1]), _ptr(inputs[2]),
                                             _ptr(outputs[0]), _ptr(outputs[1]), _ptr(outputs[2]), self._num_boxes,
                                             self._num_classes, self._image_height, self._image_width, self._w,
                                             _ptr(workspace), workspace.numel() * workspace.element_size(), _stream(stream))
        return int(-rc if rc < 0 else 0)


class BatchedNmsPlugin:
    def __init__(self, nms_method: int, nms_thresh: float, detections_per_im: int, count: int = 1):
        self._lib = L.load()
        self._nms_method, self._nms_thresh = int(nms_method), float(nms_thresh)
        self._detections_per_im, self._count = int(detections_per_im), int(count)

    def configurePlugin(self, inputDims):
        self._count = int(inputDims[0][0])

    def getNbOutputs(self) -> int:
        return 3

    def getOutputDimensions(self, index):
        return (self._detections_per_im, 4 if index == 1 else 1)

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return _rc64(self._lib.trtx_batched_nms(self._nms_method, maxBatchSize, None, None, None, None, None, None,
                                                self._count, self._detections_per_im, self._nms_thresh, None, 0, None),
                     "trtx_batched_nms(size)")

    def enqueue(self, batchSize, inputs, outputs, workspace, stream=None) -> int:
        rc = self._lib.trtx_batched_nms(self._nms_method, batchSize, _ptr(inputs[0]), _ptr(inputs[1]), _ptr(inputs[2]),
                                        _ptr(outputs[0]), _ptr(outputs[1]), _ptr(outputs[2]), self._count,
                                        self._detections_per_im, self._nms_thresh, _ptr(workspace),
                                        workspace.numel() * workspace.element_size(), _stream(stream))
        return int(-rc if rc < 0 else 0)


# --------------------------------------------------------------------------------------------------
# Pre-process (preprocess.h)
# --------------------------------------------------------------------------------------------------
class Int8CalibratorBatcher:
    """The host pre-process of Int8EntropyCalibrator2::getBatch (yolov8/src/calibrator.cpp:33-52): every image goes through
    preprocess_img (letterbox, cv::resize INTER_LINEAR) and cv::dnn::blobFromImages(1 / 255.0, swapRB); `get_batch(images)` returns
    the [B, 3, input_h, input_w] fp32 batch the calibrator copies to the device.  HOST code (trtx_calib_letterbox_host), as in the
    reference; bit-identical to OpenCV 4.13 (tests/test_calibrator_cpu.py)."""

    def __init__(self, batchsize: int, input_w: int, input_h: int):
        self._lib = L.load()
        self.batchsize, self.input_w, self.input_h = int(batchsize), int(input_w), int(input_h)
        self.input_count = 3 * self.input_w * self.input_h * self.batchsize     # calibrator.cpp:20

    def getBatchSize(self) -> int:
        return self.batchsize

    def get_batch(self, images) -> "np.ndarray":
        import numpy as np

        if len(images) != self.batchsize:
            raise L.TrtxError(f"Int8CalibratorBatcher: {len(images)} images for a batch of {self.batchsize}")
        out = np.empty((self.batchsize, 3, self.input_h, self.input_w), np.float32)
        for i, img in enumerate(images):
            img = np.ascontiguousarray(img, np.uint8)
            h, w = img.shape[:2]
            L.check(self._lib.trtx_calib_letterbox_host(img.ctypes.data_as(C.c_void_p), w, h, img.strides[0], self.input_w, self.input_h,
                                                        out[i].ctypes.data_as(C.c_void_p)), "trtx_calib_letterbox_host")
        return out


class RoiAlignPlugin:
    """rcnn/RoiAlignPlugin.h:27-170 (plugin "RoiAlign"): inputs proposals [B,N,4], features [B,C,H,W] ->
    [B, N, C, P, P].  No workspace, no device synchronisation (the reference syncs after every image)."""

    def __init__(self, pooler_resolution: int, spatial_scale: float, sampling_ratio: int, num_proposals: int,
                 out_channels: int, feature_h: int = 0, feature_w: int = 0):
        self._lib = L.load()
        self._pooler_resolution, self._spatial_scale = int(pooler_resolution), float(spatial_scale)
        self._sampling_ratio, self._num_proposals, self._out_channels = int(sampling_ratio), int(num_proposals), int(out_channels)
        self._feature_h, self._feature_w = int(feature_h), int(feature_w)

    def configurePlugin(self, inputDims):  # RoiAlignPlugin.h:140-153
        self._feature_h, self._feature_w = int(inputDims[1][1]), int(inputDims[1][2])

    def getNbOutputs(self) -> int:
        return 1

    def getOutputDimensions(self, index=0):
        return (self._num_proposals, self._out_channels, self._pooler_resolution, self._pooler_resolution)

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return 0

    def enqueue(self, batchSize, inputs, outputs, workspace=None, stream=None, mode: int | None = None) -> int:
        """mode: None = trtx_roi_align (the window kernel); L.ROI_WINDOW / L.ROI_DIRECT pick the kernel (trtx_roi_align_ex)."""
        if mode is None:
            return int(self._lib.trtx_roi_align(batchSize, _ptr(inputs[0]), _ptr(inputs[1]), _ptr(outputs[0]), self._pooler_resolution,
                                                self._spatial_scale, self._sampling_ratio, self._num_proposals, self._out_channels,
                                                self._feature_h, self._feature_w, _stream(stream)))
        return int(self._lib.trtx_roi_align_ex(batchSize, _ptr(inputs[0]), _ptr(inputs[1]), _ptr(outputs[0]), self._pooler_resolution,
                                               self._spatial_scale, self._sampling_ratio, self._num_proposals, self._out_channels,
                                               self._feature_h, self._feature_w, int(mode), _stream(stream)))


class MaskRcnnInferencePlugin:
    """rcnn/MaskRcnnInferencePlugin.h:27-140 (plugin "MaskRcnnInference"): indices [B,D] (float class ids),
    masks [B,D,num_classes,S,S] -> [B,D,1,S,S] = sigmoid of the predicted class' mask."""

    def __init__(self, detections_per_im: int, output_size: int, num_classes: int = 1):
        self._lib = L.load()
        self._detections_per_im, self._output_size, self._num_classes = int(detections_per_im), int(output_size), int(num_classes)

    def configurePlugin(self, inputDims):  # MaskRcnnInferencePlugin.h:109-120
        self._num_classes = int(inputDims[1][1])

    def getNbOutputs(self) -> int:
        return 1

    def getOutputDimensions(self, index=0):
        return (self._detections_per_im, 1, self._output_size, self._output_size)

    def getWorkspaceSize(self, maxBatchSize: int) -> int:
        return 0

    def enqueue(self, batchSize, inputs, outputs, workspace=None, stream=None) -> int:
        return int(self._lib.trtx_mask_rcnn_inference(batchSize, _ptr(inputs[0]), _ptr(inputs[1]), _ptr(outputs[0]),
                                                      self._detections_per_im, self._output_size, self._num_classes,
                                                      _stream(stream)))


def cuda_batch_preprocess(img_batch: Sequence[torch.Tensor], dst: torch.Tensor, dst_width: int, dst_height: int,
                          stream=None) -> None:
    """Drop-in for cuda_batch_preprocess (yolov8/src/preprocess.cu:119-127) with DEVICE images:
    img_batch[i] is a u8 HWC BGR cuda tensor [h, w, 3] (row-contiguous); dst is [B, 3, dst_h, dst_w] fp32/fp16.
    One launch for the whole batch, no synchronisation."""
    lib = L.load()
    n = len(img_batch)
    descs = (L.ImageDesc * n)()
    for i, im in enumerate(img_batch):
        if im.dtype != torch.uint8 or im.dim() != 3 or im.shape[2] != 3 or im.stride(2) != 1 or im.stride(1) != 3:
            raise L.TrtxError("images must be u8 HWC BGR with packed pixels")
        descs[i].data_dev = im.data_ptr()
        descs[i].height, descs[i].width = int(im.shape[0]), int(im.shape[1])
        descs[i].pitch = int(im.stride(0))
    dt = L.F32 if dst.dtype == torch.float32 else L.F16
    L.check(lib.trtx_preprocess_batch_enqueue(descs, n, _ptr(dst), dst_width, dst_height, dt, _stream(stream)),
            "trtx_preprocess_batch_enqueue")


class PreprocessPlan:
    """cuda_batch_preprocess with the descriptors prepared once for persistent device frame buffers
    (the reference rebuilds nothing either: its staging buffers are allocated in cuda_preprocess_init,
    preprocess.cu:129-134).  enqueue() is a single C call -> a single kernel launch."""

    def __init__(self, img_batch: Sequence[torch.Tensor], dst: torch.Tensor, dst_width: int, dst_height: int):
        self._lib = L.load()
        self.n = len(img_batch)
        self.descs = (L.ImageDesc * self.n)()
        self._keep = list(img_batch)
        for i, im in enumerate(img_batch):
            if im.dtype != torch.uint8 or im.dim() != 3 or im.shape[2] != 3 or im.stride(2) != 1 or im.stride(1) != 3:
                raise L.TrtxError("images must be u8 HWC BGR with packed pixels")
            self.descs[i].data_dev = im.data_ptr()
            self.descs[i].height, self.descs[i].width = int(im.shape[0]), int(im.shape[1])
            self.descs[i].pitch = int(im.stride(0))
        self.dst, self.dw, self.dh = dst, int(dst_width), int(dst_height)
        self.dt = L.F32 if dst.dtype == torch.float32 else L.F16

    def enqueue(self, stream=None) -> None:
        L.check(self._lib.trtx_preprocess_batch_enqueue(self.descs, self.n, _ptr(self.dst), self.dw, self.dh, self.dt,
                                                        _stream(stream)), "trtx_preprocess_batch_enqueue")


def get_rect(img_w: int, img_h: int, bbox, net_w: int = 640, net_h: int = 640, variant: int = L.YOLO_V8):
    """get_rect(img, bbox) of yolov8/src/postprocess.cpp:6-36 (variant YOLO_V5: yolov5/src/postprocess.cpp:4-29):
    -> (x, y, width, height) in the original image."""
    lib = L.load()
    b = (C.c_float * 4)(*[float(v) for v in bbox])
    r = (C.c_int * 4)()
    L.check(lib.trtx_get_rect(variant, net_w, net_h, img_w, img_h, b, r), "trtx_get_rect")
    return tuple(r)


def get_rect_adapt_landmark(img_w: int, img_h: int, bbox, lmk, net_w: int = 640, net_h: int = 640):
    """get_rect_adapt_landmark(img, bbox, lmk) of yolov8/src/postprocess.cpp:38-69 -> ((x, y, w, h), mapped keypoints)."""
    lib = L.load()
    b = (C.c_float * 4)(*[float(v) for v in bbox])
    k = (C.c_float * len(lmk))(*[float(v) for v in lmk])
    r = (C.c_int * 4)()
    L.check(lib.trtx_get_rect_adapt_landmark(net_w, net_h, img_w, img_h, b, k, len(lmk) // 3, r), "trtx_get_rect_adapt_landmark")
    return tuple(r), list(k)


def scale_mask(masks: torch.Tensor, img_w: int, img_h: int, out=None, stream=None) -> torch.Tensor:
    """scale_mask(mask, img) of yolov8/src/postprocess.cpp:207-226 for a stack of device masks [n, net_h, net_w] fp32 ->
    [n, img_h, img_w]: the letterboxed region, bilinearly resized (cv::resize) to the original image."""
    lib = L.load()
    n, nh, nw = masks.shape
    if out is None:
        out = torch.empty((n, img_h, img_w), dtype=torch.float32, device=masks.device)
    L.check(lib.trtx_scale_mask_enqueue(_ptr(masks), n, nw, nh, img_w, img_h, _ptr(out), _stream(stream)), "trtx_scale_mask_enqueue")
    return out


def letterbox_matrix(src_w: int, src_h: int, dst_w: int, dst_h: int):
    m = (C.c_float * 6)()
    L.load().trtx_letterbox_matrix(src_w, src_h, dst_w, dst_h, m)
    return list(m)
