"""numpy restatement of the dataset-side resampling on the hot path.

TEST INFRASTRUCTURE (see oracle/model_ref.py's header).

Follows libs/datasets/deepfake_video_audio.py:445-558
(DeepFakeVideoAudioDatasetInfer3.__getitem__): each `.npy` stream [T, C] is
transposed, resized to max_seq_len with
F.interpolate(mode='linear', align_corners=False) (:513-544) and the three
streams are concatenated video | BYOL-A | emotion2vec along C (:547).
The index math is ATen's (aten/src/ATen/native/UpSample.h,
area_pixel_compute_scale / area_pixel_compute_source_index; torch 1.11 pinned
by the reference, 2.11 here — same formula): all in fp32,
  scale = float(T_in) / float(T_out)
  src   = max(0, fma(scale, t + 0.5, -0.5));  i0 = int(src);  i1 = i0 + (i0 < T_in-1)
  l1 = src - i0;  l0 = 1 - l1
  out   = fma(l0, x[i0], l1 * x[i1])
The two fused multiply-adds are what ATen's AVX2/AVX-512 CPU kernels execute
(the compiler contracts those expressions); with them this restatement is
BIT-EXACT against F.interpolate on this image (checked in
tests/test_oracle_golden.py), without them it is only within ~1e-4.
fma(a, b, c) for fp32 operands is emulated as fp32(fp64(a) * fp64(b) + fp64(c)):
the product is exact in fp64.
"""
import numpy as np

f32 = np.float32


def linear_resize_tc(x_tc: np.ndarray, t_out: int, out_dtype=f32) -> np.ndarray:
    """[T_in, C] -> [t_out, C] (time-major in and out). out_dtype=np.float64: the same fp32 index / weight math, the
    blend l0 * x[i0] + l1 * x[i1] exact in float64 (no fp32 rounding of the product or the sum)."""
    t_in = x_tc.shape[0]
    if t_in == t_out:
        return x_tc.astype(out_dtype, copy=True)
    scale = f32(t_in) / f32(t_out)
    t = np.arange(t_out, dtype=f32)
    src = (np.float64(scale) * np.float64(t + f32(0.5)) - 0.5).astype(f32)
    src = np.where(src < 0, f32(0), src).astype(f32)
    i0 = src.astype(np.int64)
    i1 = i0 + (i0 < t_in - 1)
    l1 = (src - i0.astype(f32)).astype(f32)
    l0 = (f32(1.0) - l1).astype(f32)
    if out_dtype == np.float64:
        x64 = x_tc.astype(np.float64)
        return np.float64(l0[:, None]) * x64[i0] + np.float64(l1[:, None]) * x64[i1]
    b =(l1[:, None] * x_tc[i1]).astype(f32)
    return (np.float64(l0[:, None]) * np.float64(x_tc[i0]) + np.float64(b)).astype(f32)


def dataset_item(streams: dict, duration: float, video_id: str, max_seq_len: int = 768,
                 feat_stride: int = 1, num_frames: int = 1) -> dict:
    """The dict `__getitem__` returns (:551-556), from raw streams
    {'video' [T_v,256] (optional), 'byola' [T_b,2048], 'emo' [T_e,768]} that are
    already truncated (:482-483). feats is [C, T] like the reference's."""
    import torch
    parts = []
    first = streams["video"] if "video" in streams else streams["byola"]
    fps = first.shape[0] / duration                                   # :461
    fs = float((first.shape[0] - 1) * feat_stride + num_frames) / max_seq_len   # :495-497
    for k in ("video", "byola", "emo"):
        if k in streams:
            parts.append(linear_resize_tc(streams[k], max_seq_len))
    feats = np.concatenate(parts, axis=1).T                            # [C, T]
    return {"video_id": video_id, "feats": torch.from_numpy(np.ascontiguousarray(feats)),
            "fps": fps, "duration": duration, "feat_stride": fs, "feat_num_frames": fs}
