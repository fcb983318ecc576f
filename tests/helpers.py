"""shared test helpers (importable because pytest puts tests/ on sys.path)"""
import numpy as np

from deepfactors_b200 import synth


def box_blur25(gray):
    """cv2.blur(gray / 255, (25, 25)) bit for bit: the window sums of the fp32 pixels are exact in fp64 (every pixel is a
    multiple of 2**-32 below 1), then scaled by 1/625 and rounded to fp32 as OpenCV does; border = reflect-101."""
    f = np.pad((gray.astype(np.float32) * np.float32(1 / 255.0)).astype(np.float64), 12, mode="reflect")
    c = np.pad(f, ((1, 0), (1, 0))).cumsum(0).cumsum(1)
    s = c[25:, 25:] - c[:-25, 25:] - c[25:, :-25] + c[:-25, :-25]
    return (s * (1.0 / 625)).astype(np.float32)


def scenenet_inputs(golden):
    """inputs of tests/ut_se3aligner.cpp:58-77: 1047 -> 1052, /255, 25x25 box blur, depth mm -> m, SceneNet camera"""
    img0 = box_blur25(golden["gray_1047"])
    img1 = box_blur25(golden["gray_1052"])
    dpt0 = (golden["depth_1047_mm"].astype(np.float32) * np.float32(1 / 1000.0)).astype(np.float32)
    cam = synth.Camera.scenenet(img0.shape[1], img0.shape[0])
    return cam, img0, img1, dpt0


def tracking_pyramid(golden, oracle, levels=3):
    """keyframe 1047 / live frame 1052 as a `levels`-deep pyramid (level 0 = 320x240): images by the reference's
    GaussianBlurDown (cu_image_proc.cpp:134-184), gradients by its Sobel (:57-113), depth by 2x2 subsampling, cameras by
    CameraPyramid halving (camera_pyramid.h:41-46).  Built with the oracle so the CPU loop and the GPU see the same
    bytes."""
    cam, img0, img1, dpt0 = scenenet_inputs(golden)
    cams = synth.camera_pyramid(cam, levels)
    p0, p1, pd = [img0], [img1], [dpt0]
    for _ in range(1, levels):
        p0.append(oracle.gaussian_blur_down(p0[-1]))
        p1.append(oracle.gaussian_blur_down(p1[-1]))
        pd.append(np.ascontiguousarray(pd[-1][::2, ::2]))
    pg = [oracle.sobel_gradients(i) for i in p1]
    return cams, p0, p1, pd, pg
