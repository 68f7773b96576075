"""The checker of ekp_draw_humans: the reference's draw_humans (lib/utils/common.py:252-275) restated with cv2, and the
list[Human] it draws built from host human tables exactly as PostProcessor.humans() builds them."""
import cv2
import numpy as np

from torch_ekpose_b200.common import BodyPart, CocoPairsRender, CocoPart, Human

# lib/utils/common.py CocoColors
CocoColors = [[255, 0, 0], [255, 85, 0], [255, 170, 0], [255, 255, 0], [170, 255, 0], [85, 255, 0], [0, 255, 0],
              [0, 255, 85], [0, 255, 170], [0, 255, 255], [0, 170, 255], [0, 85, 255], [0, 0, 255], [85, 0, 255],
              [170, 0, 255], [255, 0, 255], [255, 0, 170], [255, 0, 85]]

PEAK_DT = np.dtype([("x", np.int32), ("y", np.int32), ("score", np.float32), ("id", np.int32)])


def draw_humans(npimg, humans, imgcopy=False):
    if imgcopy:
        npimg = np.copy(npimg)
    image_h, image_w = npimg.shape[:2]
    centers = {}
    for human in humans:
        for i in range(CocoPart.Background.value):
            if i not in human.body_parts.keys():
                continue
            body_part = human.body_parts[i]
            center = (int(body_part.x * image_w + 0.5), int(body_part.y * image_h + 0.5))
            centers[i] = center
            cv2.circle(npimg, center, 3, CocoColors[i], thickness=3, lineType=8, shift=0)
        for pair_order, pair in enumerate(CocoPairsRender):
            if pair[0] not in human.body_parts.keys() or pair[1] not in human.body_parts.keys():
                continue
            cv2.line(npimg, centers[pair[0]], centers[pair[1]], CocoColors[pair_order], 3)
    return npimg


def humans_of(num, parts, map_h, map_w):
    """Per image the list[Human] of a human table (num [n], parts [n, max_humans, 18] PEAK_DT), as
    PostProcessor.humans() builds it for a map of map_h x map_w."""
    out = []
    for i in range(len(num)):
        humans = []
        for k in range(int(num[i])):
            human = Human([])
            row = parts[i, k]
            for part_idx in np.nonzero(row["id"] >= 0)[0]:
                p = row[part_idx]
                human.body_parts[int(part_idx)] = BodyPart("%d-%d" % (k, part_idx), int(part_idx),
                                                           float(p["x"]) / map_w, float(p["y"]) / map_h, float(p["score"]))
            if human.body_parts:
                humans.append(human)
        out.append(humans)
    return out


def draw_batch(frames, humans_per_image, draw=draw_humans):
    """A drawn copy of host frames [n, H, W, 3]."""
    out = np.array(frames, copy=True)
    for i, humans in enumerate(humans_per_image):
        draw(out[i], humans)
    return out
