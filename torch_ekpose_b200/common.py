"""Result objects of the post-processing path.

Mirrors the output contract of /root/reference/lib/utils/common.py: ``Human`` (:51-63) with
``body_parts`` {part_idx: BodyPart} and ``score``; ``BodyPart`` (:277-298) with ``uidx``,
``part_idx``, normalised ``x``, ``y`` in [0, 1) and ``score``; the part enumeration (:6-25) and
limb table (:27-30).  Drawing (:252-275) is ``PostProcessor.draw_humans`` on the device (``ekp_draw_humans``); the
face / upper-body box heuristics of that file are host-side visualisation and out of scope (SURVEY.md section 8).
"""
from enum import Enum


class CocoPart(Enum):
    Nose = 0
    Neck = 1
    RShoulder = 2
    RElbow = 3
    RWrist = 4
    LShoulder = 5
    LElbow = 6
    LWrist = 7
    RHip = 8
    RKnee = 9
    RAnkle = 10
    LHip = 11
    LKnee = 12
    LAnkle = 13
    REye = 14
    LEye = 15
    REar = 16
    LEar = 17
    Background = 18


CocoPairs = [(1, 2), (1, 5), (2, 3), (3, 4), (5, 6), (6, 7), (1, 8), (8, 9), (9, 10), (1, 11),
             (11, 12), (12, 13), (1, 0), (0, 14), (14, 16), (0, 15), (15, 17), (2, 16), (5, 17)]
CocoPairsRender = CocoPairs[:-2]


class BodyPart:
    __slots__ = ("uidx", "part_idx", "x", "y", "score")

    def __init__(self, uidx, part_idx, x, y, score):
        self.uidx = uidx
        self.part_idx = part_idx
        self.x, self.y = x, y
        self.score = score

    def get_part_name(self):
        return CocoPart(self.part_idx)

    def __repr__(self):
        return "BodyPart:%d-(%.2f, %.2f) score=%.2f" % (self.part_idx, self.x, self.y, self.score)


class Human:
    __slots__ = ("body_parts", "pairs", "uidx_list", "score")

    def __init__(self, pairs=()):
        self.pairs = list(pairs)
        self.uidx_list = set()
        self.body_parts = {}
        self.score = 0.0

    def part_count(self):
        return len(self.body_parts)

    def get_max_score(self):
        return max(p.score for p in self.body_parts.values())

    def __repr__(self):
        return " ".join(repr(p) for p in self.body_parts.values())
