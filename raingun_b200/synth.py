"""Synthetic scenes of BASELINE.json's configs[2..4], emitted in the reference's YAML schema.

The generator is the definition of the scenes (SURVEY.md section 8d): SplitMix64 stream,
``u01 = (z >> 11) * 2**-53``, ``U(a, b) = round(a + (b - a) * u01, 6)``; per sphere the draw
order is x, y, z, radius, colour (``next_u64 & 0xFFFFFF``), albedo, selector, surface
parameters, then (textured spheres only) x_offset.  The ground plane is body 0.  Extents
stay below ~60 units so the reference's SHADOW_BIAS = 1e-13 (lib.rs:11) keeps its meaning.

The document produced is what ``serde_yaml`` would deserialize into raingun-lib's ``Scene``
(scene.rs:11-19); ``to_yaml`` writes it out for the reference CLI.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Tuple

MASK64 = (1 << 64) - 1

CLAY = "./textures/clay-ground-seamless.jpg"
EARTH = "./textures/land_ocean_ice_cloud_2048.jpg"


class SplitMix64:
    def __init__(self, seed: int) -> None:
        self.x = seed & MASK64

    def next_u64(self) -> int:
        self.x = (self.x + 0x9E3779B97F4A7C15) & MASK64
        z = self.x
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK64
        return z ^ (z >> 31)

    def u01(self) -> float:
        return (self.next_u64() >> 11) * (2.0 ** -53)

    def uniform(self, a: float, b: float) -> float:
        return round(a + (b - a) * self.u01(), 6)


@dataclass(frozen=True)
class SynthSpec:
    name: str
    width: int
    height: int
    seed: int
    spheres: int
    box_x: float
    box_y: Tuple[float, float]
    box_z: Tuple[float, float]
    radius: Tuple[float, float]
    mixed: bool          # reflecting / refractive / diffuse mix (else all diffuse)
    textured: bool       # clay ground + every 4th sphere earth-textured
    lights: int          # 3 or 4
    depth: int


SPECS: Dict[str, SynthSpec] = {
    # configs[2]: 3840x2160, 1,000 diffuse spheres + ground plane, 3 lights, depth 4
    "C3": SynthSpec("C3", 3840, 2160, 1001, 1000, 16.0, (-1.5, 12.0), (-30.0, -4.0), (0.12, 0.5),
                    False, False, 3, 4),
    # configs[3]: 3840x2160, 10,000 mixed reflective/refractive spheres, depth 8
    "C4": SynthSpec("C4", 3840, 2160, 1002, 10000, 24.0, (-1.5, 18.0), (-45.0, -4.0), (0.08, 0.35),
                    True, False, 3, 8),
    # configs[4]: 7680x4320 textured, 100,000 spheres, 4 spherical lights, depth 8
    "C5": SynthSpec("C5", 7680, 4320, 1003, 100000, 32.0, (-1.5, 24.0), (-60.0, -4.0), (0.04, 0.16),
                    True, True, 4, 8),
}


def _lights(spec: SynthSpec) -> List[Dict[str, Any]]:
    sph_a = {"Spherical": {"position": [-6.0, 14.0, -5.0], "color": "#ee0077", "intensity": 8000.0}}
    sph_b = {"Spherical": {"position": [14.0, 16.0, -12.0], "color": "#ffffee", "intensity": 9000.0}}
    if spec.lights == 3:
        return [{"Directional": {"direction": {"x": 0.4, "y": -1.0, "z": -0.9}, "color": "#ffffee",
                                 "intensity": 7.0}}, sph_a, sph_b]
    return [sph_a, sph_b,
            {"Spherical": {"position": [-20.0, 20.0, -40.0], "color": "#c8ffc8", "intensity": 12000.0}},
            {"Spherical": {"position": [20.0, 10.0, -55.0], "color": "#ffffff", "intensity": 12000.0}}]


def make_scene_doc(spec: SynthSpec, spheres: Optional[int] = None, depth: Optional[int] = None
                   ) -> Dict[str, Any]:
    """The YAML document (as Python data) of a synthetic scene.  ``spheres`` / ``depth``
    shrink the scene for parity tests; the stream is the same, just cut short."""
    n = spec.spheres if spheres is None else int(spheres)
    rng = SplitMix64(spec.seed)
    ground_col: Dict[str, Any] = {"Color": "#808080"}
    if spec.textured:
        ground_col = {"Texture": {"image": CLAY, "x_offset": 0.0, "y_offset": 0.0}}
    bodies: List[Dict[str, Any]] = [{"Plane": {
        "origin": [0.0, -2.0, -5.0], "normal": [0.0, -1.0, 0.0],
        "material": {"coloration": ground_col, "albedo": 0.3, "surface": "Diffuse"}}}]
    for i in range(n):
        x = rng.uniform(-spec.box_x, spec.box_x)
        y = rng.uniform(*spec.box_y)
        z = rng.uniform(*spec.box_z)
        r = rng.uniform(*spec.radius)
        colour = "#%06x" % (rng.next_u64() & 0xFFFFFF)
        albedo = rng.uniform(0.2, 0.9)
        s = rng.uniform(0.0, 1.0)
        surface: Any = "Diffuse"
        if spec.mixed:
            if s < 0.4:
                surface = {"Reflecting": {"reflectivity": rng.uniform(0.2, 0.9)}}
            elif s < 0.8:
                index = rng.uniform(1.1, 1.8)
                surface = {"Refractive": {"index": index, "transparency": rng.uniform(0.7, 1.0)}}
        coloration: Dict[str, Any] = {"Color": colour}
        if spec.textured and i % 4 == 0:
            coloration = {"Texture": {"image": EARTH, "x_offset": rng.uniform(0.0, 1.0), "y_offset": 0.0}}
        bodies.append({"Sphere": {"center": [x, y, z], "radius": r,
                                  "material": {"coloration": coloration, "albedo": albedo,
                                               "surface": surface}}})
    return {"fov": 90.0, "defaultColor": "#667fff",
            "maxRecursionDepth": spec.depth if depth is None else int(depth),
            "lights": _lights(spec), "bodies": bodies}


def to_yaml(doc: Dict[str, Any]) -> str:
    import yaml

    return "---\n" + yaml.safe_dump(doc, sort_keys=False, default_flow_style=None)


def make_scene(name: str, spheres: Optional[int] = None, depth: Optional[int] = None,
               texture_loader=None):
    """SceneData of a named synthetic config (``C3`` / ``C4`` / ``C5``)."""
    from .scene import default_texture_loader, scene_from_dict

    spec = SPECS[name]
    doc = make_scene_doc(spec, spheres, depth)
    return scene_from_dict(doc, texture_loader or default_texture_loader), spec


# B4: the box-and-disk counterpart of C4, kept out of SPECS (the benchmark's configs).  Same volume, lights
# and depth as C4 / C3; `spheres` counts its bodies and `radius` is the range of a box's half-extents.
B4 = SynthSpec("B4", 3840, 2160, 1004, 10000, 24.0, (-1.5, 18.0), (-45.0, -4.0), (0.06, 0.3),
               True, False, 3, 8)
B4_DISK_RADIUS = (0.08, 0.35)


def make_box_scene_doc(bodies: Optional[int] = None, depth: Optional[int] = None) -> Dict[str, Any]:
    """The YAML document of B4: 3840x2160, depth 8, C3's three lights, a ground plane (body 0) and
    10,000 boxes and disks in C4's volume.  SplitMix64 seed 1004, ``U`` as for C3-C5; per body the
    draw order is x, y, z, a kind selector, then for a selector below 0.7 an AABB with half-extents
    U(0.06, 0.3) drawn for x, y, z (bounds rounded to 6 decimals), else a Disk with radius
    U(0.08, 0.35) and normal components U(-1, 1) drawn for x, y, z; then colour, albedo, surface
    selector and surface parameters exactly as C4 draws them.  ``bodies`` / ``depth`` shrink the
    scene for parity tests; the stream is the same, just cut short."""
    spec = B4
    n = spec.spheres if bodies is None else int(bodies)
    rng = SplitMix64(spec.seed)
    out: List[Dict[str, Any]] = [{"Plane": {
        "origin": [0.0, -2.0, -5.0], "normal": [0.0, -1.0, 0.0],
        "material": {"coloration": {"Color": "#808080"}, "albedo": 0.3, "surface": "Diffuse"}}}]
    for _ in range(n):
        x = rng.uniform(-spec.box_x, spec.box_x)
        y = rng.uniform(*spec.box_y)
        z = rng.uniform(*spec.box_z)
        if rng.uniform(0.0, 1.0) < 0.7:
            hx, hy, hz = (rng.uniform(*spec.radius) for _ in range(3))
            lo = [round(x - hx, 6), round(y - hy, 6), round(z - hz, 6)]
            hi = [round(x + hx, 6), round(y + hy, 6), round(z + hz, 6)]
            kind, geom = "AABB", {"bounds": [lo, hi]}
        else:
            r = rng.uniform(*B4_DISK_RADIUS)
            normal = [rng.uniform(-1.0, 1.0) for _ in range(3)]
            kind, geom = "Disk", {"origin": [x, y, z], "normal": normal, "radius": r}
        colour = "#%06x" % (rng.next_u64() & 0xFFFFFF)
        albedo = rng.uniform(0.2, 0.9)
        s = rng.uniform(0.0, 1.0)
        surface: Any = "Diffuse"
        if s < 0.4:
            surface = {"Reflecting": {"reflectivity": rng.uniform(0.2, 0.9)}}
        elif s < 0.8:
            index = rng.uniform(1.1, 1.8)
            surface = {"Refractive": {"index": index, "transparency": rng.uniform(0.7, 1.0)}}
        geom["material"] = {"coloration": {"Color": colour}, "albedo": albedo, "surface": surface}
        out.append({kind: geom})
    return {"fov": 90.0, "defaultColor": "#667fff",
            "maxRecursionDepth": spec.depth if depth is None else int(depth),
            "lights": _lights(spec), "bodies": out}


def make_box_scene(name: str = "B4", bodies: Optional[int] = None, depth: Optional[int] = None,
                   texture_loader=None):
    """SceneData of the box-and-disk scene ``B4`` (see make_box_scene_doc) and its spec."""
    from .scene import default_texture_loader, scene_from_dict

    if name != "B4":
        raise KeyError(name)
    doc = make_box_scene_doc(bodies, depth)
    return scene_from_dict(doc, texture_loader or default_texture_loader), B4
