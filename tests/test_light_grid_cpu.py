"""Light grids (raingun_b200/csrc/rg_light_grid.h), the CPU side: the binning and the ray key are __host__ __device__,
so compile them with g++ and check the property the tracer relies on.  For shadow rays built exactly as k_shade builds
them (o = hp + n * 1e-13, d = light_direction_from, tmax = light_distance), every sphere whose FP64 test (the
reference's, bodies.rs:92-99) returns t <= tmax must be in the list of the ray's key cell or on the light's always
list, unless the key sends the ray back to the 3-D walk.  CPU-only."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from raingun_b200.synth import SPECS, make_scene_doc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HARNESS = r'''
#include <cstdio>
#include <cstdlib>
#include <random>
#include <set>
#include <vector>
#include "rg_light_grid.h"
using namespace rg;

// bodies.rs:92-99 as rg_exact.cuh::sphere_intersect (compiled with -ffp-contract=off)
static bool sphere_intersect(const double *c, const double *o, const double *d, double &t) {
    const double h[3] = {c[0] - o[0], c[1] - o[1], c[2] - o[2]};
    const double adj = (h[0] * d[0] + h[1] * d[1]) + h[2] * d[2];
    const double opp2 = ((h[0] * h[0] + h[1] * h[1]) + h[2] * h[2]) - adj * adj;
    const double r2 = c[3] * c[3];
    if (opp2 > r2) return false;
    const double th = std::sqrt(r2 - opp2), d0 = adj - th, d1 = adj + th;
    const bool n0 = d0 < 0.0, n1 = d1 < 0.0;
    t = n0 ? d1 : (n1 ? d0 : std::fmin(d0, d1));
    return !(n0 && n1);
}
static void normalize(double *v) {
    const double inv = 1.0 / std::sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]);
    for (int k = 0; k < 3; ++k) v[k] = v[k] * inv;
}

int main(int argc, char **argv) {
    FILE *f = std::fopen(argv[1], "rb");
    uint32_t n, nl, rays;
    if (std::fread(&n, 4, 1, f) != 1 || std::fread(&nl, 4, 1, f) != 1 || std::fread(&rays, 4, 1, f) != 1) return 2;
    std::vector<double> sph(4 * (size_t)n), lights(4 * (size_t)nl);   // light: kind, v (directional: normalised -direction)
    if (std::fread(sph.data(), 8, sph.size(), f) != sph.size() || std::fread(lights.data(), 8, lights.size(), f) != lights.size()) return 2;
    std::fclose(f);
    double scale = 1.0;
    for (uint32_t i = 0; i < n; ++i) {
        const double *c = &sph[4 * (size_t)i];
        const double m = std::max(std::max(std::fabs(c[0]), std::fabs(c[1])), std::fabs(c[2])) + std::fabs(c[3]);
        if (m < 1e6) scale = std::max(scale, 1.0 + m);
    }
    std::mt19937_64 rng(11);
    std::normal_distribution<double> gauss;
    std::uniform_real_distribution<double> uni(0.0, 1.0);
    long long checked = 0, hits = 0, fallback = 0, listed_total = 0, keyed = 0;
    for (uint32_t l = 0; l < nl; ++l) {
        const uint32_t kind = (uint32_t)lights[4 * l];
        const double *v = &lights[4 * l + 1];
        double sl = scale;
        if (kind) sl = std::max(sl, 1.0 + std::max(std::max(std::fabs(v[0]), std::fabs(v[1])), std::fabs(v[2])));
        LightGridInfo g;
        if (!lg_setup(g, kind, v, sph.data(), n, sl, 2.0)) { std::printf("no grid for light %u\n", l); return 3; }
        g.base = 0;
        g.always = lg_key_cells(g);
        std::vector<std::set<uint32_t>> cells(g.always + 1);
        for (uint32_t i = 0; i < n; ++i) {
            int r[6][4];
            const int k = lg_item_ranges(g, &sph[4 * (size_t)i], sph[4 * (size_t)i + 3], r);
            if (k < 0) { cells[g.always].insert(i); continue; }
            for (int fc = 0; fc < 6; ++fc)
                for (int y = r[fc][2]; y <= r[fc][3]; ++y)
                    for (int x = r[fc][0]; x <= r[fc][1]; ++x) cells[lg_cell_index(g, fc, x, y)].insert(i);
        }
        for (uint32_t q = 0; q < rays; ++q) {
            // a hit point: on a random sphere's surface (normal = normalize(hp - c)), or on the ground plane y = -2
            double hp[3], nrm[3];
            if (q % 4 == 3) {
                hp[0] = (uni(rng) - 0.5) * 4.0 * scale; hp[1] = -2.0; hp[2] = -uni(rng) * 4.0 * scale;
                nrm[0] = 0.0; nrm[1] = 1.0; nrm[2] = 0.0;
            } else {
                const double *c = &sph[4 * (size_t)(rng() % n)];
                double e[3] = {gauss(rng), gauss(rng), gauss(rng)};
                normalize(e);
                for (int k = 0; k < 3; ++k) hp[k] = c[k] + e[k] * c[3];
                for (int k = 0; k < 3; ++k) nrm[k] = hp[k] - c[k];
                normalize(nrm);
            }
            double o[3], d[3], tmax;
            for (int k = 0; k < 3; ++k) o[k] = hp[k] + nrm[k] * 1e-13;
            if (kind == 0) {
                for (int k = 0; k < 3; ++k) d[k] = v[k];
                tmax = INFINITY;
            } else {
                for (int k = 0; k < 3; ++k) d[k] = v[k] - hp[k];
                normalize(d);
                const double w[3] = {v[0] - hp[0], v[1] - hp[1], v[2] - hp[2]};
                tmax = std::sqrt((w[0] * w[0] + w[1] * w[1]) + w[2] * w[2]);
            }
            double depth = 0.0;
            const long long key = lg_ray_key(g, o, d, tmax, depth);
            ++checked;
            if (key == -2) { ++fallback; continue; }
            if (key >= 0) { ++keyed; listed_total += (long long)cells[(size_t)key].size(); }
            const float dray = (float)depth;   // compared as the tracer does: FP32, record depth rounded down, ray up
            for (uint32_t i = 0; i < n; ++i) {
                double t;
                if (!sphere_intersect(&sph[4 * (size_t)i], o, d, t) || !(t <= tmax)) continue;
                ++hits;
                if (cells[g.always].count(i)) continue;
                const bool in_cell = key >= 0 && cells[(size_t)key].count(i);
                const float di = lg_float_down(lg_item_depth(g, &sph[4 * (size_t)i], sph[4 * (size_t)i + 3]));
                if (!in_cell || di > std::nextafter(dray, INFINITY)) {
                    std::printf("MISSED light %u ray %u item %u t %.17g tmax %.17g key %lld listed %d depth %g ray depth %g\n", l, q, i,
                                t, tmax, key, (int)in_cell, (double)di, depth);
                    return 1;
                }
            }
        }
        std::printf("light %u kind %u dim %d x %d always %zu\n", l, kind, g.dim[0], g.dim[1], cells[g.always].size());
    }
    std::printf("ok checked %lld hits %lld fallback %lld mean_list %.3f\n", checked, hits, fallback,
                keyed ? (double)listed_total / keyed : 0.0);
    return 0;
}
'''


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("lg")
    cpp = d / "lg_test.cpp"
    cpp.write_text(HARNESS)
    exe = d / "lg_test"
    r = subprocess.run([gxx, "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "raingun_b200", "csrc"),
                        str(cpp), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe, d


def _lights(doc):
    out = []
    for l in doc["lights"]:
        if "Directional" in l:
            v = l["Directional"]["direction"]
            n = -np.array([v["x"], v["y"], v["z"]], float)
            inv = 1.0 / np.sqrt((n[0] * n[0] + n[1] * n[1]) + n[2] * n[2])
            out.append((0.0, n[0] * inv, n[1] * inv, n[2] * inv))
        else:
            out.append((1.0, *map(float, l["Spherical"]["position"])))
    return out


def _run(harness, spheres, lights, rays=4000):
    exe, d = harness
    path = d / "scene.bin"
    sph = np.asarray(spheres, np.float64).reshape(-1, 4)
    with open(path, "wb") as f:
        f.write(np.array([len(sph), len(lights), rays], np.uint32).tobytes())
        f.write(sph.tobytes())
        f.write(np.asarray(lights, np.float64).reshape(-1, 4).tobytes())
    r = subprocess.run([str(exe), str(path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    last = r.stdout.strip().splitlines()[-1].split()
    stats = dict(zip(last[1::2], map(float, last[2::2])))
    assert stats["hits"] > 0
    assert stats["fallback"] <= 0.05 * stats["checked"], r.stdout   # the light grids serve nearly every ray
    return stats


def _synth(name, n):
    doc = make_scene_doc(SPECS[name], spheres=n)
    sph = [(*b["Sphere"]["center"], b["Sphere"]["radius"]) for b in doc["bodies"] if "Sphere" in b]
    return np.array(sph, float), _lights(doc)


@pytest.mark.parametrize("name,n", [("C4", 1500), ("C5", 3000), ("C3", 1000)])
def test_every_hit_is_listed_on_synthetic_scenes(harness, name, n):
    sph, lights = _synth(name, n)
    _run(harness, sph, lights)


def test_light_inside_and_on_spheres(harness):
    """A light at a sphere's centre and one exactly on another's surface: those spheres go on the always list."""
    sph, _ = _synth("C4", 800)
    c0, c1 = sph[0], sph[1]
    lights = [(1.0, c0[0], c0[1], c0[2]), (1.0, c1[0] + c1[3], c1[1], c1[2]), (1.0, c1[0], c1[1] + 0.5 * c1[3] + 1e-12, c1[2])]
    _run(harness, sph, lights)


def test_axis_parallel_directional_lights(harness):
    sph, _ = _synth("C4", 800)
    lights = [(0.0, 0.0, 1.0, 0.0), (0.0, 1.0, 0.0, 0.0), (0.0, 0.0, 0.0, -1.0)]
    _run(harness, sph, lights)


def test_coordinates_in_the_thousands(harness):
    sph, lights = _synth("C4", 1000)
    big = sph.copy()
    big[:, :3] = big[:, :3] * 150.0 + np.array([2500.0, 1000.0, -3000.0])
    big[:, 3] *= 150.0
    lights = [(0.0, *lights[0][1:]), (1.0, 2600.0, 4000.0, -2900.0), (1.0, -1500.0, 3000.0, -6000.0)]
    _run(harness, big, lights)
