// nbtool — what the reference has no CLI for (SURVEY.md 8f rank 4): reproducible synthetic systems, ensembles of
// systems and state files, all in the reference's own input format (nbody.cc:22-39) so that every file also goes
// through `hw5` and through samples/nbody.cc.  Host code above the C ABI; `hw5 <input> <output>` stays flag-free.
//
//   nbtool gen <n> <seed> <out.in> [n_devices=4]          synthetic system (SURVEY 8d config C5)
//   nbtool advance <in> <steps> <out.in>                   run_step x steps from step 0 (nbody.cc:51-89), state written
//   nbtool ensemble <in> <members> <steps> <out.txt>       members k = 0..S-1: velocities scaled by (1 + 1e-9 k)
//                                                          (config C4), same n, split over all visible GPUs, one
//                                                          line per member: k min_dist argmin_step hit_step
//   nbtool ensemble-list <list.txt> <steps> <out.txt>      the same for the input files named in list.txt (equal n)
//   nbtool diag <in> [step=0]                              mass, energies, momentum and angular momentum of the state
//                                                          with the masses of `step` (nb_diagnostics), one line each
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/nbody_b200.h"

namespace {

struct Sys {
    int n = 0, planet = 0, asteroid = 0;
    std::vector<double> q, v, m;
    std::vector<unsigned char> dev;
};

int fail(int rc, const char* what) {
    fprintf(stderr, "nbtool: %s: %s: %s\n", what, nb_strerror(rc), nb_last_error_detail());
    return 1;
}

int load(const char* path, Sys& s) {
    int rc = nb_read_header(path, &s.n, &s.planet, &s.asteroid);
    if (rc) return rc;
    s.q.resize(3 * (size_t)s.n), s.v.resize(3 * (size_t)s.n), s.m.resize(s.n), s.dev.resize(s.n);
    return nb_read_input(path, s.n, &s.n, &s.planet, &s.asteroid, s.q.data(), s.v.data(), s.m.data(), s.dev.data());
}

// S systems of the same n (system-major arrays) to step_end, split over the visible GPUs, one host thread per GPU
int run_members(int n, int S, std::vector<double>& q, std::vector<double>& v, const std::vector<double>& m,
                const std::vector<unsigned char>& dev, const std::vector<int>& planet, const std::vector<int>& asteroid,
                int step_end, std::vector<nb_events>& ev, double* gpu_seconds) {
    int G = 0;
    int rc = nb_device_count(&G);
    if (rc) return rc;
    if (G > S) G = S;
    std::vector<int> rcs(G, NB_OK);
    std::vector<double> secs(G, 0.0);
    std::vector<std::thread> th;
    ev.assign(S, nb_events{});
    for (int g = 0; g < G; g++) {
        th.emplace_back([&, g]() {
            const int s0 = (int)((long long)S * g / G), s1 = (int)((long long)S * (g + 1) / G);
            if (s1 == s0) return;
            rcs[g] = nb_ensemble_run(g, NB_MATH_FAST, NB_KIND_Q2, s1 - s0, n, q.data() + (size_t)s0 * 3 * n,
                                     v.data() + (size_t)s0 * 3 * n, m.data() + (size_t)s0 * n, dev.data() + (size_t)s0 * n,
                                     planet.data() + s0, asteroid.data() + s0, nullptr, 0, step_end, ev.data() + s0, &secs[g]);
        });
    }
    for (auto& t : th) t.join();
    *gpu_seconds = 0;
    for (int g = 0; g < G; g++) {
        if (rcs[g]) return rcs[g];
        if (secs[g] > *gpu_seconds) *gpu_seconds = secs[g];
    }
    return NB_OK;
}

int write_members(const char* path, const std::vector<nb_events>& ev) {
    FILE* f = fopen(path, "wb");
    if (!f) return NB_ERR_IO;
    for (size_t k = 0; k < ev.size(); k++)
        fprintf(f, "%zu %.16e %d %d\n", k, sqrt(ev[k].min_d2), ev[k].argmin_step, ev[k].hit_step);
    return fclose(f) == 0 ? NB_OK : NB_ERR_IO;
}

int usage() {
    fprintf(stderr,
            "usage: nbtool gen <n> <seed> <out.in> [n_devices]\n"
            "       nbtool advance <in> <steps> <out.in>\n"
            "       nbtool ensemble <in> <members> <steps> <out.txt>\n"
            "       nbtool ensemble-list <list.txt> <steps> <out.txt>\n"
            "       nbtool diag <in> [step]\n");
    return 2;
}

}  // namespace

int main(int argc, char** argv) {
    if (argc < 2) return usage();
    const std::string cmd = argv[1];
    if (cmd == "gen" && (argc == 5 || argc == 6)) {
        const int n = atoi(argv[2]), nd = argc == 6 ? atoi(argv[5]) : 4;
        if (n < 2) return usage();
        Sys s;
        s.n = n, s.q.resize(3 * (size_t)n), s.v.resize(3 * (size_t)n), s.m.resize(n), s.dev.resize(n);
        int rc = nb_generate_system(n, strtoull(argv[3], nullptr, 10), nd, s.q.data(), s.v.data(), s.m.data(), s.dev.data(),
                                    &s.planet, &s.asteroid);
        if (rc) return fail(rc, "gen");
        rc = nb_write_input(argv[4], n, s.planet, s.asteroid, s.q.data(), s.v.data(), s.m.data(), s.dev.data());
        return rc ? fail(rc, argv[4]) : 0;
    }
    if (cmd == "advance" && argc == 5) {
        Sys s;
        int rc = load(argv[2], s);
        if (rc) return fail(rc, argv[2]);
        const int steps = atoi(argv[3]);
        rc = nb_run_steps(0, NB_MATH_FAST, s.n, s.q.data(), s.v.data(), s.m.data(), s.dev.data(), 0, steps);
        if (rc) return fail(rc, "advance");
        rc = nb_write_input(argv[4], s.n, s.planet, s.asteroid, s.q.data(), s.v.data(), s.m.data(), s.dev.data());
        return rc ? fail(rc, argv[4]) : 0;
    }
    if (cmd == "diag" && (argc == 3 || argc == 4)) {
        Sys s;
        int rc = load(argv[2], s);
        if (rc) return fail(rc, argv[2]);
        const int step = argc == 4 ? atoi(argv[3]) : 0;
        nb_diag d;
        double secs = 0;
        rc = nb_diagnostics(0, 1, s.n, s.q.data(), s.v.data(), s.m.data(), s.dev.data(), step, &d, &secs);
        if (rc) return fail(rc, "diag");
        printf("step %d\nn %d\nmass %.17g\nkinetic %.17g\npotential %.17g\nenergy %.17g\n", d.step, d.n, d.mass, d.kinetic,
               d.potential, d.kinetic + d.potential);
        const char* axis = "xyz";
        for (int c = 0; c < 3; c++) printf("momentum_%c %.17g\n", axis[c], d.momentum[c]);
        for (int c = 0; c < 3; c++) printf("angular_momentum_%c %.17g\n", axis[c], d.angular_momentum[c]);
        fprintf(stderr, "nbtool: %d bodies: %.6f s of kernels\n", s.n, secs);
        return 0;
    }
    if ((cmd == "ensemble" && argc == 6) || (cmd == "ensemble-list" && argc == 5)) {
        std::vector<Sys> members;
        int steps;
        const char* out;
        if (cmd == "ensemble") {
            Sys base;
            int rc = load(argv[2], base);
            if (rc) return fail(rc, argv[2]);
            const int S = atoi(argv[3]);
            if (S < 1) return usage();
            steps = atoi(argv[4]), out = argv[5];
            members.assign(S, base);
            for (int k = 0; k < S; k++)
                for (auto& x : members[k].v) x *= (1.0 + 1e-9 * k);  // SURVEY 8d config C4; k = 0 is the input itself
        } else {
            FILE* f = fopen(argv[2], "rb");
            if (!f) return fail(NB_ERR_IO, argv[2]);
            char line[4096];
            while (fgets(line, sizeof line, f)) {
                line[strcspn(line, "\r\n")] = 0;
                if (!line[0] || line[0] == '#') continue;
                members.emplace_back();
                int rc = load(line, members.back());
                if (rc) {
                    fclose(f);
                    return fail(rc, line);
                }
                if (members.back().n != members[0].n) {
                    fclose(f);
                    fprintf(stderr, "nbtool: %s has %d bodies, the first file %d: one ensemble = one n\n", line,
                            members.back().n, members[0].n);
                    return 1;
                }
            }
            fclose(f);
            if (members.empty()) return usage();
            steps = atoi(argv[3]), out = argv[4];
        }
        const int S = (int)members.size(), n = members[0].n;
        std::vector<double> q((size_t)S * 3 * n), v((size_t)S * 3 * n), m((size_t)S * n);
        std::vector<unsigned char> dev((size_t)S * n);
        std::vector<int> planet(S), asteroid(S);
        for (int k = 0; k < S; k++) {
            memcpy(&q[(size_t)k * 3 * n], members[k].q.data(), 3 * n * sizeof(double));
            memcpy(&v[(size_t)k * 3 * n], members[k].v.data(), 3 * n * sizeof(double));
            memcpy(&m[(size_t)k * n], members[k].m.data(), n * sizeof(double));
            memcpy(&dev[(size_t)k * n], members[k].dev.data(), n);
            planet[k] = members[k].planet, asteroid[k] = members[k].asteroid;
        }
        std::vector<nb_events> ev;
        double secs = 0;
        int rc = run_members(n, S, q, v, m, dev, planet, asteroid, steps, ev, &secs);
        if (rc) return fail(rc, "ensemble");
        fprintf(stderr, "nbtool: %d systems x %d bodies, %d steps: %.3f s of kernels\n", S, n, steps, secs);
        rc = write_members(out, ev);
        return rc ? fail(rc, out) : 0;
    }
    return usage();
}
