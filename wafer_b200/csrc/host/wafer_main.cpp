// wafer_main.cpp — `wafer-b200`: the reference's driver (src/main.rs:94-240, src/grid.rs:31-246) over the C ABI.
//
// Same wafer.yaml, same CLI flags (-c/--config, -s/--script, -d), same per-state loop, same table rows
// (output.rs:497-521) and observables record (output.rs:32-45, 533-547).  Everything numerical happens in
// libwafer_b200.so on the GPU, the array files included (wafer_load_array, wafer_write_array); this file is host glue: configuration,
// potential / initial-condition selection, the observables files, printing.
//
//   wafer-b200 -c wafer.yaml                 run (one process per GPU; RANK / WORLD_SIZE / LOCAL_RANK select a slab)
//   wafer-b200 -c wafer.yaml --check-config  parse + validate only, print the configuration as JSON (no GPU needed)
//   wafer-b200 -c wafer.yaml --seed N        key of the Gaussian initial condition (default 0): same N, same start
#include <sys/stat.h>
#include <sys/types.h>
#include <unistd.h>

#include <cerrno>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <fstream>
#include <iostream>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/wafer_b200.h"
#include "config.hpp"
#include "formats.hpp"

using namespace wafer_host;

namespace {

struct Dims {
    size_t nx, ny, nz, e, px, py, pz;
    explicit Dims(const Config& c) : nx(c.nx), ny(c.ny), nz(c.nz), e(c.ext()), px(nx + 2 * e), py(ny + 2 * e), pz(nz + 2 * e) {}
    size_t padded() const { return px * py * pz; }
    size_t p(size_t i, size_t j, size_t k) const { return (i * py + j) * pz + k; }
};

std::string ordinal(unsigned n) {
    const char* suf = "th";
    if (n % 100 < 11 || n % 100 > 13) {
        if (n % 10 == 1) suf = "st";
        else if (n % 10 == 2) suf = "nd";
        else if (n % 10 == 3) suf = "rd";
    }
    return std::to_string(n) + suf;
}

// array files in (input.rs:32-127, 513-662), embedded as fill_data / read_csv do (input.rs:149-176, 641-657; formats.hpp
// embed_work is the host restatement): what 0 psi, 1 V, 2 push a lower state.  The file found is decoded on the device
// (wafer_load_array); a file it does not take (not in the host writers' layout, or too large for the device) goes
// through formats.hpp's reader and the wafer_*_resampled entry, with that path's messages and refusals.  Out:
// wafer_write_array (write_array_file below).
bool load_input(wafer_ctx* ctx, int what, const std::string& stem, int file_type, const Dims& d) {
    int used = 0;
    if (!find_array(stem, file_type, &used)) return false;
    if (wafer_load_array(ctx, what, used, (stem + extension(used)).c_str(), nullptr) == WAFER_OK) return true;
    const Array3 a = read_typed(stem, used);
    if (a.nx < 2 || a.ny < 2 || a.nz < 2) throw std::runtime_error("ArrayShape: " + stem + " cannot be resized");
    const uint32_t from_csv = used == 1 ? 1 : 0;
    if (!from_csv && a.nx == d.px && a.ny == d.py && a.nz == d.pz)
        throw std::runtime_error("input array already has the padded size: the reference's fill_data cannot load it (input.rs:167-169)");
    static const char* entry[3] = {"wafer_set_phi_resampled", "wafer_set_potential_resampled", "wafer_push_lower_resampled"};
    const int rc = what == 0 ? wafer_set_phi_resampled(ctx, a.data.data(), a.nx, a.ny, a.nz, from_csv)
                   : what == 1 ? wafer_set_potential_resampled(ctx, a.data.data(), a.nx, a.ny, a.nz, from_csv)
                               : wafer_push_lower_resampled(ctx, a.data.data(), a.nx, a.ny, a.nz, from_csv);
    if (rc != WAFER_OK) throw std::runtime_error(std::string(entry[what]) + ": " + wafer_last_error(ctx));
    return true;
}

// input::script_potential (input.rs:186-248): JSON grid on stdin, one float per stdout line, work area x-major
void script_potential(const Config& c, std::vector<double>& padded, const Dims& d) {
    char tmpl[] = "/tmp/wafer_script_XXXXXX";
    const int fd = mkstemp(tmpl);
    if (fd < 0) throw std::runtime_error("StdIn: cannot create a temporary file");
    char buf[256];
    const int len = snprintf(buf, sizeof buf, "{\"grid\":{\"dn\":%.17g,\"x\":%llu,\"y\":%llu,\"z\":%llu}}", c.dn,
                             (unsigned long long)c.nx, (unsigned long long)c.ny, (unsigned long long)c.nz);
    if (write(fd, buf, len) != len) throw std::runtime_error("StdIn: short write");
    close(fd);
    const std::string cmd = "\"" + c.script_location + "\" < " + tmpl;
    FILE* p = popen(cmd.c_str(), "r");
    if (!p) throw std::runtime_error("SpawnPython: " + c.script_location);
    std::fill(padded.begin(), padded.end(), 0.0);
    size_t n = 0;
    char line[128];
    while (fgets(line, sizeof line, p)) {
        char* end = nullptr;
        const double v = strtod(line, &end);
        if (end == line) { pclose(p); unlink(tmpl); throw std::runtime_error("ParseFloat: script output"); }
        if (n < d.nx * d.ny * d.nz) {
            const size_t i = n / (d.ny * d.nz), j = (n / d.nz) % d.ny, k = n % d.nz;
            padded[d.p(i + d.e, j + d.e, k + d.e)] = v;
        }
        ++n;
    }
    const int rc = pclose(p);
    unlink(tmpl);
    if (rc != 0) throw std::runtime_error("SpawnPython: script exited with status " + std::to_string(rc));
    if (n != d.nx * d.ny * d.nz) throw std::runtime_error("ArrayShape: script printed " + std::to_string(n) + " values");
}

// potential.rs:374-398 (host copies for the FullCornell pot_sub array, potential.rs:326-341 at WORK indices)
double alphas(double mu) {
    const double nf = 2.0, b0 = 11. - 2. * nf / 3., b1 = 51. - 19. * nf / 3.;
    const double b2 = 2857. - 5033. * nf / 9. + 325. * nf * nf / 27., r = 2.3, l = 2. * std::log(mu / r), ll = std::log(l);
    return 4. * M_PI * (1. - 2. * b1 * ll / (b0 * b0 * l) + 4. * b1 * b1 * ((ll - 0.5) * (ll - 0.5) + b2 * b0 / (8. * b1 * b1) - 5.0 / 4.0) / (b0 * b0 * b0 * b0 * l * l)) / (b0 * l);
}
double debye_mu(double t) { return 1.4 * std::sqrt((1. + 2.0 / 6.) * 4. * M_PI * alphas(2. * M_PI * t)) * t * 0.2; }

std::vector<double> full_cornell_pot_sub(const Config& c) {
    std::vector<double> out(c.nx * c.ny * c.nz);
    const double xi = 0.0, mu1 = debye_mu(1.0);
    for (size_t i = 0; i < c.nx; ++i)
        for (size_t j = 0; j < c.ny; ++j)
            for (size_t k = 0; k < c.nz; ++k) {
                const double dx = (double)i - ((double)c.nx + 1.) / 2., dy = (double)j - ((double)c.ny + 1.) / 2.;
                const double dz = (double)k - ((double)c.nz + 1.) / 2.;
                const double r = c.dn * std::sqrt(dx * dx + dy * dy + dz * dz);
                const double md = mu1 * 1. + (0.07 * std::pow(xi, 0.2)) * (1. - c.dn * c.dn * dz * dz / (r * r)) * std::pow(1. + xi, -0.29);
                out[(i * c.ny + j) * c.nz + k] = c.sig / md + 4. * c.mass;
            }
    return out;
}

struct Run {
    Config cfg;
    wafer_ctx* ctx = nullptr;
    int rank = 0, world = 1;
    std::string outdir;
    bool quiet = false;
    void ck(int rc, const char* what) const {
        if (rc != WAFER_OK) throw std::runtime_error(std::string(what) + ": " + wafer_last_error(ctx));
    }
};

// output.rs:497-521
std::string measurement_row(double tau, double diff, const wafer_observables& o) {
    char b[160];
    if (tau > 0.0)
        snprintf(b, sizeof b, "     │%11.3f │%19.10e │%15.5f │%15.5e │", tau, o.energy / o.norm2, std::sqrt(o.r2 / o.norm2), diff);
    else
        snprintf(b, sizeof b, "     │%11.3f │%19.10e │%15.5f │%15s │", tau, o.energy / o.norm2, std::sqrt(o.r2 / o.norm2), "--   ");
    return b;
}

void write_observables(const Run& r, unsigned wnum, const wafer_observables& o) {
    // ObservablesOutput (output.rs:32-45, 533-547)
    const double rn = std::sqrt(o.r2 / o.norm2), energy = o.energy / o.norm2, binding = (o.energy - o.v_infinity) / o.norm2;
    const double l_r = (double)r.cfg.nx / rn;
    if (!r.quiet) {
        if (wnum == 0) printf("══▶ Ground state energy = %.15g\n══▶ Ground state binding energy = %.15g\n", energy, binding);
        else printf("══▶ %s excited state energy = %.15g\n══▶ %s excited state binding energy = %.15g\n", ordinal(wnum).c_str(), energy,
                    ordinal(wnum).c_str(), binding);
        printf("══▶ rᵣₘₛ = %.15g\n══▶ L/rᵣₘₛ = %.15g\n\n", rn, l_r);
    }
    if (r.outdir.empty() || r.rank != 0) return;
    const int ft = r.cfg.file_type;
    const std::string stem = r.outdir + "/observables_" + std::to_string(wnum);
    if (ft == 0) {  // rmp-serde: the struct as a 5-element array (output.rs:604-620)
        std::string o;
        mp::put_array_header(o, 5);
        mp::put_uint(o, wnum);
        mp::put_f64(o, energy); mp::put_f64(o, binding); mp::put_f64(o, rn); mp::put_f64(o, l_r);
        write_file(stem + ".mpk", o);
        return;
    }
    const std::string path = stem + (ft == 1 ? ".csv" : ".json");
    FILE* f = fopen(path.c_str(), "w");
    if (!f) throw std::runtime_error("CreateFile: " + path);
    if (ft == 1) fprintf(f, "state,energy,binding_energy,r,l_r\n%u,%.17g,%.17g,%.17g,%.17g\n", wnum, energy, binding, rn, l_r);
    else fprintf(f, "{\"state\":%u,\"energy\":%.17g,\"binding_energy\":%.17g,\"r\":%.17g,\"l_r\":%.17g}\n", wnum, energy, binding, rn, l_r);
    fclose(f);
}

// output.rs:79-216: the work area of psi (what 0) or V (what 1), encoded on the device, formats.hpp's bytes.  With
// world > 1 every rank calls it and writes its planes into the one file.
void write_array_file(const Run& r, int what, const std::string& stem) {
    if (r.cfg.file_type > 2) throw std::runtime_error("output.file_type Yaml / Ron is not supported by this build (use Messagepack, Csv or Json)");
    r.ck(wafer_write_array(r.ctx, what, r.cfg.file_type, (stem + extension(r.cfg.file_type)).c_str(), nullptr), "wafer_write_array");
}

void save_wavefunction(const Run& r, unsigned wnum, bool converged) {
    if (r.outdir.empty()) return;
    write_array_file(r, 0, r.outdir + "/wavefunction_" + std::to_string(wnum) + (converged ? "" : "_partial"));
}

// grid.rs:50-246 for one state; returns true when converged
bool solve(Run& r, unsigned wnum) {
    const Config& c = r.cfg;
    const Dims d(c);
    if (wnum > 0) {
        // grid.rs:60-96: a wavefunction_{wnum} file in ./input wins, else start from the previous converged state
        if (!load_input(r.ctx, 0, "input/wavefunction_" + std::to_string(wnum), c.file_type, d)) {
            // grid.rs:95 clones w_store[wnum-1] and lets rounding noise seed the new state (SURVEY F7); here the
            // clone is multiplied by a fixed symmetry-free polynomial so the start is well defined and reproducible
            r.ck(wafer_phi_seed_from_lower(r.ctx, wnum - 1), "wafer_phi_seed_from_lower");
        }
    }
    if (!r.quiet && r.rank == 0) {
        if (wnum == 0) printf("\n═════╤════════════╤════════ Ground state caclulation ════════╤════════════════╤═════\n");
        else printf("\n═════╤════════════╤═════ %s excited state caclulation ═════╤════════════════╤═════\n", ordinal(wnum).c_str());
        printf("     │  Time (τ)  │       Energy       │      rᵣₘₛ      │   Difference   │\n");
        printf("─────┼────────────┼────────────────────┼────────────────┼────────────────┼─────\n");
    }
    uint64_t step = 0;
    double last_energy = 1.7976931348623157e308;
    bool converged = false;
    wafer_observables obs{};
    for (;;) {
        r.ck(wafer_check(r.ctx, (uint8_t)wnum, &obs), "wafer_check");                                   // grid.rs:127-135
        if (!std::isfinite(obs.energy) || !std::isfinite(obs.norm2) || obs.norm2 == 0.0)
            throw std::runtime_error("non-finite observables (the reference's R64 would panic here)");
        const double norm_energy = obs.energy / obs.norm2, tau = (double)step * c.dt;
        if (c.snap_update && step % *c.snap_update == 0) {                                               // grid.rs:137-158
            r.ck(wafer_symmetrise(r.ctx, c.init_symmetry), "wafer_symmetrise");                          // grid.rs:137-139
            r.ck(wafer_normalise(r.ctx, obs.norm2), "wafer_normalise");
            save_wavefunction(r, wnum, false);
        }
        const double diff = std::fabs(norm_energy - last_energy);
        if (!r.quiet && r.rank == 0) { puts(measurement_row(tau, diff, obs).c_str()); fflush(stdout); }
        if (diff < c.tolerance) { converged = true; break; }                                             // grid.rs:162-192
        last_energy = norm_energy;
        if (c.max_steps && step > *c.max_steps) break;                                                   // grid.rs:211-213
        r.ck(wafer_evolve(r.ctx, (uint8_t)wnum, c.screen_update), "wafer_evolve");                       // grid.rs:216
        step += c.screen_update;
    }
    if (converged) {
        if (!r.quiet && r.rank == 0) printf("═════╧════════════╧════════════════════╧════════════════╧════════════════╧═════\n");
        if (r.rank == 0) write_observables(r, wnum, obs);
        if (c.snap_update && !r.outdir.empty() && r.rank == 0)                                           // grid.rs:174-190
            unlink((r.outdir + "/wavefunction_" + std::to_string(wnum) + "_partial" + extension(c.file_type)).c_str());
    }
    if (c.save_wavefns) save_wavefunction(r, wnum, converged);                                           // grid.rs:223-237
    if (converged) r.ck(wafer_push_lower_from_phi(r.ctx), "wafer_push_lower_from_phi");                  // grid.rs:241
    return converged;
}

// rank 0 writes the ncclUniqueId and its output directory (empty: none) to a file, the others poll for it (no MPI /
// torch needed); every rank writes its planes of the array files there
void rendezvous(const std::string& path, int rank, uint8_t id[128], std::string& outdir) {
    if (rank == 0) {
        if (wafer_nccl_unique_id(id) != WAFER_OK) throw std::runtime_error(std::string("wafer_nccl_unique_id: ") + wafer_last_error(nullptr));
        const std::string tmp = path + ".tmp";
        FILE* f = fopen(tmp.c_str(), "wb");
        if (!f || fwrite(id, 1, 128, f) != 128 || fwrite(outdir.data(), 1, outdir.size(), f) != outdir.size())
            throw std::runtime_error("rendezvous: cannot write " + tmp);
        fclose(f);
        rename(tmp.c_str(), path.c_str());
    } else {
        for (int tries = 0; tries < 600; ++tries) {
            FILE* f = fopen(path.c_str(), "rb");
            if (f) {
                const size_t n = fread(id, 1, 128, f);
                char buf[4096];
                const size_t m = n == 128 ? fread(buf, 1, sizeof buf, f) : 0;
                fclose(f);
                if (n == 128) {
                    outdir.assign(buf, m);
                    return;
                }
            }
            std::this_thread::sleep_for(std::chrono::milliseconds(100));
        }
        throw std::runtime_error("rendezvous: timed out waiting for " + path);
    }
}

int env_int(const char* k, int dflt) {
    const char* v = getenv(k);
    return v ? atoi(v) : dflt;
}

}  // namespace

int main(int argc, char** argv) {
    std::string config_file = "wafer.yaml", script = "gen_potential.py", outroot = "output", rdv;
    bool check_only = false, no_output = false, quiet = false;
    uint64_t seed = 0;  // fixed default: runs are reproducible and every rank of a multi-GPU run draws the same field
    int verbosity = 0;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto next = [&]() -> std::string {
            if (i + 1 >= argc) { fprintf(stderr, "missing value for %s\n", a.c_str()); exit(2); }
            return argv[++i];
        };
        if (a == "-c" || a == "--config") config_file = next();
        else if (a == "-s" || a == "--script") script = next();
        else if (a == "-d" || a == "-dd" || a == "-ddd") verbosity += (int)a.size() - 1;
        else if (a == "--check-config") check_only = true;
        else if (a == "--seed") {
            const std::string v = next();
            char* end = nullptr;
            errno = 0;
            const unsigned long long n = strtoull(v.c_str(), &end, 10);
            if (v.empty() || v[0] == '-' || *end != 0 || errno == ERANGE) {
                fprintf(stderr, "--seed expects an unsigned 64-bit integer, got %s\n", v.c_str());
                return 2;
            }
            seed = n;
        }
        else if (a == "--selftest-trilerp") {
            // the reference's `interpolation` unit test input (input.rs:733-748): 2x2x2 [1..8] -> 4x4x4
            Array3 v, out;
            v.nx = v.ny = v.nz = 2;
            v.data = {1, 2, 3, 4, 5, 6, 7, 8};
            out.nx = out.ny = out.nz = 4;
            out.data.assign(64, 0.0);
            trilerp_resize(v, out);
            for (double d : out.data) printf("%.17g\n", d);
            return 0;
        } else if (a == "--selftest-formats") {
            // write a deterministic 3x4x5 array in every supported format under the given directory, read it back
            const std::string dir = next();
            Array3 v;
            v.nx = 3; v.ny = 4; v.nz = 5;
            for (int i = 0; i < 60; ++i) v.data.push_back(std::sin(0.37 * i) * std::pow(10.0, (i % 7) - 3));
            for (int ft = 0; ft < 3; ++ft) {
                write_array(dir + "/array", ft, v);
                Array3 back;
                if (!read_array(dir + "/array", ft, back) || back.nx != 3 || back.ny != 4 || back.nz != 5 || back.data != v.data) {
                    fprintf(stderr, "format %d round trip failed\n", ft);
                    return 1;
                }
            }
            std::vector<double> padded(5 * 6 * 7);
            embed_work(v, padded, 3, 4, 5, 1, /*from_csv=*/true);  // a work-sized csv is copied straight in (input.rs:641-650)
            if (extract_work(padded.data(), 3, 4, 5, 1).data != v.data) return 1;
            // a work-sized Messagepack / Json array is NOT "same" for the reference (input.rs:161-172): it is re-sampled
            // on a basis of padded-size many points; check the first axis against the formula
            embed_work(v, padded, 3, 4, 5, 1, false);
            {
                const Array3 w = extract_work(padded.data(), 3, 4, 5, 1);
                const double xl = 2.0 / 4.0;  // linspace(0, 2, 5)[1]
                const double want = v.at(0, 0, 0) * (1. - xl) + v.at(1, 0, 0) * xl;
                if (std::fabs(w.at(1, 0, 0) - want) > 1e-15 * std::fabs(want) || w.at(0, 0, 0) != v.at(0, 0, 0)) return 1;
            }
            puts("formats ok");
            return 0;
        }
        else if (a == "--no-output") no_output = true;
        else if (a == "--output-root") outroot = next();
        else if (a == "--rendezvous-file") rdv = next();
        else if (a == "-q" || a == "--quiet") quiet = true;
        else if (a == "-h" || a == "--help") {
            puts("wafer-b200 [-c wafer.yaml] [-s gen_potential.py] [-d] [--check-config] [--no-output] [--output-root DIR] [-q]\n"
                 "           [--seed N]   key of the Gaussian initial condition (default 0); the same N gives the same start\n"
                 "                        on any number of GPUs");
            return 0;
        } else { fprintf(stderr, "unknown argument %s\n", a.c_str()); return 2; }
    }
    (void)verbosity;
    try {
        Run r;
        r.cfg = load_config_file(config_file);
        r.cfg.seed = seed;
        r.quiet = quiet;
        if (r.cfg.potential == 13) r.cfg.script_location = "./" + script;  // config.rs:344-350
        if (check_only) {
            puts(config_json(r.cfg).c_str());
            return 0;
        }
        const Config& c = r.cfg;
        r.rank = env_int("RANK", 0);
        r.world = env_int("WORLD_SIZE", 1);
        if (!no_output && r.rank == 0) {
            // output::check_output_dir (output.rs:680-745): ./output/<project>_<date>/ + a copy of the configuration
            char date[64];
            const time_t now = time(nullptr);
            strftime(date, sizeof date, "%Y-%m-%d_%H:%M:%S", localtime(&now));
            mkdir(outroot.c_str(), 0755);
            r.outdir = outroot + "/" + c.project_name + "_" + date;
            mkdir(r.outdir.c_str(), 0755);
            std::ifstream src(config_file, std::ios::binary);
            std::ofstream dst(r.outdir + "/wafer.yaml", std::ios::binary);
            dst << src.rdbuf();
        }
        uint8_t id[128];
        if (r.world > 1) rendezvous(rdv.empty() ? "/tmp/wafer_b200_nccl_id_" + std::to_string(getppid()) : rdv, r.rank, id, r.outdir);
        wafer_params p{};
        p.nx = c.nx; p.ny = c.ny; p.nz = c.nz; p.ext = (uint32_t)c.ext();
        p.dn = c.dn; p.dt = c.dt; p.mass = c.mass;
        p.device = env_int("LOCAL_RANK", -1);
        p.rank = (uint32_t)r.rank; p.world = (uint32_t)r.world; p.nccl_id = r.world > 1 ? id : nullptr;
        p.max_lower = c.wavemax;
        if (wafer_create(&p, &r.ctx) != WAFER_OK) throw std::runtime_error(std::string("wafer_create: ") + wafer_last_error(nullptr));
        const Dims d(c);
        const auto t0 = std::chrono::steady_clock::now();

        // potential::load_arrays (potential.rs:75-175)
        if (c.potential == 12) {  // FromFile
            if (!load_input(r.ctx, 1, "input/potential", c.file_type, d)) throw std::runtime_error("LoadPotential: input/potential.{mpk,csv,json} not found");
        } else if (c.potential == 13) {  // FromScript
            std::vector<double> v(d.padded());
            script_potential(c, v, d);
            r.ck(wafer_set_potential(r.ctx, v.data()), "wafer_set_potential");
        } else {
            r.ck(wafer_generate_potential(r.ctx, c.potential, c.sig), "wafer_generate_potential");
        }
        if (c.potential == 8) {  // FullCornell: variable pot_sub (potential.rs:134-144)
            const std::vector<double> ps = full_cornell_pot_sub(c);
            r.ck(wafer_set_pot_sub_array(r.ctx, ps.data()), "wafer_set_pot_sub_array");
        } else {                 // potential.rs:346-363
            const double ps = c.potential == 6 ? 1. / c.dn : (c.potential == 7 ? 4.0 * c.mass : 0.0);
            r.ck(wafer_set_pot_sub_scalar(r.ctx, ps), "wafer_set_pot_sub_scalar");
        }
        if (c.save_potential && !r.outdir.empty()) write_array_file(r, 1, r.outdir + "/potential");  // potential.rs:163-172

        // run (grid.rs:31-47): lower states from ./input when starting above the ground state
        for (unsigned w = 0; w < c.wavenum; ++w) {  // input::load_wavefunctions (input.rs:487-505)
            if (!load_input(r.ctx, 2, "input/wavefunction_" + std::to_string(w), c.file_type, d))
                throw std::runtime_error("LoadWavefunction: input/wavefunction_" + std::to_string(w) + ".{mpk,csv,json} is required when wavenum > 0");
        }
        // config::set_initial_conditions (config.rs:577-627)
        if (c.wavenum == 0) {
            if (c.init_condition == 0) {
                if (!load_input(r.ctx, 0, "input/wavefunction_0", c.file_type, d)) throw std::runtime_error("LoadWavefunction: input/wavefunction_0.{mpk,csv,json} not found");
            } else if (c.init_condition == 1) {  // Gaussian (config.rs:636-642): thread_rng there; seeded on the device here
                r.ck(wafer_generate_gaussian(r.ctx, c.sig, c.seed), "wafer_generate_gaussian");
            } else {
                r.ck(wafer_generate_initial_condition(r.ctx, c.init_condition), "wafer_generate_initial_condition");
            }
            r.ck(wafer_symmetrise(r.ctx, c.init_symmetry), "wafer_symmetrise");                          // config.rs:625
        }
        int rc = 0;
        for (unsigned wnum = c.wavenum; wnum <= c.wavemax; ++wnum) {
            if (!solve(r, wnum)) {  // Err(MaxStep) aborts the remaining states (grid.rs:44, 244)
                fprintf(stderr, "Error: Maximum step limit reached before convergence of state %u\n", wnum);
                rc = 1;
                break;
            }
        }
        wafer_synchronize(r.ctx);
        if (!quiet && r.rank == 0) {
            const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            printf("Simulation complete. Elapsed time: %.3fs; %llu kernel launches; sweep variant %s\n", s,
                   (unsigned long long)wafer_kernel_launches(r.ctx), wafer_sweep_variant(r.ctx));
        }
        wafer_destroy(r.ctx);
        return rc;
    } catch (const std::exception& e) {
        fprintf(stderr, "Error: %s\n", e.what());
        return 1;
    }
}
