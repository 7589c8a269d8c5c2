// config.hpp — the reference's `wafer.yaml` schema (src/config.rs:292-333, annotated sample wafer.yaml:13-102) for the
// C++ front end.  Host-side only, no GPU code.  The YAML subset parser handles what the schema uses: nested block
// mappings by indentation, scalars, `#` comments.  Checks and error texts follow Config::parse (config.rs:362-370)
// and errors.rs.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <fstream>
#include <map>
#include <optional>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

namespace wafer_host {

struct ConfigError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// PotentialType (config.rs:74-104), InitialCondition (config.rs:153-170), CentralDifference (config.rs:213-239),
// FileType (config.rs:253-289), SymmetryConstraint (config.rs:186-197): index = position in the enum
inline const std::vector<std::string>& potential_names() {
    static const std::vector<std::string> v = {"NoPotential", "Cube", "QuadWell", "Periodic", "Coulomb", "ComplexCoulomb",
                                               "ElipticalCoulomb", "SimpleCornell", "FullCornell", "Harmonic",
                                               "ComplexHarmonic", "Dodecahedron", "FromFile", "FromScript"};
    return v;
}
inline const std::vector<std::string>& ic_names() {
    static const std::vector<std::string> v = {"FromFile", "Gaussian", "Coulomb", "Constant", "Boolean"};
    return v;
}
inline const std::vector<std::string>& cd_names() {
    static const std::vector<std::string> v = {"ThreePoint", "FivePoint", "SevenPoint"};
    return v;
}
inline const std::vector<std::string>& filetype_names() {
    static const std::vector<std::string> v = {"Messagepack", "Csv", "Json", "Yaml", "Ron"};
    return v;
}
inline const std::vector<std::string>& symmetry_names() {
    static const std::vector<std::string> v = {"NotConstrained", "AboutZ", "AntisymAboutZ", "AboutY", "AntisymAboutY"};
    return v;
}

struct Config {
    std::string project_name;
    uint64_t nx = 0, ny = 0, nz = 0;  // grid.size
    double dn = 0, dt = 0;            // grid.dn, grid.dt
    double tolerance = 0;
    int central_difference = 0;       // index into cd_names(); ext = index + 1, bb = 2 ext
    std::optional<uint64_t> max_steps;
    unsigned wavenum = 0, wavemax = 0;
    uint64_t screen_update = 0;
    std::optional<uint64_t> snap_update;
    int file_type = 0;
    bool save_wavefns = false, save_potential = false;
    int potential = 0;
    double mass = 0;
    int init_condition = 0;
    double sig = 0;
    int init_symmetry = 0;
    std::string script_location;  // set from the command line, never from YAML (config.rs:331)
    uint64_t seed = 0;            // --seed: key of the Gaussian initial condition (the reference draws from thread_rng)

    int ext() const { return central_difference + 1; }
    std::string file_extension() const {  // FileType::extentsion (config.rs:280-288)
        static const char* e[] = {".mpk", ".csv", ".json", ".yaml", ".ron"};
        return e[file_type];
    }
};

namespace detail {
inline std::string trim(const std::string& s) {
    const size_t a = s.find_first_not_of(" \t\r\n");
    if (a == std::string::npos) return "";
    const size_t b = s.find_last_not_of(" \t\r\n");
    return s.substr(a, b - a + 1);
}
inline std::string strip_comment(const std::string& line) {
    // YAML: '#' starts a comment at line start or after whitespace (wafer.yaml:9-10)
    for (size_t i = 0; i < line.size(); ++i)
        if (line[i] == '#' && (i == 0 || line[i - 1] == ' ' || line[i - 1] == '\t')) return line.substr(0, i);
    return line;
}
inline std::string unquote(const std::string& s) {
    if (s.size() >= 2 && ((s.front() == '"' && s.back() == '"') || (s.front() == '\'' && s.back() == '\'')))
        return s.substr(1, s.size() - 2);
    return s;
}
// flattens nested block mappings into "a.b.c" -> scalar
inline std::map<std::string, std::string> flatten_yaml(std::istream& in) {
    std::map<std::string, std::string> out;
    std::vector<std::pair<int, std::string>> stack;  // (indent, key)
    std::string raw;
    int lineno = 0;
    while (std::getline(in, raw)) {
        ++lineno;
        std::string line = strip_comment(raw);
        if (trim(line).empty()) continue;
        if (line.find('\t') != std::string::npos && trim(line.substr(0, line.find_first_not_of(" \t"))).empty() &&
            line[0] == '\t')
            throw ConfigError("Deserialize: tab indentation at line " + std::to_string(lineno));
        const int indent = (int)line.find_first_not_of(' ');
        const std::string body = trim(line);
        const size_t colon = body.find(':');
        if (colon == std::string::npos) throw ConfigError("Deserialize: expected `key: value` at line " + std::to_string(lineno));
        const std::string key = trim(body.substr(0, colon));
        const std::string val = trim(body.substr(colon + 1));
        while (!stack.empty() && stack.back().first >= indent) stack.pop_back();
        std::string path;
        for (auto& s : stack) path += s.second + ".";
        path += key;
        if (val.empty()) stack.emplace_back(indent, key);
        else out[path] = unquote(val);
    }
    return out;
}
inline int enum_index(const std::vector<std::string>& names, const std::string& v, const std::string& what) {
    for (size_t i = 0; i < names.size(); ++i)
        if (names[i] == v) return (int)i;
    throw ConfigError("Deserialize: unknown variant `" + v + "` for " + what);
}
inline double to_f64(const std::string& s, const std::string& key) {
    char* end = nullptr;
    const double v = std::strtod(s.c_str(), &end);
    if (end == s.c_str() || *end != 0 || !std::isfinite(v)) throw ConfigError("Deserialize: `" + key + "` is not a finite number: " + s);
    return v;
}
inline uint64_t to_u64(const std::string& s, const std::string& key) {
    char* end = nullptr;
    if (!s.empty() && s[0] == '-') throw ConfigError("Deserialize: `" + key + "` must be non-negative: " + s);
    const unsigned long long v = std::strtoull(s.c_str(), &end, 10);
    if (end == s.c_str() || *end != 0) throw ConfigError("Deserialize: `" + key + "` is not an integer: " + s);
    return v;
}
inline bool to_bool(const std::string& s, const std::string& key) {
    if (s == "true") return true;
    if (s == "false") return false;
    throw ConfigError("Deserialize: `" + key + "` is not a bool: " + s);
}
}  // namespace detail

// Config::load + Config::parse (config.rs:337-370) without the output-directory side effects
inline Config load_config(std::istream& in) {
    using namespace detail;
    const auto kv = flatten_yaml(in);
    auto need = [&](const std::string& k) -> const std::string& {
        auto it = kv.find(k);
        if (it == kv.end()) throw ConfigError("Deserialize: missing field `" + k + "`");
        return it->second;
    };
    auto opt = [&](const std::string& k) -> std::optional<std::string> {
        auto it = kv.find(k);
        if (it == kv.end() || it->second == "~" || it->second == "null") return std::nullopt;
        return it->second;
    };
    Config c;
    c.project_name = need("project_name");
    c.nx = to_u64(need("grid.size.x"), "grid.size.x");
    c.ny = to_u64(need("grid.size.y"), "grid.size.y");
    c.nz = to_u64(need("grid.size.z"), "grid.size.z");
    c.dn = to_f64(need("grid.dn"), "grid.dn");
    c.dt = to_f64(need("grid.dt"), "grid.dt");
    c.tolerance = to_f64(need("tolerance"), "tolerance");
    c.central_difference = enum_index(cd_names(), need("central_difference"), "central_difference");
    if (auto m = opt("max_steps")) c.max_steps = to_u64(*m, "max_steps");
    const uint64_t wn = to_u64(need("wavenum"), "wavenum"), wm = to_u64(need("wavemax"), "wavemax");
    if (wn > 255 || wm > 255) throw ConfigError("Deserialize: wavenum / wavemax are u8");
    c.wavenum = (unsigned)wn;
    c.wavemax = (unsigned)wm;
    c.screen_update = to_u64(need("output.screen_update"), "output.screen_update");
    if (auto s = opt("output.snap_update")) c.snap_update = to_u64(*s, "output.snap_update");
    // the reference computes step % snap_update (grid.rs:137): 0 would be a division by zero there too — refuse it up front
    if (c.snap_update && *c.snap_update == 0) throw ConfigError("output.snap_update must be positive when given");
    c.file_type = enum_index(filetype_names(), need("output.file_type"), "output.file_type");
    // Yaml / Ron array files are valid in the reference but not written by this front end: say so before any GPU work,
    // not when a converged wavefunction is about to be saved
    if (c.file_type > 2) throw ConfigError("output.file_type " + filetype_names()[c.file_type] + " is not supported by this build (use Messagepack, Csv or Json)");
    c.save_wavefns = to_bool(need("output.save_wavefns"), "output.save_wavefns");
    c.save_potential = to_bool(need("output.save_potential"), "output.save_potential");
    c.potential = enum_index(potential_names(), need("potential"), "potential");
    c.mass = to_f64(need("mass"), "mass");
    c.init_condition = enum_index(ic_names(), need("init_condition"), "init_condition");
    c.sig = to_f64(need("sig"), "sig");
    c.init_symmetry = enum_index(symmetry_names(), need("init_symmetry"), "init_symmetry");
    // Config::parse (config.rs:362-370); messages from errors.rs (LargeDt, LargeWavenum)
    if (c.dt > c.dn * c.dn / 3.) throw ConfigError("LargeDt: Temporal step (grid.dt) is too large for the spatial step: must be <= grid.dn^2/3");
    if (c.wavenum > c.wavemax) throw ConfigError("LargeWavenum: wavenum can not be larger than wavemax");
    if (c.nx == 0 || c.ny == 0 || c.nz == 0) throw ConfigError("Deserialize: grid.size must be positive");
    if (c.screen_update == 0) throw ConfigError("Deserialize: output.screen_update must be positive");
    // an antisymmetric state about an axis of one site is identically zero: its first check would divide 0 by 0
    if ((c.init_symmetry == 2 && c.nz == 1) || (c.init_symmetry == 4 && c.ny == 1))
        throw ConfigError("init_symmetry " + symmetry_names()[c.init_symmetry] + " needs more than one site along " +
                          (c.init_symmetry == 2 ? "z" : "y") + ": the constrained state would be zero everywhere");
    return c;
}

inline Config load_config_file(const std::string& path) {
    std::ifstream f(path);
    if (!f) throw ConfigError("ConfigLoad: cannot open " + path);
    return load_config(f);
}

inline std::string config_json(const Config& c) {
    std::ostringstream o;
    o.precision(17);
    o << "{\"project_name\": \"" << c.project_name << "\", \"grid\": {\"size\": {\"x\": " << c.nx << ", \"y\": " << c.ny
      << ", \"z\": " << c.nz << "}, \"dn\": " << c.dn << ", \"dt\": " << c.dt << "}, \"tolerance\": " << c.tolerance
      << ", \"central_difference\": \"" << cd_names()[c.central_difference] << "\", \"max_steps\": ";
    if (c.max_steps) o << *c.max_steps; else o << "null";
    o << ", \"wavenum\": " << c.wavenum << ", \"wavemax\": " << c.wavemax << ", \"output\": {\"screen_update\": "
      << c.screen_update << ", \"snap_update\": ";
    if (c.snap_update) o << *c.snap_update; else o << "null";
    o << ", \"file_type\": \"" << filetype_names()[c.file_type] << "\", \"save_wavefns\": " << (c.save_wavefns ? "true" : "false")
      << ", \"save_potential\": " << (c.save_potential ? "true" : "false") << "}, \"potential\": \""
      << potential_names()[c.potential] << "\", \"mass\": " << c.mass << ", \"init_condition\": \"" << ic_names()[c.init_condition]
      << "\", \"sig\": " << c.sig << ", \"init_symmetry\": \"" << symmetry_names()[c.init_symmetry] << "\", \"ext\": " << c.ext()
      << ", \"seed\": " << c.seed << "}";
    return o.str();
}

}  // namespace wafer_host
