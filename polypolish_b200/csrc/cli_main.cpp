// cli_main.cpp — the `polypolish` command line, drop-in for the reference's (main.rs:23-126).
//
// Same subcommands, flag names (note the underscores), defaults and validation messages:
//   polypolish filter --in1 F --in2 F --out1 F --out2 F [--orientation auto] [--low 0.1] [--high 99.9]
//   polypolish polish [--debug F] [-i|--fraction_invalid 0.2] [-v|--fraction_valid 0.5] [-m|--max_errors 10]
//                     [-d|--min_depth 5] [--careful] <ASSEMBLY> [SAM]...
// Polished FASTA on stdout, log on stderr, "Error: <msg>" + exit 1 on user errors (misc.rs:29-33).
// Additive flags: --device N (first GPU), --gpus N (polish: contigs shard across N GPUs), --quiet, --host-parse (polish: parse the
// SAM text on the host instead of on the device; same output).  All compute happens in libpolypolish_b200.so on the GPU.
#include <cstdio>
#include <unistd.h>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <string>
#include <vector>

#include "../../include/pp_abi.h"

static const char* BANNER =
    "  _____        _                       _  _       _     \n"
    " |  __ \\      | |                     | |(_)     | |    \n"
    " | |__) |___  | | _   _  _ __    ___  | | _  ___ | |__  \n"
    " |  ___// _ \\ | || | | || '_ \\  / _ \\ | || |/ __|| '_ \\ \n"
    " | |   | (_) || || |_| || |_) || (_) || || |\\__ \\| | | |\n"
    " |_|    \\___/ |_| \\__, || .__/  \\___/ |_||_||___/|_| |_|\n"
    "                   __/ || |                             \n"
    "                  |___/ |_|                             \n";

[[noreturn]] static void quit_with_error(const std::string& text) {   // misc.rs:29-33
    fprintf(stderr, "\nError: %s\n", text.c_str());
    exit(1);
}

[[noreturn]] static void usage_error(const std::string& text) {      // clap argument errors exit with 2
    fprintf(stderr, "error: %s\n\nFor more information, try '--help'.\n", text.c_str());
    exit(2);
}

static void help() {                      // `polypolish`, `polypolish -h`: the layout of clap 4's derived help (main.rs:23-42)
    fputs(BANNER, stdout);
    puts("\nshort-read polishing of long-read assemblies\ngithub.com/rrwick/Polypolish\n");
    puts("Usage: polypolish <COMMAND>\n");
    puts("Commands:\n  filter  filter paired-end alignments based on insert size\n  polish  polish a long-read assembly using short-read alignments\n");
    puts("Options:\n  -h, --help     Print help\n  -V, --version  Print version");
}

static void help_filter() {               // main.rs:46-75
    puts("filter paired-end alignments based on insert size\n");
    puts("Usage: polypolish filter [OPTIONS] --in1 <IN1> --in2 <IN2> --out1 <OUT1> --out2 <OUT2>\n");
    puts("Options:");
    puts("      --in1 <IN1>                  Input SAM file - first read in pairs");
    puts("      --in2 <IN2>                  Input SAM file - first second in pairs");
    puts("      --out1 <OUT1>                Output SAM file - first read in pairs");
    puts("      --out2 <OUT2>                Output SAM file - first second in pairs");
    puts("      --orientation <ORIENTATION>  Expected pair orientation [default: auto]");
    puts("      --low <LOW>                  Low percentile threshold [default: 0.1]");
    puts("      --high <HIGH>                High percentile threshold [default: 99.9]");
    puts("  -h, --help                       Print help");
    puts("  -V, --version                    Print version");
    puts("\nB200 build, additive options: --device <N> (GPU, default 0), --quiet, --host-parse");
}

static void help_polish() {               // main.rs:77-108
    puts("polish a long-read assembly using short-read alignments\n");
    puts("Usage: polypolish polish [OPTIONS] <ASSEMBLY> [SAM]...\n");
    puts("Arguments:");
    puts("  <ASSEMBLY>  Assembly to polish (one file in FASTA format)");
    puts("  [SAM]...    Short read alignments (one or more files in SAM format)\n");
    puts("Options:");
    puts("      --debug <DEBUG>");
    puts("          Optional file to store per-base information for debugging purposes");
    puts("  -i, --fraction_invalid <FRACTION_INVALID>");
    puts("          A base must make up less than this fraction of the read depth to be considered invalid [default: 0.2]");
    puts("  -v, --fraction_valid <FRACTION_VALID>");
    puts("          A base must make up at least this fraction of the read depth to be considered valid [default: 0.5]");
    puts("  -m, --max_errors <MAX_ERRORS>");
    puts("          Ignore alignments with more than this many mismatches and indels [default: 10]");
    puts("  -d, --min_depth <MIN_DEPTH>");
    puts("          A base must occur at least this many times in the pileup to be considered valid [default: 5]");
    puts("      --careful");
    puts("          Ignore any reads with multiple alignments");
    puts("  -h, --help");
    puts("          Print help");
    puts("  -V, --version");
    puts("          Print version");
    puts("\nB200 build, additive options: --device <N> (first GPU, default 0), --gpus <N> (contigs shard over N GPUs), --quiet, --host-parse");
    puts("Alignment files may also be BAM (recognised by content, not by name)");
}

// clap accepts `--name=value`, `-m5` / `-m=5` and a `--` separator (everything after it is positional): normalise those forms
// into separate tokens.  `value_shorts` = the short options that take a value.
struct Token { std::string text; bool positional; };
static std::vector<Token> normalise_args(int argc, char** argv, int first, const char* value_shorts) {
    std::vector<Token> out;
    bool rest = false;
    for (int i = first; i < argc; ++i) {
        const std::string a = argv[i];
        if (rest) { out.push_back({a, true}); continue; }
        if (a == "--") { rest = true; continue; }
        if (a.size() > 2 && a[0] == '-' && a[1] == '-') {
            const size_t eq = a.find('=');
            if (eq != std::string::npos) { out.push_back({a.substr(0, eq), false}); out.push_back({a.substr(eq + 1), true}); continue; }
        } else if (a.size() > 2 && a[0] == '-' && a[1] != '-' && strchr(value_shorts, a[1])) {
            out.push_back({a.substr(0, 2), false});
            out.push_back({a.substr(a[2] == '=' ? 3 : 2), true});
            continue;
        }
        out.push_back({a, false});
    }
    return out;
}

static double parse_f64(const char* flag, const char* s) {
    char* end = nullptr;
    double v = strtod(s, &end);
    if (!s[0] || (end && *end)) usage_error(std::string("invalid value '") + s + "' for '" + flag + "': invalid float literal");
    return v;
}
static uint32_t parse_u32(const char* flag, const char* s) {
    char* end = nullptr;
    if (s[0] == '-') usage_error(std::string("invalid value '") + s + "' for '" + flag + "': invalid digit found in string");
    unsigned long long v = strtoull(s, &end, 10);
    if (!s[0] || (end && *end) || v > 0xFFFFFFFFull) usage_error(std::string("invalid value '") + s + "' for '" + flag + "'");
    return (uint32_t)v;
}

// A one-shot process pays CUDA's start-up for every GPU the driver shows it (about a second on an 8-GPU box).  Before the first
// CUDA call the process is therefore narrowed to the GPUs it will use: CUDA_VISIBLE_DEVICES = entries [device, device + gpus) of
// the caller's own list (or of 0, 1, 2, ... when the variable is not set).  Inside the process the devices are then 0 .. gpus-1.
static bool restrict_visible_devices(int device, int gpus) {   // true: the chosen GPUs are now devices 0 .. gpus-1 of this process
    std::vector<std::string> ids;
    if (const char* cur = getenv("CUDA_VISIBLE_DEVICES")) {
        std::string s = cur, item;
        for (size_t i = 0; i <= s.size(); ++i) {
            if (i == s.size() || s[i] == ',') { if (!item.empty()) ids.push_back(item); item.clear(); }
            else item += s[i];
        }
        if ((int)ids.size() < device + gpus) return false;    // not enough entries: leave it to pp_create to report
    } else {
        for (int i = 0; i < device + gpus; ++i) ids.push_back(std::to_string(i));
    }
    std::string v;
    for (int i = device; i < device + gpus; ++i) { if (!v.empty()) v += ','; v += ids[(size_t)i]; }
    return setenv("CUDA_VISIBLE_DEVICES", v.c_str(), 1) == 0;
}

// POLYPOLISH_TIMING=1: wall-clock marks on stderr (process start-up vs the command itself)
static void mark(const char* what) {
    static const auto t0 = std::chrono::steady_clock::now();
    static const bool on = getenv("POLYPOLISH_TIMING") != nullptr;
    if (on) fprintf(stderr, "[timing] %8.1f ms  %s\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(), what);
}

// The value after the option at tok[i] (which then points at the value).
static const char* need(const std::vector<Token>& tok, size_t& i, const char* flag) {
    if (i + 1 >= tok.size()) usage_error(std::string("a value is required for '") + flag + "' but none was supplied");
    return tok[++i].text.c_str();
}

// The options of `polish` (except --debug and --gpus), `filter` and the additive ones every command takes.  Each parser takes the
// option at tok[i] (and its value) and says whether it was one of its options.
struct FilterArgs { std::string in1, in2, out1, out2, orientation = "auto"; double low = 0.1, high = 99.9; };
struct CommonArgs { int device = 0; bool quiet = false, host_parse = false; };

static bool polish_option(const std::vector<Token>& tok, size_t& i, pp_polish_params& prm) {
    const std::string& a = tok[i].text;
    if (a == "-i" || a == "--fraction_invalid") prm.fraction_invalid = parse_f64("--fraction_invalid <FRACTION_INVALID>", need(tok, i, "--fraction_invalid"));
    else if (a == "-v" || a == "--fraction_valid") prm.fraction_valid = parse_f64("--fraction_valid <FRACTION_VALID>", need(tok, i, "--fraction_valid"));
    else if (a == "-m" || a == "--max_errors") prm.max_errors = parse_u32("--max_errors <MAX_ERRORS>", need(tok, i, "--max_errors"));
    else if (a == "-d" || a == "--min_depth") prm.min_depth = parse_u32("--min_depth <MIN_DEPTH>", need(tok, i, "--min_depth"));
    else if (a == "--careful") prm.careful = 1;
    else return false;
    return true;
}

static bool filter_option(const std::vector<Token>& tok, size_t& i, FilterArgs& f) {
    const std::string& a = tok[i].text;
    if (a == "--in1") f.in1 = need(tok, i, "--in1 <IN1>");
    else if (a == "--in2") f.in2 = need(tok, i, "--in2 <IN2>");
    else if (a == "--out1") f.out1 = need(tok, i, "--out1 <OUT1>");
    else if (a == "--out2") f.out2 = need(tok, i, "--out2 <OUT2>");
    else if (a == "--orientation") f.orientation = need(tok, i, "--orientation <ORIENTATION>");
    else if (a == "--low") f.low = parse_f64("--low <LOW>", need(tok, i, "--low"));
    else if (a == "--high") f.high = parse_f64("--high <HIGH>", need(tok, i, "--high"));
    else return false;
    return true;
}

static bool common_option(const std::vector<Token>& tok, size_t& i, CommonArgs& c) {
    const std::string& a = tok[i].text;
    if (a == "--device") c.device = (int)parse_u32("--device", need(tok, i, "--device"));
    else if (a == "--quiet") c.quiet = true;
    else if (a == "--host-parse") c.host_parse = true;
    else return false;
    return true;
}

// A token that is no option of the command: an error when it looks like an option, else a positional argument.
static void positional(const std::string& a, std::vector<std::string>& pos) {
    if (a.size() > 1 && a[0] == '-' && a != "-") usage_error("unexpected argument '" + a + "' found");
    pos.push_back(a);
}

// Contexts on `gpus` GPUs from c.device on; the process exits when there is no usable one.
static std::vector<pp_ctx*> create_contexts(const CommonArgs& c, int gpus) {
    const int base = restrict_visible_devices(c.device, gpus) ? 0 : c.device;
    std::vector<pp_ctx*> ctxs(gpus, nullptr);
    for (int g = 0; g < gpus; ++g)
        if (pp_create(base + g, &ctxs[g]) != PP_OK) quit_with_error("no usable Blackwell (sm_100) GPU: this build has no CPU fallback");
    if (c.host_parse) pp_set_parser(ctxs[0], 1);
    return ctxs;
}

static void check(int rc, const std::vector<pp_ctx*>& ctxs) {
    if (rc == PP_OK) return;
    std::string m = pp_last_error(ctxs[0]);
    for (auto c : ctxs) pp_destroy(c);
    quit_with_error(m);
}

int main(int argc, char** argv) {
    mark("main");
    if (argc < 2) { help(); return 2; }
    std::string cmd = argv[1];
    if (cmd == "-h" || cmd == "--help") { help(); return 0; }
    if (cmd == "-V" || cmd == "--version") { puts("Polypolish v0.6.1"); return 0; }
    CommonArgs common;
    if (cmd == "polish") {
        pp_polish_params prm{0.2, 0.5, 10, 5, 0};
        std::string debug;
        int gpus = 1;
        std::vector<std::string> pos;
        const std::vector<Token> tok = normalise_args(argc, argv, 2, "ivmd");
        for (size_t i = 0; i < tok.size(); ++i) {
            const std::string& a = tok[i].text;
            if (tok[i].positional) { pos.push_back(a); continue; }
            if (a == "-h" || a == "--help") { help_polish(); return 0; }
            else if (a == "-V" || a == "--version") { puts("Polypolish-polish v0.6.1"); return 0; }
            else if (a == "--debug") debug = need(tok, i, "--debug <DEBUG>");
            else if (a == "--gpus") gpus = (int)parse_u32("--gpus", need(tok, i, "--gpus"));
            else if (!polish_option(tok, i, prm) && !common_option(tok, i, common)) positional(a, pos);
        }
        if (pos.empty()) usage_error("the following required arguments were not provided:\n  <ASSEMBLY>");
        if (gpus < 1) gpus = 1;
        const std::vector<pp_ctx*> ctxs = create_contexts(common, gpus);
        mark("contexts created");
        std::vector<const char*> sams;
        for (size_t i = 1; i < pos.size(); ++i) sams.push_back(pos[i].c_str());
        char* out = nullptr;
        uint64_t n = 0;
        if (!common.quiet) fprintf(stderr, "Starting Polypolish polish (B200 build %s, %d GPU%s)\n\n", pp_version(), gpus, gpus > 1 ? "s" : "");
        check(pp_polish_files_multi(ctxs.data(), gpus, pos[0].c_str(), sams.data(), (int)sams.size(), &prm, debug.empty() ? nullptr : debug.c_str(),
                                    &out, &n, common.quiet ? 0 : 1), ctxs);
        mark("polished");
        fwrite(out, 1, n, stdout);
        if (!common.quiet) fprintf(stderr, "Finished!\n");
        mark("output written");
        // A one-shot process has nothing left to do: the contexts, the driver's tear-down and the runtime's static destructors
        // (30 - 1000 ms on these boxes) are skipped - the kernel reclaims everything.  Output files first.
        if (fflush(stdout) != 0 || ferror(stdout)) quit_with_error("unable to write to stdout");
        fflush(stderr);
        _exit(0);
    }
    if (cmd == "filter") {
        FilterArgs f;
        const std::vector<Token> tok = normalise_args(argc, argv, 2, "");
        for (size_t i = 0; i < tok.size(); ++i) {
            const std::string& a = tok[i].text;
            if (tok[i].positional) usage_error("unexpected argument '" + a + "' found");
            if (a == "-h" || a == "--help") { help_filter(); return 0; }
            else if (a == "-V" || a == "--version") { puts("Polypolish-filter v0.6.1"); return 0; }
            else if (!filter_option(tok, i, f) && !common_option(tok, i, common)) usage_error("unexpected argument '" + a + "' found");
        }
        if (f.in1.empty() || f.in2.empty() || f.out1.empty() || f.out2.empty())
            usage_error("the following required arguments were not provided:\n  --in1 <IN1>\n  --in2 <IN2>\n  --out1 <OUT1>\n  --out2 <OUT2>");
        const std::vector<pp_ctx*> ctxs = create_contexts(common, 1);
        if (!common.quiet) fprintf(stderr, "Starting Polypolish filter (B200 build %s)\n\n", pp_version());
        check(pp_filter_files(ctxs[0], f.in1.c_str(), f.in2.c_str(), f.out1.c_str(), f.out2.c_str(), f.orientation.c_str(), f.low, f.high,
                              common.quiet ? 0 : 1), ctxs);
        if (!common.quiet) fprintf(stderr, "Finished!\n");
        fflush(stderr);
        _exit(0);                                           // (see `polish`: nothing left to do, the tear-down is skipped)
    }
    if (cmd == "filter-polish") {
        // ADDITIVE (not in the reference): `filter` and `polish` of its output as one command, no intermediate files unless named
        pp_polish_params prm{0.2, 0.5, 10, 5, 0};
        FilterArgs f;
        std::vector<std::string> pos;
        const std::vector<Token> tok = normalise_args(argc, argv, 2, "ivmd");
        for (size_t i = 0; i < tok.size(); ++i) {
            const std::string& a = tok[i].text;
            if (tok[i].positional) { pos.push_back(a); continue; }
            if (a == "-h" || a == "--help") {
                puts("filter paired-end alignments based on insert size, then polish the assembly with the filtered alignments (one pass, B200 build only)\n");
                puts("Usage: polypolish filter-polish [OPTIONS] --in1 <IN1> --in2 <IN2> <ASSEMBLY>\n");
                puts("Options: those of `filter` (--out1 / --out2 optional: written only when given) and of `polish` (except --debug)");
                return 0;
            }
            else if (!filter_option(tok, i, f) && !polish_option(tok, i, prm) && !common_option(tok, i, common)) positional(a, pos);
        }
        if (f.in1.empty() || f.in2.empty() || pos.size() != 1)
            usage_error("the following required arguments were not provided:\n  --in1 <IN1>\n  --in2 <IN2>\n  <ASSEMBLY>");
        const std::vector<pp_ctx*> ctxs = create_contexts(common, 1);
        if (!common.quiet) fprintf(stderr, "Starting Polypolish filter + polish (B200 build %s)\n\n", pp_version());
        char* out = nullptr;
        uint64_t n = 0;
        check(pp_filter_polish_files(ctxs[0], pos[0].c_str(), f.in1.c_str(), f.in2.c_str(), f.out1.empty() ? nullptr : f.out1.c_str(),
                                     f.out2.empty() ? nullptr : f.out2.c_str(), f.orientation.c_str(), f.low, f.high, &prm, &out, &n,
                                     common.quiet ? 0 : 1), ctxs);
        fwrite(out, 1, n, stdout);
        if (!common.quiet) fprintf(stderr, "Finished!\n");
        if (fflush(stdout) != 0 || ferror(stdout)) quit_with_error("unable to write to stdout");
        fflush(stderr);
        _exit(0);
    }
    usage_error("unrecognized subcommand '" + cmd + "'");
}
