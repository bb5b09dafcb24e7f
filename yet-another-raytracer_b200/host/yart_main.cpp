// yart_main.cpp -- the reference's command line as a native host program on the C ABI (include/yart.h only).
//
// The reference is a compiled binary: `raytracer --scene david [--output ..] [--width ..] [--height ..] [--samples ..]
// [--max-depth ..] [--workers ..] [--vfov ..] [--aperture ..]` (clap derive `Cli`, main.rs:78-107; main :777-781).  This
// is that front end in C++17 with the same flags, the same option resolution (resolve_render_options /
// resolve_dimensions, main.rs:166-209, through yart_resolve_dimensions), the same value checks (clap's range(1..) and
// parse_positive_usize, main.rs:148-158), the same "<path> rendered in N seconds" line (main.rs:763-767) and a PNG file
// at the end (main.rs:769-774) -- with the tile jobs on a thread pool replaced by yart_render on one or more GPUs.
//
// Additions: --seed S (the reference is OS-seeded), --device D, --gpus N (N GPUs of this box: one host thread per
// context, yart_comm_init + yart_film_reduce = one in-place ncclReduce of the f64 film), --order near|reference,
// --unbiased-light-pick / --russian-roulette / --depth-zero-black / --next-event (better sampling, OFF by default), --assets DIR,
// --dry-run (print the resolved options as one JSON line and exit: what the reference's unit tests check,
// main.rs:868-915), --list-scenes.  `--workers` is accepted and ignored.  There is no CPU mode.
//
// build (build.py does this): g++ -std=c++17 -O2 -Iinclude host/yart_main.cpp -o yart -L. -lyart_b200 -Wl,-rpath,'$ORIGIN' -pthread
#include <algorithm>
#include <cerrno>
#include <chrono>
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <string>
#include <thread>
#include <vector>

#include "yart.h"

namespace {

// ---------------------------------------------------------------------------------------------------------
// a minimal PNG encoder (RGBA8, zlib "stored" blocks): the reference saves through the `image` crate (main.rs:774);
// any decoder reads this file, and no third-party library is needed on the host side
// ---------------------------------------------------------------------------------------------------------
uint32_t crc32_of(const uint8_t* p, size_t n, uint32_t crc = 0) {
  static uint32_t table[256];
  static bool ready = false;
  if (!ready) {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c & 1u) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
      table[i] = c;
    }
    ready = true;
  }
  crc = ~crc;
  for (size_t i = 0; i < n; ++i) crc = table[(crc ^ p[i]) & 0xFFu] ^ (crc >> 8);
  return ~crc;
}
void put_u32(std::vector<uint8_t>& v, uint32_t x) {
  for (int s = 24; s >= 0; s -= 8) v.push_back((uint8_t)(x >> s));
}
void put_chunk(std::vector<uint8_t>& out, const char type[4], const std::vector<uint8_t>& data) {
  put_u32(out, (uint32_t)data.size());
  std::vector<uint8_t> body(type, type + 4);
  body.insert(body.end(), data.begin(), data.end());
  out.insert(out.end(), body.begin(), body.end());
  put_u32(out, crc32_of(body.data(), body.size()));
}
bool write_png(const std::string& path, const uint8_t* rgba, uint32_t w, uint32_t h) {
  std::vector<uint8_t> raw; // filter byte 0 + the row
  raw.reserve((size_t)h * (1 + (size_t)w * 4));
  for (uint32_t y = 0; y < h; ++y) {
    raw.push_back(0);
    raw.insert(raw.end(), rgba + (size_t)y * w * 4, rgba + (size_t)(y + 1) * w * 4);
  }
  std::vector<uint8_t> z = {0x78, 0x01}; // zlib header, no compression
  uint32_t a = 1, b = 0;                 // Adler-32
  size_t off = 0;
  do { // stored blocks of at most 65535 bytes: BFINAL, LEN, ~LEN, data
    const size_t n = std::min<size_t>(65535, raw.size() - off);
    z.push_back(off + n == raw.size() ? 1 : 0);
    z.push_back((uint8_t)(n & 0xFF));
    z.push_back((uint8_t)(n >> 8));
    z.push_back((uint8_t)(~n & 0xFF));
    z.push_back((uint8_t)((~n >> 8) & 0xFF));
    z.insert(z.end(), raw.begin() + (long)off, raw.begin() + (long)(off + n));
    for (size_t i = off; i < off + n; ++i) {
      a = (a + raw[i]) % 65521u;
      b = (b + a) % 65521u;
    }
    off += n;
  } while (off < raw.size());
  put_u32(z, (b << 16) | a);
  std::vector<uint8_t> out = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1A, '\n'};
  std::vector<uint8_t> ihdr;
  put_u32(ihdr, w);
  put_u32(ihdr, h);
  const uint8_t tail[5] = {8, 6, 0, 0, 0}; // 8 bits, RGBA, deflate, no filter method, no interlace
  ihdr.insert(ihdr.end(), tail, tail + 5);
  put_chunk(out, "IHDR", ihdr);
  put_chunk(out, "IDAT", z);
  put_chunk(out, "IEND", {});
  FILE* f = fopen(path.c_str(), "wb");
  if (!f) return false;
  const bool ok = fwrite(out.data(), 1, out.size(), f) == out.size();
  return fclose(f) == 0 && ok;
}

// ---------------------------------------------------------------------------------------------------------
// command line (clap's behaviour where the reference's tests pin it: main.rs:831-842)
// ---------------------------------------------------------------------------------------------------------
struct Cli {
  std::string scene, output, assets = "assets/_unpacked", order = "near";
  uint32_t width = 0, height = 0, samples = 0, max_depth = 0, workers = 0; // 0 = not given
  double vfov = -1.0, aperture = -1.0;                                      // < 0 = not given
  bool have_vfov = false, have_aperture = false;
  uint64_t seed = 1;
  int device = 0, gpus = 1;
  uint32_t flags = 0;
  bool dry_run = false, list_scenes = false;
};

[[noreturn]] void usage_error(const std::string& msg) { // clap exits with status 2 on a usage error
  fprintf(stderr, "error: %s\n\nUsage: yart --scene <SCENE> [--output <OUTPUT>] [--width <WIDTH>] [--height <HEIGHT>] "
                  "[--samples <SAMPLES>] [--max-depth <MAX_DEPTH>] [--workers <WORKERS>] [--vfov <VFOV>] [--aperture <APERTURE>]\n"
                  "            [--seed S] [--device D] [--gpus N] [--order near|reference] [--assets DIR] [--dry-run] [--list-scenes]\n"
                  "            [--unbiased-light-pick] [--russian-roulette] [--depth-zero-black] [--next-event]\n",
          msg.c_str());
  exit(2);
}

uint32_t positive(const char* flag, const std::string& text) { // parse_positive_usize (main.rs:148-158) / range(1..)
  char* end = nullptr;
  errno = 0;
  const unsigned long long v = strtoull(text.c_str(), &end, 10);
  if (text.empty() || *end != '\0' || text[0] == '-' || text[0] == '+' || errno != 0 || v > 0xFFFFFFFFull)
    usage_error("invalid value '" + text + "' for '" + flag + "': invalid integer `" + text + "`");
  if (v == 0) usage_error("invalid value '" + text + "' for '" + flag + "': value must be greater than 0");
  return (uint32_t)v;
}
double real(const char* flag, const std::string& text) {
  char* end = nullptr;
  const double v = strtod(text.c_str(), &end);
  if (text.empty() || *end != '\0') usage_error("invalid value '" + text + "' for '" + flag + "': invalid float literal");
  return v;
}

Cli parse(int argc, char** argv) {
  Cli c;
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i], val;
    bool inline_val = false;
    const size_t eq = a.find('=');
    if (a.rfind("--", 0) == 0 && eq != std::string::npos) { // --flag=value
      val = a.substr(eq + 1);
      a = a.substr(0, eq);
      inline_val = true;
    }
    auto value = [&]() -> std::string {
      if (inline_val) return val;
      if (i + 1 >= argc) usage_error("a value is required for '" + a + "' but none was supplied");
      return argv[++i];
    };
    if (a == "--scene") c.scene = value();
    else if (a == "--output") c.output = value();
    else if (a == "--width") c.width = positive("--width", value());
    else if (a == "--height") c.height = positive("--height", value());
    else if (a == "--samples") c.samples = positive("--samples", value());
    else if (a == "--max-depth") c.max_depth = positive("--max-depth", value());
    else if (a == "--workers") c.workers = positive("--workers", value());
    else if (a == "--vfov") { c.vfov = real("--vfov", value()); c.have_vfov = true; }
    else if (a == "--aperture") { c.aperture = real("--aperture", value()); c.have_aperture = true; }
    else if (a == "--seed") c.seed = strtoull(value().c_str(), nullptr, 10);
    else if (a == "--device") c.device = atoi(value().c_str());
    else if (a == "--gpus") c.gpus = (int)positive("--gpus", value());
    else if (a == "--order") c.order = value();
    else if (a == "--assets") c.assets = value();
    else if (a == "--unbiased-light-pick") c.flags |= YART_FLAG_UNBIASED_LIGHT_PICK;
    else if (a == "--russian-roulette") c.flags |= YART_FLAG_RUSSIAN_ROULETTE;
    else if (a == "--depth-zero-black") c.flags |= YART_FLAG_DEPTH_ZERO_BLACK;
    else if (a == "--next-event") c.flags |= YART_FLAG_NEXT_EVENT;
    else if (a == "--dry-run") c.dry_run = true;
    else if (a == "--list-scenes") c.list_scenes = true;
    else if (a == "--help" || a == "-h") {
      printf("Render predefined raytracer scenes (B200; the reference's flags, see the header of host/yart_main.cpp)\n");
      exit(0);
    } else usage_error("unexpected argument '" + a + "' found");
  }
  if (c.list_scenes) return c;
  if (c.scene.empty()) usage_error("the following required arguments were not provided:\n  --scene <SCENE>");
  bool known = false;
  std::string all;
  for (int k = 0; k < yart_preset_count(); ++k) {
    known = known || c.scene == yart_preset_name(k);
    all += std::string(k ? ", " : "") + yart_preset_name(k);
  }
  if (!known) usage_error("invalid value '" + c.scene + "' for '--scene <SCENE>'\n  [possible values: " + all + "]");
  if (c.order != "near" && c.order != "reference") usage_error("invalid value '" + c.order + "' for '--order'");
  return c;
}

int die(const char* what, const yart_ctx* ctx) {
  fprintf(stderr, "yart: %s: %s\n", what, ctx ? yart_last_error(ctx) : yart_last_error_global());
  return 1;
}

} // namespace

int main(int argc, char** argv) {
  const Cli cli = parse(argc, argv);
  if (cli.list_scenes) {
    for (int k = 0; k < yart_preset_count(); ++k) printf("%s\n", yart_preset_name(k));
    return 0;
  }
  // resolve_render_config (main.rs:434-446): preset, then the option overrides
  yart_preset* preset = nullptr;
  if (yart_preset_build(cli.scene.c_str(), cli.assets.c_str(), cli.seed, &preset) != YART_OK) return die("yart_preset_build", nullptr);
  if (*yart_preset_note(preset)) fprintf(stderr, "note: %s\n", yart_preset_note(preset));
  yart_preset_info pi;
  yart_preset_get_info(preset, &pi);
  uint32_t width = 0, height = 0;
  yart_resolve_dimensions(pi.width, pi.height, cli.width, cli.height, &width, &height);
  const uint32_t spp = cli.samples ? cli.samples : pi.samples_per_pixel;
  const uint32_t max_depth = cli.max_depth ? cli.max_depth : pi.max_depth;
  const uint32_t workers = cli.workers ? cli.workers : pi.workers;
  const double vfov = cli.have_vfov ? cli.vfov : pi.vfov, aperture = cli.have_aperture ? cli.aperture : pi.aperture;
  const std::string output = !cli.output.empty() ? cli.output : (std::filesystem::path("output") / pi.output_filename).string();
  if (cli.dry_run) { // RenderOptions (main.rs:122-132) as data
    printf("{\"output_path\": \"%s\", \"width\": %u, \"height\": %u, \"samples_per_pixel\": %u, \"max_depth\": %u, \"workers\": %u, "
           "\"vfov\": %.17g, \"aperture\": %.17g}\n", output.c_str(), width, height, spp, max_depth, workers, vfov, aperture);
    yart_preset_free(preset);
    return 0;
  }
  yart_camera cam; // render()'s camera (main.rs:605-625); a negative vfov / aperture cannot mean "default" here
  yart_preset_camera(preset, width, height, -1.0, -1.0, &cam);
  cam.vfov_degrees = vfov;
  cam.aperture = aperture;

  const auto start = std::chrono::steady_clock::now(); // the reference's timer starts in render() (main.rs:591)
  const int n = cli.gpus;
  if (cli.device < 0 || cli.device + n > yart_device_count()) {
    fprintf(stderr, "yart: --device %d --gpus %d: %d GPU(s) visible (there is no CPU mode)\n", cli.device, n, yart_device_count());
    return 1;
  }
  std::vector<yart_ctx*> ctxs(n, nullptr);
  std::vector<double*> films(n, nullptr);
  std::vector<yart_stats> stats(n);
  std::vector<int> rcs(n, YART_OK);
  for (int r = 0; r < n; ++r)
    if (yart_ctx_create(cli.device + r, &ctxs[r]) != YART_OK) return die("yart_ctx_create (no CPU fallback)", nullptr);
  yart_comm* comm = nullptr;
  if (n > 1 && yart_comm_init(ctxs.data(), n, &comm) != YART_OK) return die("yart_comm_init", nullptr);

  auto shard = [&](int r, uint32_t& lo, uint32_t& hi) { // contiguous, balanced sample ranges (sizes differ by <= 1)
    const uint32_t base = spp / (uint32_t)n, extra = spp % (uint32_t)n;
    lo = (uint32_t)r * base + std::min<uint32_t>((uint32_t)r, extra);
    hi = lo + base + ((uint32_t)r < extra ? 1u : 0u);
  };
  auto work = [&](int r) { // one host thread per context: scene upload (QBVH build on its GPU) + its sample range
    yart_ctx* ctx = ctxs[r];
    if ((rcs[r] = yart_ctx_set_scene(ctx, yart_preset_scene(preset))) != YART_OK) return;
    if ((rcs[r] = yart_film_create(ctx, width, height, &films[r])) != YART_OK) return;
    yart_render_opts o;
    memset(&o, 0, sizeof o);
    o.width = width;
    o.height = height;
    shard(r, o.sample_begin, o.sample_end);
    o.max_depth = max_depth;
    o.order = cli.order == "near" ? YART_ORDER_NEAR : YART_ORDER_REFERENCE;
    o.flags = YART_FLAG_DEVICE_PTRS | cli.flags;
    o.seed = cli.seed;
    memset(&stats[r], 0, sizeof(yart_stats));
    if (o.sample_end > o.sample_begin) rcs[r] = yart_render(ctx, &cam, &o, films[r], &stats[r]);
  };
  if (n == 1) {
    work(0);
  } else {
    std::vector<std::thread> threads;
    for (int r = 0; r < n; ++r) threads.emplace_back(work, r);
    for (auto& t : threads) t.join();
  }
  for (int r = 0; r < n; ++r)
    if (rcs[r] != YART_OK) return die("render", ctxs[r]);
  if (comm && yart_film_reduce(comm, films.data(), width, height, 0) != YART_OK) {
    fprintf(stderr, "yart: yart_film_reduce: %s\n", yart_comm_last_error(comm));
    return 1;
  }
  // finalise on the root GPU (main.rs:710-718) and bring the RGBA8 image home
  std::vector<double> film((size_t)width * height * 3);
  std::vector<uint8_t> rgba((size_t)width * height * 4);
  if (yart_film_read(ctxs[0], films[0], width, height, film.data()) != YART_OK) return die("yart_film_read", ctxs[0]);
  if (yart_film_finalize(ctxs[0], film.data(), width, height, spp, 0, rgba.data()) != YART_OK) return die("yart_film_finalize", ctxs[0]);

  const auto secs = std::chrono::duration_cast<std::chrono::seconds>(std::chrono::steady_clock::now() - start).count();
  printf("%s rendered in %lld seconds\n", output.c_str(), (long long)secs); // main.rs:763-767
  uint64_t rays = 0, paths = 0;
  double ms = 0.0;
  for (const yart_stats& s : stats) {
    rays += s.rays;
    paths += s.paths;
    ms = std::max(ms, s.gpu_ms);
  }
  printf("  %" PRIu64 " paths, %" PRIu64 " rays, %.1f Mrays/s on %d GPU(s)\n", paths, rays, ms > 0 ? (double)rays / ms / 1e3 : 0.0, n);
  const std::filesystem::path parent = std::filesystem::path(output).parent_path(); // main.rs:769-773
  std::error_code ec;
  if (!parent.empty()) std::filesystem::create_directories(parent, ec);
  if (!write_png(output, rgba.data(), width, height)) {
    fprintf(stderr, "yart: cannot write %s\n", output.c_str());
    return 1;
  }
  if (comm) yart_comm_destroy(comm);
  for (int r = 0; r < n; ++r) {
    yart_film_destroy(ctxs[r], films[r]);
    yart_ctx_destroy(ctxs[r]);
  }
  yart_preset_free(preset);
  return 0;
}
