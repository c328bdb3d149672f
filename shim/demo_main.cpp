// demo_main.cpp -- the reference's start-up sequence (main.cpp:94-108) without the window: load the scene with the
// reference's own MeshS/Material code, build form factors and converge the lighting through the shim classes.
//   shim_demo <scene.obj> <mtl_dir/> <method 0|1|2> <emission_value> <seed> [rands.bin] [matrix cache file]   (cwd must hold color_tables/srgb.coeff)
// Prints one line of results the parity test compares with the Python path.
#include <chrono>
#include <cstdio>
#include <cstring>
#include <vector>
#define TINYOBJLOADER_IMPLEMENTATION
#include <tiny_obj_loader.h>
#undef TINYOBJLOADER_IMPLEMENTATION
#include "OptixPrimeFunctionality.h"
#include "Lightning.h"
#include "Camera.h" // reference header, unchanged: gen_rays_for_screen (Camera.h:54-80)

// headless stand-ins for Drawer::RenderContext / Drawer::DebugLine (Drawer.h:36-63 drags in GLFW / GLEW): same member names,
// so the shim's traceScreen / intersectMouse templates take either
struct HeadlessRenderContext {
    std::vector<std::vector<MatrixIndex>> &trianglesonScreen;
    Lightning &lightning;
    std::vector<glm::vec3> &optixView;
    MeshS &mesh;
    Camera &camera;
    bool &radiosityRendering;
    bool &antialiasing;
    int supersampling;
};
struct HeadlessDebugLine { bool left = true; std::vector<int> debugtriangles; };

// 8-bit RGB PNG with stored (uncompressed) deflate blocks: what the reference's `i` key saves through ImageExporter, minus
// the OpenGL read-back.  Bottom row first, like glReadPixels.
static void write_png(const char *path, const std::vector<glm::vec3> &img, int w, int h) {
    std::vector<unsigned char> raw;
    for (int y = h - 1; y >= 0; y--) {
        raw.push_back(0);
        for (int x = 0; x < w; x++)
            for (int c = 0; c < 3; c++) raw.push_back((unsigned char)(std::min(1.f, std::max(0.f, img[(size_t)y * w + x][c])) * 255.f + 0.5f));
    }
    auto crc = [](const std::vector<unsigned char> &d) {
        unsigned c = 0xffffffffu;
        for (unsigned char b : d) { c ^= b; for (int k = 0; k < 8; k++) c = (c >> 1) ^ (0xedb88320u & (0u - (c & 1u))); }
        return c ^ 0xffffffffu;
    };
    auto be32 = [](std::vector<unsigned char> &v, unsigned x) { for (int s = 24; s >= 0; s -= 8) v.push_back((unsigned char)(x >> s)); };
    FILE *f = fopen(path, "wb");
    if (!f) return;
    auto chunk = [&](const char *tag, const std::vector<unsigned char> &data) {
        std::vector<unsigned char> td(tag, tag + 4), len;
        td.insert(td.end(), data.begin(), data.end());
        be32(len, (unsigned)data.size());
        fwrite(len.data(), 1, 4, f);
        fwrite(td.data(), 1, td.size(), f);
        std::vector<unsigned char> c;
        be32(c, crc(td));
        fwrite(c.data(), 1, 4, f);
    };
    fwrite("\x89PNG\r\n\x1a\n", 1, 8, f);
    std::vector<unsigned char> ihdr;
    be32(ihdr, (unsigned)w); be32(ihdr, (unsigned)h);
    const unsigned char tail[5] = { 8, 2, 0, 0, 0 };
    ihdr.insert(ihdr.end(), tail, tail + 5);
    chunk("IHDR", ihdr);
    std::vector<unsigned char> z = { 0x78, 0x01 };
    unsigned a = 1, b = 0;
    for (unsigned char v : raw) { a = (a + v) % 65521u; b = (b + a) % 65521u; }
    for (size_t off = 0; off < raw.size(); off += 65535) {
        const size_t n = std::min<size_t>(65535, raw.size() - off);
        z.push_back(off + n == raw.size() ? 1 : 0);
        z.push_back((unsigned char)(n & 255)); z.push_back((unsigned char)(n >> 8));
        z.push_back((unsigned char)(~n & 255)); z.push_back((unsigned char)((~n >> 8) & 255));
        z.insert(z.end(), raw.begin() + off, raw.begin() + off + n);
    }
    be32(z, (b << 16) | a);
    chunk("IDAT", z);
    chunk("IEND", {});
    fclose(f);
}

int main(int argc, char **argv) {
    if (argc < 6) { fprintf(stderr, "usage: shim_demo scene.obj mtl_dir/ method emission seed\n"); return 2; }
    std::vector<float> wavelengths = { 200.0, 250.0, 300.0, 350.0, 400.0, 450.0, 500.0, 550.0, 600.0 }; // main.cpp:94
    MeshS mesh(argv[1], argv[2], wavelengths);
    for (auto &m : mesh.materials) // the UV lamp's M is undefined behaviour in the reference (Material.cpp:52-54): use M = 0
        if (m.spectral_values.size() && m.spectral_values[0] == 0.0f && m.spectral_values.back() == 0.0f && m.rgbcolor == glm::vec3(0.f))
            m.M.setZero();
    const int ndev = getenv("DAISY_DEMO_NDEV") ? atoi(getenv("DAISY_DEMO_NDEV")) : 1; // GPUs behind this one process
    OptixPrimeFunctionality optixP(mesh, 0, atol(argv[5]), ndev);
    if (argc > 6) { // optional: a binary file of S x {u,v} floats replaces the rand() pattern (repeatable across C runtimes)
        std::vector<UV> r(RAYS_PER_PATCH);
        FILE *f = fopen(argv[6], "rb");
        if (f && fread(r.data(), sizeof(UV), r.size(), f) == r.size()) optixP.setSamples(r);
        if (f) fclose(f);
    }
    float emission = (float)atof(argv[4]);
    int method = atoi(argv[3]);
    // large scenes: the matrix has more non-zeros than an Eigen int index holds and lives on the GPUs only
    if (getenv("DAISY_DEMO_NO_REFILL")) optixP.refill_RadMat = false;
    const auto t0 = std::chrono::high_resolution_clock::now();
    Lightning *l = Lightning::get_lightning(method, mesh, optixP, emission, wavelengths, true, argc > 7 ? argv[7] : nullptr); // main.cpp:108 passes matfile
    // DAISY_DEMO_CONVERGE=device: solve again from reset() with the stop rule on the device; the SOLVE line must not change
    const char *conv = getenv("DAISY_DEMO_CONVERGE");
    if (conv && strcmp(conv, "device") == 0) {
        l->reset();
        l->converge_lightning_on_device();
    }
    // DAISY_DEMO_RECONVERGE=1: one warm restart from the converged values (reconverge_lightning); RESTART reports its passes
    if (getenv("DAISY_DEMO_RECONVERGE")) {
        l->reconverge_lightning();
        double sr = 0;
        for (auto &band : l->lightningvalues) for (float v : band) sr += v;
        printf("RESTART passes=%d sumB=%.9e\n", l->numpasses, sr);
    }
    const double solve_s = std::chrono::duration<double>(std::chrono::high_resolution_clock::now() - t0).count();
    double sum = 0;
    for (auto &band : l->lightningvalues) for (float v : band) sum += v;
    glm::vec3 c = l->get_color_of_patch(mesh.numtriangles / 2);
    printf("SOLVE patches=%d gpus=%d passes=%d sumB=%.9e seconds=%.3f (form factors + converge_lightning, Lightning::get_lightning)\n", mesh.numtriangles, ndev,
           l->numpasses, sum, solve_s);
    if (getenv("DAISY_DEMO_SOLVE_ONLY")) { delete l; return 0; }
    // the batched visibility entry point on its own (OptixPrimeFunctionality.cpp:169-242): count and sum of the triplets
    std::vector<parallellism::Tripl> unoccluded;
    std::vector<Eigen::Triplet<double>> tr = optixP.calculateAllVisibility(unoccluded, mesh, optixP.rands);
    double tsum = 0;
    for (auto &t : tr) tsum += t.value();
    // the per-pair debugging entry points (InputHandler.cpp:184, OptixPrimeFunctionality.cpp:456-469) on two fixed patches
    const int pa = 3, pb = mesh.numtriangles / 2 + 5;
    float nus = optixP.p2pFormfactorNusselt(pa, pb, mesh), p2p = optixP.p2pFormfactor(pa, pb, mesh);
    std::vector<optix_functionality::Hit> picks(2);
    picks[0].t = 1; picks[0].triangleId = pa; picks[0].uv.x = 0.25f; picks[0].uv.y = 0.5f;
    picks[1].t = 1; picks[1].triangleId = pb; picks[1].uv.x = 0.3f; picks[1].uv.y = 0.3f;
    bool shot = optixP.shootPatchRay(picks, mesh);
    // the step right after the solve (main.cpp:113, Drawer.cpp:200): camera ray cast + interpolated patch colours, and a pick
    double img_sum = 0;
    int pick = -1;
    if (const char *png = getenv("DAISY_DEMO_PNG")) {
        Camera camera(160, 120, 4);
        glm::vec3 lo(1e30f), hi(-1e30f);
        for (auto &v : mesh.vertices) { lo = glm::min(lo, v); hi = glm::max(hi, v); }
        const glm::vec3 mid = 0.5f * (lo + hi);
        camera.dir = optix::make_float3(mid.x, mid.y, mid.z);
        camera.eye = optix::make_float3(mid.x, mid.y, hi.z + 1.6f * (hi.z - lo.z)); // look into the scene along -z
        std::vector<std::vector<MatrixIndex>> trianglesonScreen;
        std::vector<glm::vec3> optixView;
        bool radiosityRendering = true, antiAliasing = true;
        HeadlessRenderContext rc{ trianglesonScreen, *l, optixView, mesh, camera, radiosityRendering, antiAliasing, 4 };
        optixP.traceScreen(rc);
        for (auto &p : optixView) img_sum += p.x + p.y + p.z;
        write_png(png, optixView, camera.pixwidth, camera.pixheight);
        HeadlessDebugLine dl;
        std::vector<optix_functionality::Hit> patches(2);
        optixP.intersectMouse(dl, 80.0, 60.0, camera, trianglesonScreen, optixView, patches, mesh);
        pick = dl.debugtriangles.empty() ? -1 : dl.debugtriangles[0];
        printf("\nIMAGE sum=%.6e pick=%d onscreen=%zu\n", img_sum, pick, trianglesonScreen.size());
    }
    printf("RESULT passes=%d sumB=%.9e color=%.6f,%.6f,%.6f rand0=%.9g tripl=%zu,%.12e nusselt=%.9e p2p=%.9e shoot=%d\n", l->numpasses, sum, c.x,
           c.y, c.z, optixP.rands[0].u, tr.size(), tsum, nus, p2p, shot ? 1 : 0);
    delete l;
    return 0;
}
