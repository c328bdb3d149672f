// Lightning.h -- drop-in replacement of the reference's Lightning family (visual studio/Lightning.h) running the
// gather on the GPU through the C-ABI.  Same factory and virtual interface (get_lightning, get_color_of_patch,
// converge_lightning, increment_lightpass, reset).  Include after OptixPrimeFunctionality.h, like the reference.
#pragma once
#include <cmath>
#include <fstream>
#include <iostream>
#include <vector>
#include "color.h" // reference header, unchanged (cie1931WavelengthToXYZFit, XYZToRGB)

class Lightning {
public:
    static Lightning *get_lightning(int method, MeshS &mesh, OptixPrimeFunctionality &optixP, float &emissionval,
                                    std::vector<float> wavelengthsvec, bool cuda_enabled = false, char *matfile = nullptr);
    virtual glm::vec3 get_color_of_patch(int) = 0;
    virtual void converge_lightning() { // Lightning.h:145-151, :336-340, :410-415
        int passes = 0;
        check(daisy_group_solver_converge(solver, threshold, per_band, 0, &passes));
        numpasses = passes;
        fetch();
    }
    // converge_lightning with the stop rule evaluated by the pass kernels: same passes and bit-identical values, without a host
    // round trip per pass (daisy_group_solver_converge_device)
    void converge_lightning_on_device() {
        int passes = 0;
        check(daisy_group_solver_converge_device(solver, threshold, per_band, 0, &passes));
        numpasses = passes;
        fetch();
    }
    virtual void increment_lightpass() {
        check(daisy_group_solver_step(solver, nullptr));
        numpasses = daisy_group_solver_numpasses(solver);
        fetch();
    }
    virtual void reset() {
        check(daisy_group_solver_reset(solver));
        numpasses = 0;
        fetch();
    }
    // warm restart after the matrix (updateGeometry + updateRadiosityMatrix), the emission or the materials changed: one pass
    // from the current lightningvalues instead of from the emission (daisy_group_solver_restart); numpasses becomes 1
    void restart() {
        check(daisy_group_solver_restart(solver, nullptr));
        numpasses = daisy_group_solver_numpasses(solver);
        fetch();
    }
    // restart + converge_lightning: the stop rule then looks at the sum of |residual| (a warm residual has both signs)
    void reconverge_lightning() {
        check(daisy_group_solver_restart(solver, nullptr));
        converge_lightning();
    }
    virtual ~Lightning() { daisy_group_solver_destroy(solver); }
    int numpasses = 0;
    std::vector<std::vector<float>> lightningvalues, residualvector; // K x N, band-major (Lightning.h:107-109)

protected:
    bool cuda_on = false;
    SpMat RadMat;
    float emission_value = 0;
    daisy_group_solver *solver = nullptr; // one solver per GPU of optixP's group behind one handle
    double threshold = 1e-4;
    int per_band = 1;
    int K = 0, N = 0;

    void initMat(MeshS &mesh, OptixPrimeFunctionality &optixP) { // Lightning.h:75-83
        RadMat = SpMat(mesh.numtriangles, mesh.numtriangles);
        if (cuda_on) optixP.cudaCalculateRadiosityMatrix(RadMat, mesh);
        else optixP.calculateRadiosityMatrix(RadMat, mesh);
    }
    // On-disk cache of the matrix, byte-compatible with the reference (Lightning.h:21-73): five ints (rows, cols, nnz,
    // outerSize, innerSize), then the CSC value array, the outer index array (outerSize ints) and the inner index array.
    // (The reference's reader takes the 4th/5th int in swapped roles; the matrix is square, so both are N.)
    void SerializeMat(SpMat &m, char *matfile) {
        m.makeCompressed();
        std::ofstream f(matfile, std::ios::binary);
        if (!f.is_open()) return;
        const int hdr[5] = { (int)m.rows(), (int)m.cols(), (int)m.nonZeros(), (int)m.outerSize(), (int)m.innerSize() };
        f.write((const char *)hdr, sizeof(hdr));
        f.write((const char *)m.valuePtr(), sizeof(float) * (size_t)m.nonZeros());
        f.write((const char *)m.outerIndexPtr(), sizeof(int) * (size_t)m.outerSize());
        f.write((const char *)m.innerIndexPtr(), sizeof(int) * (size_t)m.nonZeros());
    }
    bool DeserializeMat(SpMat &m, char *matfile) {
        std::ifstream f(matfile, std::ios::binary);
        if (!f.is_open()) return false;
        int hdr[5];
        f.read((char *)hdr, sizeof(hdr));
        const int rows = hdr[0], cols = hdr[1], nnz = hdr[2], outer = hdr[3];
        std::vector<float> val((size_t)nnz);
        std::vector<int> op((size_t)outer + 1), ip((size_t)nnz);
        f.read((char *)val.data(), sizeof(float) * (size_t)nnz);
        f.read((char *)op.data(), sizeof(int) * (size_t)outer);
        f.read((char *)ip.data(), sizeof(int) * (size_t)nnz);
        if (!f) return false;
        op[outer] = nnz; // the file holds outerSize entries, i.e. no closing sentinel
        m.resize(rows, cols);
        m.makeCompressed();
        m.resizeNonZeros(nnz);
        std::copy(val.begin(), val.end(), m.valuePtr());
        std::copy(ip.begin(), ip.end(), m.innerIndexPtr());
        std::copy(op.begin(), op.end(), m.outerIndexPtr());
        return true;
    }
    // the cached matrix goes to the GPUs as it is, CSC arrays only: validated there, then scattered into every device's rows
    // (entries not listed become +0.0, as in a dense load of the same matrix)
    void upload(SpMat &m, OptixPrimeFunctionality &optixP, int n) {
        if (m.rows() != n || m.cols() != n) { // write_csc reads n + 1 column starts: a cache of another mesh is refused here
            std::cerr << "Cached matrix is " << m.rows() << " x " << m.cols() << ", the mesh has " << n << " patches: not loaded" << std::endl;
            return;
        }
        m.makeCompressed();
        check(daisy_group_formfactors_write_csc(optixP.group, (int64_t)m.nonZeros(), m.valuePtr(), m.innerIndexPtr(), m.outerIndexPtr()));
    }
    void initMatFromFile(MeshS &mesh, OptixPrimeFunctionality &optixP, char *matfile) { // Lightning.h:84-96
        RadMat = SpMat(mesh.numtriangles, mesh.numtriangles);
        if (DeserializeMat(RadMat, matfile)) {
            upload(RadMat, optixP, mesh.numtriangles);
            std::cout << "Deserialized matrix" << std::endl;
        } else {
            initMat(mesh, optixP);
            SerializeMat(RadMat, matfile);
            std::cout << "Loaded & Serialized matrix" << std::endl;
        }
    }
    void initMatMaybeCached(MeshS &mesh, OptixPrimeFunctionality &optixP, char *matfile) {
        if (matfile) initMatFromFile(mesh, optixP, matfile); // the reference's main() always takes this path (main.cpp:108)
        else initMat(mesh, optixP);
    }
    void create(MeshS &mesh, OptixPrimeFunctionality &optixP, int K_, const std::vector<float> &E, const std::vector<float> &M) {
        K = K_; N = mesh.numtriangles;
        check(daisy_group_solver_create(optixP.group, K, E.data(), M.data(), (int)mesh.materials.size(), mesh.materialIndexPerTriangle.data(), &solver));
        lightningvalues.assign(K, std::vector<float>(N));
        residualvector.assign(K, std::vector<float>(N));
    }
    void fetch() {
        std::vector<float> B((size_t)K * N), R((size_t)K * N);
        if (!check(daisy_group_solver_read(solver, B.data(), R.data()))) return;
        for (int k = 0; k < K; k++) {
            std::copy(B.begin() + (size_t)k * N, B.begin() + (size_t)(k + 1) * N, lightningvalues[k].begin());
            std::copy(R.begin() + (size_t)k * N, R.begin() + (size_t)(k + 1) * N, residualvector[k].begin());
        }
    }
    static bool check(int rc) {
        if (rc != DAISY_OK) std::cerr << "An error occurred with error code " << rc << " and message " << daisy_last_error() << std::endl;
        return rc == DAISY_OK;
    }
};

class SpectralLightning : public Lightning { // Lightning.h:99-295
public:
    SpectralLightning(MeshS &mesh, OptixPrimeFunctionality &optixP, float &emissionval, std::vector<float> wavelengthsvec,
                      bool cuda_enabled = false, char *matfile = nullptr) {
        cuda_on = cuda_enabled; emission_value = emissionval; threshold = 200; per_band = 0;
        int Kw = (int)wavelengthsvec.size(), Np = mesh.numtriangles, nm = (int)mesh.materials.size();
        for (float w : wavelengthsvec) xyz_per_wavelength.push_back(daisy_color::cie1931WavelengthToXYZFit(w));
        std::vector<float> E((size_t)Kw * Np, 0.f), M((size_t)nm * Kw * Kw);
        for (int i = 0; i < Kw; i++) // set_sampled_emission, :263-273
            for (int j = 0; j < Np; j++) {
                float se = mesh.materials[mesh.materialIndexPerTriangle[j]].spectral_emission[i];
                if (se > 0.0) E[(size_t)i * Np + j] = se * emission_value;
            }
        for (int m = 0; m < nm; m++) // set_reflectionmatrix, :287-292 (one matrix per material instead of per patch)
            std::copy(mesh.materials[m].M.data(), mesh.materials[m].M.data() + Kw * Kw, M.begin() + (size_t)m * Kw * Kw);
        initMatMaybeCached(mesh, optixP, matfile);
        create(mesh, optixP, Kw, E, M);
        reset();
        std::cout << "Lightning has been initialized" << std::endl;
        converge_lightning();
    }
    glm::vec3 get_color_of_patch(int i) override { // update_color_cache, :168-183
        glm::vec3 xyz(0.f);
        for (int j = 0; j < K; j++) xyz += xyz_per_wavelength[j] * lightningvalues[j][i];
        glm::vec3 rgb(0.f);
        daisy_color::XYZToRGB(xyz, rgb);
        float maxval = fmaxf(rgb[0], fmaxf(rgb[1], rgb[2]));
        if (maxval > 1) rgb = { rgb[0] / maxval, rgb[1] / maxval, rgb[2] / maxval };
        return rgb;
    }
private:
    std::vector<glm::vec3> xyz_per_wavelength;
};

class RGBLightning : public Lightning { // Lightning.h:298-384
public:
    RGBLightning(MeshS &mesh, OptixPrimeFunctionality &optixP, float &emissionval, bool cuda_enabled = false, char *matfile = nullptr) {
        cuda_on = cuda_enabled; emission_value = emissionval;
        int Np = mesh.numtriangles, nm = (int)mesh.materials.size();
        std::vector<float> E((size_t)3 * Np, 0.f), M((size_t)nm * 9, 0.f);
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < Np; j++) {
                float e = mesh.materials[mesh.materialIndexPerTriangle[j]].emission[i];
                if (e > 0.0) E[(size_t)i * Np + j] = e * emission_value;
            }
        for (int m = 0; m < nm; m++)
            for (int i = 0; i < 3; i++)
                if (mesh.materials[m].rgbcolor[i] > 0.0) M[(size_t)m * 9 + i * 3 + i] = mesh.materials[m].rgbcolor[i];
        initMatMaybeCached(mesh, optixP, matfile);
        create(mesh, optixP, 3, E, M);
        reset();
        converge_lightning();
    }
    glm::vec3 get_color_of_patch(int i) override { return { lightningvalues[0][i], lightningvalues[1][i], lightningvalues[2][i] }; }
};

class BWLightning : public Lightning { // Lightning.h:386-443
public:
    BWLightning(MeshS &mesh, OptixPrimeFunctionality &optixP, float &emissionval, char *matfile = nullptr) {
        emission_value = emissionval; // cuda_on stays false, as in the reference (:393)
        int Np = mesh.numtriangles, nm = (int)mesh.materials.size();
        std::vector<float> E((size_t)Np, 0.f), M((size_t)nm, 1.f);
        for (int j = 0; j < Np; j++) {
            float e = mesh.materials[mesh.materialIndexPerTriangle[j]].emission[0];
            if (e > 0.0) E[j] = e * emission_value;
        }
        initMatMaybeCached(mesh, optixP, matfile);
        create(mesh, optixP, 1, E, M);
        reset();
        converge_lightning();
        std::cout << "Number of light passes " << numpasses << std::endl;
    }
    glm::vec3 get_color_of_patch(int i) override { return { lightningvalues[0][i], lightningvalues[0][i], lightningvalues[0][i] }; }
};

inline Lightning *Lightning::get_lightning(int method, MeshS &mesh, OptixPrimeFunctionality &optixP, float &emissionval,
                                           std::vector<float> wavelengthsvec, bool cuda_enabled, char *matfile) {
    if (method == 0) return new BWLightning(mesh, optixP, emissionval, matfile);
    if (method == 1) return new RGBLightning(mesh, optixP, emissionval, cuda_enabled, matfile);
    if (method == 2) return new SpectralLightning(mesh, optixP, emissionval, wavelengthsvec, cuda_enabled, matfile);
    return nullptr;
}
