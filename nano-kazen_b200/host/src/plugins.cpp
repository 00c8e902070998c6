/* plugins.cpp -- kazen's registered plugin classes as GPU-feeding descriptors, the scene
 * flattening into include/kzgpu.h tables, and the render driver.
 *
 * Registered names, XML properties and defaults are kazen's (SURVEY Appendix D):
 *   scene | obj | diffuse kazenstandard normalmap | area | perspective thinlens |
 *   independent stratified correlated pmj02bn | constanttexture imagetexture background colorramp blend |
 *   gaussian mitchell tent box | path_mis (GPU) | gpu_bvh (new: accelerator as a plugin)
 */
#include <kazen/scene.h>
#include <chrono>
#include <cmath>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <unordered_map>

namespace kazen {

static const float kPi = 3.14159265358979323846f;

/* =============================================================== reconstruction filters (rfilter.cpp:10-102) */
kz_filter_desc ReconstructionFilter::tabulate() const {
    kz_filter_desc d;
    d.radius = m_radius;
    for (int i = 0; i < 32; ++i) d.table[i] = eval((m_radius * i) / 32);     /* block.cpp:16-19 */
    d.table[32] = 0.0f;
    return d;
}
class GaussianFilter : public ReconstructionFilter {
public:
    GaussianFilter(const PropertyList &p) { m_radius = p.getFloat("radius", 2.0f); m_stddev = p.getFloat("stddev", 0.5f); }
    float eval(float x) const override {
        const float alpha = -1.0f / (2.0f * m_stddev * m_stddev);
        return std::max(0.0f, std::exp(alpha * x * x) - std::exp(alpha * m_radius * m_radius));
    }
    std::string toString() const override { return fmt("GaussianFilter[radius=%f, stddev=%f]", m_radius, m_stddev); }
private:
    float m_stddev;
};
class MitchellNetravaliFilter : public ReconstructionFilter {
public:
    MitchellNetravaliFilter(const PropertyList &p) { m_radius = p.getFloat("radius", 2.0f); m_B = p.getFloat("B", 1.0f / 3.0f); m_C = p.getFloat("C", 1.0f / 3.0f); }
    float eval(float x) const override {
        x = std::fabs(2.0f * x / m_radius);
        const float x2 = x * x, x3 = x2 * x;
        if (x < 1) return 1.0f / 6.0f * ((12 - 9 * m_B - 6 * m_C) * x3 + (-18 + 12 * m_B + 6 * m_C) * x2 + (6 - 2 * m_B));
        if (x < 2) return 1.0f / 6.0f * ((-m_B - 6 * m_C) * x3 + (6 * m_B + 30 * m_C) * x2 + (-12 * m_B - 48 * m_C) * x + (8 * m_B + 24 * m_C));
        return 0.0f;
    }
    std::string toString() const override { return fmt("MitchellNetravaliFilter[radius=%f, B=%f, C=%f]", m_radius, m_B, m_C); }
private:
    float m_B, m_C;
};
class TentFilter : public ReconstructionFilter {
public:
    TentFilter(const PropertyList &) { m_radius = 1.0f; }
    float eval(float x) const override { return std::max(0.0f, 1.0f - std::fabs(x)); }
    std::string toString() const override { return "TentFilter[]"; }
};
class BoxFilter : public ReconstructionFilter {
public:
    BoxFilter(const PropertyList &) { m_radius = 0.5f; }
    float eval(float) const override { return 1.0f; }
    std::string toString() const override { return "BoxFilter[]"; }
};
KAZEN_REGISTER_CLASS(GaussianFilter, "gaussian");
KAZEN_REGISTER_CLASS(MitchellNetravaliFilter, "mitchell");
KAZEN_REGISTER_CLASS(TentFilter, "tent");
KAZEN_REGISTER_CLASS(BoxFilter, "box");

/* =============================================================== textures (texture.cpp:10-270) */
static kz_texture_desc blankTexture(int type) {
    kz_texture_desc t; memset(&t, 0, sizeof(t));
    t.type = type; t.image = -1; t.scale = 1.f; t.child[0] = t.child[1] = t.child[2] = -1;
    return t;
}
static int memoized(FlattenCtx &ctx, const Object *o) { auto it = ctx.memo.find(o); return it == ctx.memo.end() ? -1 : it->second; }

class ConstantTexture : public Texture {
public:
    ConstantTexture(const PropertyList &p) { m_color = p.getColor("color", Color3{0.5f, 0.5f, 0.5f}); }
    int flatten(FlattenCtx &ctx) const override {
        int k = memoized(ctx, this); if (k >= 0) return k;
        kz_texture_desc t = blankTexture(KZ_TEX_CONSTANT);
        t.color[0] = m_color.r; t.color[1] = m_color.g; t.color[2] = m_color.b;
        ctx.textures.push_back(t);
        return ctx.memo[this] = (int)ctx.textures.size() - 1;
    }
    std::string toString() const override { return fmt("ConstantTexture[color=%f %f %f]", m_color.r, m_color.g, m_color.b); }
private:
    Color3 m_color;
};
class ImageTexture : public Texture {
public:
    ImageTexture(const PropertyList &p) {
        m_filename = resolvePath(p.getString("filename"));
        m_colorspace = p.getString("colorspace", "srgb");
        m_scale = p.getFloat("scale", 1.0f);
        std::string err;
        if (!readImage(m_filename, m_w, m_h, m_rgb, err)) throw Exception("imagetexture \"" + m_filename + "\": " + err);
    }
    int flatten(FlattenCtx &ctx) const override {
        int k = memoized(ctx, this); if (k >= 0) return k;
        ctx.image_data.push_back(m_rgb);
        kz_image_desc im; im.width = m_w; im.height = m_h; im.rgb = nullptr;       /* pointer patched once all images exist */
        ctx.images.push_back(im);
        kz_texture_desc t = blankTexture(KZ_TEX_IMAGE);
        t.image = (int)ctx.images.size() - 1; t.scale = m_scale; t.srgb = m_colorspace == "srgb";
        ctx.textures.push_back(t);
        return ctx.memo[this] = (int)ctx.textures.size() - 1;
    }
    std::string toString() const override { return "ImageTexture[" + m_filename + "]"; }
private:
    std::string m_filename, m_colorspace; float m_scale; int m_w = 0, m_h = 0; std::vector<float> m_rgb;
};
/* unary / ternary nodes keep their children by id like the reference's addChild() */
class BackgroundTexture : public Texture {
public:
    BackgroundTexture(const PropertyList &p) { m_intensity = p.getFloat("intensity", 1.0f); }
    ~BackgroundTexture() override { delete m_nested; }
    void addChild(Object *o) override {
        if (o->getClassType() != ETexture) throw Exception("BackgroundTexture::addChild(<" + classTypeName(o->getClassType()) + ">) is not supported!");
        if (m_nested) throw Exception("There is already a nested texture defined!");
        m_nested = static_cast<Texture *>(o);
    }
    int flatten(FlattenCtx &ctx) const override {
        int k = memoized(ctx, this); if (k >= 0) return k;
        kz_texture_desc t = blankTexture(KZ_TEX_BACKGROUND);
        t.a = m_intensity; t.child[0] = m_nested ? m_nested->flatten(ctx) : -1;
        ctx.textures.push_back(t);
        return ctx.memo[this] = (int)ctx.textures.size() - 1;
    }
    std::string toString() const override { return fmt("BackgroundTexture[intensity=%f]", m_intensity); }
private:
    float m_intensity; Texture *m_nested = nullptr;
};
class ColorRampTexture : public Texture {
public:
    ColorRampTexture(const PropertyList &p) { m_min = p.getFloat("min", 0.0f); m_max = p.getFloat("max", 1.0f); }
    ~ColorRampTexture() override { delete m_nested; }
    void addChild(Object *o) override {
        if (o->getClassType() != ETexture) throw Exception("ColorRampTexture::addChild(<" + classTypeName(o->getClassType()) + ">) is not supported!");
        m_nested = static_cast<Texture *>(o);
    }
    int flatten(FlattenCtx &ctx) const override {
        int k = memoized(ctx, this); if (k >= 0) return k;
        kz_texture_desc t = blankTexture(KZ_TEX_COLORRAMP);
        t.a = m_min; t.b = m_max; t.child[0] = m_nested ? m_nested->flatten(ctx) : -1;
        ctx.textures.push_back(t);
        return ctx.memo[this] = (int)ctx.textures.size() - 1;
    }
    std::string toString() const override { return fmt("ColorRampTexture[min=%f, max=%f]", m_min, m_max); }
private:
    float m_min, m_max; Texture *m_nested = nullptr;
};
class BlendTexture : public Texture {
public:
    BlendTexture(const PropertyList &p) { m_blendmode = p.getString("blendmode", "mix"); }
    ~BlendTexture() override { delete m_mask; delete m_in1; delete m_in2; }
    void addChild(Object *o) override {
        if (o->getClassType() != ETexture) throw Exception("BlendTexture::addChild(<" + classTypeName(o->getClassType()) + ">) is not supported!");
        Texture *t = static_cast<Texture *>(o);
        if (o->getId() == "mask") { if (m_mask) throw Exception("There is already a mask defined!"); m_mask = t; }
        else if (o->getId() == "input1") { if (m_in1) throw Exception("There is already an input1 defined!"); m_in1 = t; }
        else if (o->getId() == "input2") { if (m_in2) throw Exception("There is already an input2 defined!"); m_in2 = t; }
        else delete t;      /* texture.cpp:236-250 ignores other ids */
    }
    int flatten(FlattenCtx &ctx) const override {
        int k = memoized(ctx, this); if (k >= 0) return k;
        kz_texture_desc t = blankTexture(KZ_TEX_BLEND);
        t.mode = m_blendmode == "mix" ? KZ_BLEND_MIX : (m_blendmode == "multiply" ? KZ_BLEND_MULTIPLY : KZ_BLEND_OTHER);
        t.child[0] = m_mask ? m_mask->flatten(ctx) : -1; t.child[1] = m_in1 ? m_in1->flatten(ctx) : -1; t.child[2] = m_in2 ? m_in2->flatten(ctx) : -1;
        ctx.textures.push_back(t);
        return ctx.memo[this] = (int)ctx.textures.size() - 1;
    }
    std::string toString() const override { return "BlendTexture[" + m_blendmode + "]"; }
private:
    std::string m_blendmode; Texture *m_mask = nullptr, *m_in1 = nullptr, *m_in2 = nullptr;
};
KAZEN_REGISTER_CLASS(ConstantTexture, "constanttexture");
KAZEN_REGISTER_CLASS(ImageTexture, "imagetexture");
KAZEN_REGISTER_CLASS(BackgroundTexture, "background");
KAZEN_REGISTER_CLASS(ColorRampTexture, "colorramp");
KAZEN_REGISTER_CLASS(BlendTexture, "blend");

/* =============================================================== BSDFs */
static kz_bsdf_desc blankBsdf(int type) {
    kz_bsdf_desc b; memset(&b, 0, sizeof(b));
    b.type = type; b.base_color = b.roughness = b.metallic = b.normal_map = b.nested = -1;
    b.int_ior = 1.5046f; b.ext_ior = 1.000277f;
    return b;
}
class Diffuse : public BSDF {       /* bsdf.cpp:20-92 */
public:
    Diffuse(const PropertyList &p) { m_albedo = p.getColor("albedo", Color3{0.5f, 0.5f, 0.5f}); }
    int flatten(FlattenCtx &ctx) const override {
        int k = memoized(ctx, this); if (k >= 0) return k;
        kz_bsdf_desc b = blankBsdf(KZ_BSDF_DIFFUSE);
        b.albedo[0] = m_albedo.r; b.albedo[1] = m_albedo.g; b.albedo[2] = m_albedo.b;
        ctx.bsdfs.push_back(b);
        return ctx.memo[this] = (int)ctx.bsdfs.size() - 1;
    }
    std::string toString() const override { return fmt("Diffuse[albedo=%f %f %f]", m_albedo.r, m_albedo.g, m_albedo.b); }
private:
    Color3 m_albedo;
};
class KazenStandardSurface : public BSDF {      /* bsdf.cpp:1157-1418 */
public:
    KazenStandardSurface(const PropertyList &p) {
        m_anisotropy = p.getFloat("anisotropy", 0.f); m_specular = p.getFloat("specular", 0.5f); m_specularTint = p.getFloat("specularTint", 0.5f);
        m_clearcoat = p.getFloat("clearcoat", 0.f); m_clearcoatRoughness = p.getFloat("clearcoatRoughness", 0.5f);
        m_sheen = p.getFloat("sheen", 0.f); m_sheenTint = p.getFloat("sheenTint", 0.5f);
    }
    ~KazenStandardSurface() override { delete m_baseColor; delete m_metallic; delete m_roughness; }
    void addChild(Object *o) override {        /* bsdf.cpp:1373-1395 */
        if (o->getClassType() != ETexture) throw Exception("KazenStandardSurface::addChild(<" + classTypeName(o->getClassType()) + ">) is not supported!");
        Texture *t = static_cast<Texture *>(o);
        if (o->getId() == "baseColor") { if (m_baseColor) throw Exception("There is already an baseColor defined!"); m_baseColor = t; }
        else if (o->getId() == "metallic") { if (m_metallic) throw Exception("There is already an metallic defined!"); m_metallic = t; }
        else if (o->getId() == "roughness") { if (m_roughness) throw Exception("There is already an roughness defined!"); m_roughness = t; }
        else throw Exception("KazenStandardSurface: unknown texture id \"" + o->getId() + "\"");
    }
    void activate() override {                 /* the reference dereferences the three textures unconditionally */
        if (!m_baseColor || !m_metallic || !m_roughness) throw Exception("kazenstandard needs baseColor, roughness and metallic textures");
    }
    int flatten(FlattenCtx &ctx) const override {
        int k = memoized(ctx, this); if (k >= 0) return k;
        kz_bsdf_desc b = blankBsdf(KZ_BSDF_KISS);
        b.base_color = m_baseColor->flatten(ctx); b.roughness = m_roughness->flatten(ctx); b.metallic = m_metallic->flatten(ctx);
        b.anisotropy = m_anisotropy; b.specular = m_specular; b.specular_tint = m_specularTint; b.clearcoat = m_clearcoat;
        b.clearcoat_roughness = m_clearcoatRoughness; b.sheen = m_sheen; b.sheen_tint = m_sheenTint;
        ctx.bsdfs.push_back(b);
        return ctx.memo[this] = (int)ctx.bsdfs.size() - 1;
    }
    std::string toString() const override { return "KazenStandardSurface[]"; }
private:
    Texture *m_baseColor = nullptr, *m_metallic = nullptr, *m_roughness = nullptr;
    float m_anisotropy, m_specular, m_specularTint, m_clearcoat, m_clearcoatRoughness, m_sheen, m_sheenTint;
};
class NormalMap : public BSDF {     /* bsdf.cpp:281-417 */
public:
    NormalMap(const PropertyList &) {}
    ~NormalMap() override { delete m_normalMap; delete m_nested; }
    void addChild(Object *o) override {
        if (o->getClassType() == ETexture) m_normalMap = static_cast<Texture *>(o);
        else if (o->getClassType() == EBSDF) m_nested = static_cast<BSDF *>(o);
        else throw Exception("addChild is not supported other than normal maps and nested BSDF");
    }
    void activate() override { if (!m_normalMap || !m_nested) throw Exception("normalmap needs a texture and a nested bsdf"); }
    int flatten(FlattenCtx &ctx) const override {
        int k = memoized(ctx, this); if (k >= 0) return k;
        kz_bsdf_desc b = blankBsdf(KZ_BSDF_NORMALMAP);
        b.nested = m_nested->flatten(ctx); b.normal_map = m_normalMap->flatten(ctx);
        ctx.bsdfs.push_back(b);
        return ctx.memo[this] = (int)ctx.bsdfs.size() - 1;
    }
    std::string toString() const override { return "NormalMap[]"; }
private:
    Texture *m_normalMap = nullptr; BSDF *m_nested = nullptr;
};
/* ---- SURVEY 8(f)-1: the remaining BSDF plugins (bsdf.cpp:98-276, 629-1145) ---- */
static float alphaFromRoughness(float roughness) { return std::max(0.001f, roughness * roughness); }     /* bsdf.cpp:696-701 */
class SimpleBsdf : public BSDF {        /* parameter-only BSDFs share the flatten boilerplate */
public:
    int flatten(FlattenCtx &ctx) const override {
        int k = memoized(ctx, this); if (k >= 0) return k;
        kz_bsdf_desc b = m_desc;
        if (m_albedoTex) b.base_color = m_albedoTex->flatten(ctx);
        ctx.bsdfs.push_back(b);
        return ctx.memo[this] = (int)ctx.bsdfs.size() - 1;
    }
    ~SimpleBsdf() override { delete m_albedoTex; }
protected:
    kz_bsdf_desc m_desc = blankBsdf(KZ_BSDF_DIFFUSE);
    Texture *m_albedoTex = nullptr;
};
class Dielectric : public SimpleBsdf {
public:
    Dielectric(const PropertyList &p) { m_desc = blankBsdf(KZ_BSDF_DIELECTRIC); m_desc.int_ior = p.getFloat("intIOR", 1.5046f); m_desc.ext_ior = p.getFloat("extIOR", 1.000277f); }
    std::string toString() const override { return fmt("Dielectric[intIOR=%f, extIOR=%f]", m_desc.int_ior, m_desc.ext_ior); }
};
class Mirror : public SimpleBsdf {
public:
    Mirror(const PropertyList &) { m_desc = blankBsdf(KZ_BSDF_MIRROR); }
    std::string toString() const override { return "Mirror[]"; }
};
class Lambertian : public SimpleBsdf {
public:
    Lambertian(const PropertyList &) { m_desc = blankBsdf(KZ_BSDF_LAMBERTIAN); }
    void addChild(Object *o) override {
        if (o->getClassType() != ETexture) throw Exception("addChild is not supported other than albedi maps");
        delete m_albedoTex; m_albedoTex = static_cast<Texture *>(o);
    }
    void activate() override { if (!m_albedoTex) throw Exception("lambertian needs an albedo texture"); }
    std::string toString() const override { return "Lambertian[]"; }
};
class GGX : public SimpleBsdf {
public:
    GGX(const PropertyList &p) { m_desc = blankBsdf(KZ_BSDF_GGX); m_desc.alpha = p.getFloat("roughness", 0.5f); m_desc.anisotropy = p.getFloat("anisotropy", 0.f); }
    void addChild(Object *o) override {
        if (o->getClassType() != ETexture) throw Exception("addChild is not supported other than albedi maps");
        delete m_albedoTex; m_albedoTex = static_cast<Texture *>(o);
    }
    void activate() override { if (!m_albedoTex) throw Exception("ggx needs an albedo texture"); }
    std::string toString() const override { return "GGX[]"; }
};
class RoughConductor : public SimpleBsdf {
public:
    RoughConductor(const PropertyList &p) {
        m_desc = blankBsdf(KZ_BSDF_ROUGHCONDUCTOR);
        m_desc.alpha = alphaFromRoughness(p.getFloat("alpha", 0.1f));
        const std::string mat = p.getString("material", "Au");
        static const float tab[3][6] = {{0.1431189557f, 0.3749570432f, 1.4424785571f, 3.9831604247f, 2.3857207478f, 1.6032152899f},
                                        {0.2004376970f, 0.9240334304f, 1.1022119527f, 3.9129485033f, 2.4528477015f, 2.1421879552f},
                                        {4.3696828663f, 2.9167024892f, 1.6547005413f, 5.2064337956f, 4.2313645277f, 3.7549467933f}};
        const int k = mat == "Au" ? 0 : (mat == "Cu" ? 1 : (mat == "Cr" ? 2 : -1));
        if (k < 0) throw Exception("roughconductor: unknown material \"" + mat + "\" (Au | Cu | Cr); the reference leaves eta/k uninitialised here");
        for (int c = 0; c < 3; ++c) { m_desc.eta[c] = tab[k][c]; m_desc.k[c] = tab[k][3 + c]; }
    }
    std::string toString() const override { return fmt("RoughConductor[alpha=%f]", m_desc.alpha); }
};
class RoughPlastic : public SimpleBsdf {
public:
    RoughPlastic(const PropertyList &p) {
        m_desc = blankBsdf(KZ_BSDF_ROUGHPLASTIC);
        m_desc.alpha = alphaFromRoughness(p.getFloat("alpha", 0.1f));
        m_desc.int_ior = p.getFloat("intIOR", 1.5046f); m_desc.ext_ior = p.getFloat("extIOR", 1.000277f);
        const Color3 kd = p.getColor("kd", Color3{0.5f, 0.5f, 0.5f});
        m_desc.albedo[0] = kd.r; m_desc.albedo[1] = kd.g; m_desc.albedo[2] = kd.b;
    }
    std::string toString() const override { return fmt("RoughPlastic[alpha=%f]", m_desc.alpha); }
};
class RoughDielectric : public SimpleBsdf {
public:
    RoughDielectric(const PropertyList &p) {
        m_desc = blankBsdf(KZ_BSDF_ROUGHDIELECTRIC);
        m_desc.int_ior = p.getFloat("intIOR", 1.5046f); m_desc.ext_ior = p.getFloat("extIOR", 1.000277f);
        m_desc.alpha = alphaFromRoughness(p.getFloat("roughness", 0.1f));
    }
    std::string toString() const override { return "RoughDielectric"; }
};
KAZEN_REGISTER_CLASS(Diffuse, "diffuse");
KAZEN_REGISTER_CLASS(KazenStandardSurface, "kazenstandard");
KAZEN_REGISTER_CLASS(NormalMap, "normalmap");
KAZEN_REGISTER_CLASS(Dielectric, "dielectric");
KAZEN_REGISTER_CLASS(Mirror, "mirror");
KAZEN_REGISTER_CLASS(Lambertian, "lambertian");
KAZEN_REGISTER_CLASS(GGX, "ggx");
KAZEN_REGISTER_CLASS(RoughConductor, "roughconductor");
KAZEN_REGISTER_CLASS(RoughPlastic, "roughplastic");
KAZEN_REGISTER_CLASS(RoughDielectric, "roughdielectric");

/* =============================================================== lights (light.cpp:7-66) */
class AreaLight : public Light {
public:
    AreaLight(const PropertyList &p) {
        m_color = p.getColor("color", Color3{1.f, 1.f, 1.f}); m_intensity = p.getFloat("intensity", 1.f);
        m_visible = p.getBoolean("lightPrimaryVisibility", false);
    }
    kz_light_desc describe() const override {
        kz_light_desc l;
        l.radiance[0] = m_intensity * m_color.r; l.radiance[1] = m_intensity * m_color.g; l.radiance[2] = m_intensity * m_color.b;
        l.primary_visibility = m_visible ? 1 : 0;
        return l;
    }
    std::string toString() const override { return fmt("AreaLight[color=%f %f %f, intensity=%f]", m_color.r, m_color.g, m_color.b, m_intensity); }
private:
    Color3 m_color; float m_intensity; bool m_visible;
};
KAZEN_REGISTER_CLASS(AreaLight, "area");

/* =============================================================== cameras (camera.cpp:14-270) */
void Camera::readCommon(const PropertyList &p) {
    m_width = p.getInteger("width", 1280); m_height = p.getInteger("height", 720);
    m_cameraToWorld = p.getTransform("toWorld", Transform());
    m_fov = p.getFloat("fov", 30.0f); m_near = p.getFloat("nearClip", 1e-4f); m_far = p.getFloat("farClip", 1e4f);
}
void Camera::addChild(Object *obj) {
    if (obj->getClassType() != EReconstructionFilter) throw Exception("Camera::addChild(<" + classTypeName(obj->getClassType()) + ">) is not supported!");
    if (m_rfilter) throw Exception("Camera: tried to register multiple reconstruction filters!");
    m_rfilter = static_cast<ReconstructionFilter *>(obj);
}
void Camera::activate() {
    const float aspect = m_width / (float)m_height;
    const float recip = 1.0f / (m_far - m_near), cot = 1.0f / std::tan((m_fov / 2.0f) * (kPi / 180.0f));
    Mat4 P = Mat4::identity();
    P.m[0][0] = cot; P.m[1][1] = cot; P.m[2][2] = m_far * recip; P.m[2][3] = -m_near * m_far * recip; P.m[3][2] = 1.f; P.m[3][3] = 0.f;
    Mat4 T = Mat4::identity(); T.m[0][3] = -1.0f; T.m[1][3] = -1.0f / aspect;
    Mat4 S = Mat4::identity(); S.m[0][0] = -0.5f; S.m[1][1] = -0.5f * aspect;
    m_sampleToCamera = (S * (T * P)).inverse();
    if (!m_rfilter) m_rfilter = static_cast<ReconstructionFilter *>(ObjectFactory::createInstance("gaussian", PropertyList()));
}
static void fillCamera(kz_camera_desc &c, int type, int w, int h, const Mat4 &s2c, const Transform &c2w, float nearc, float farc, float ap, float focus) {
    c.type = type; c.width = w; c.height = h;
    memcpy(c.sample_to_camera, s2c.m, sizeof(c.sample_to_camera));
    memcpy(c.camera_to_world, c2w.matrix.m, sizeof(c.camera_to_world));
    c.near_clip = nearc; c.far_clip = farc; c.aperture_radius = ap; c.focus_distance = focus;
}
class PerspectiveCamera : public Camera {
public:
    PerspectiveCamera(const PropertyList &p) { readCommon(p); }
    kz_camera_desc describe() const override { kz_camera_desc c; fillCamera(c, KZ_CAM_PERSPECTIVE, m_width, m_height, m_sampleToCamera, m_cameraToWorld, m_near, m_far, 1.f, 0.f); return c; }
    std::string toString() const override { return fmt("PerspectiveCamera[%dx%d, fov=%f]", m_width, m_height, m_fov); }
};
class ThinlensCamera : public Camera {
public:
    ThinlensCamera(const PropertyList &p) { readCommon(p); m_aperture = p.getFloat("apertureRadius", 1.0f); m_focus = p.getFloat("focusDistance", 0.0f); }
    kz_camera_desc describe() const override { kz_camera_desc c; fillCamera(c, KZ_CAM_THINLENS, m_width, m_height, m_sampleToCamera, m_cameraToWorld, m_near, m_far, m_aperture, m_focus); return c; }
    std::string toString() const override { return fmt("ThinlensCamera[%dx%d, fov=%f, aperture=%f, focus=%f]", m_width, m_height, m_fov, m_aperture, m_focus); }
private:
    float m_aperture, m_focus;
};
KAZEN_REGISTER_CLASS(PerspectiveCamera, "perspective");
KAZEN_REGISTER_CLASS(ThinlensCamera, "thinlens");

/* =============================================================== samplers: constructor rounding (sampler.cpp:20-22,83-93,178-189,275-289) */
static kz_sampler_desc samplerDesc(int type, uint32_t spp, uint64_t seed, int rx, int ry) {
    kz_sampler_desc s; memset(&s, 0, sizeof(s));
    s.type = type; s.sample_count = spp; s.seed = seed; s.res_x = rx; s.res_y = ry;
    return s;
}
class Independent : public Sampler {
public:
    /* the reference leaves m_seed uninitialised (sampler.cpp:20-22,44: UB); this build defaults it to 1 like the other samplers */
    Independent(const PropertyList &p) { m_sampleCount = (uint32_t)p.getInteger("sampleCount", 1); m_seed = (uint64_t)p.getInteger("seed", 1); }
    kz_sampler_desc describe() const override { return samplerDesc(KZ_SAMPLER_INDEPENDENT, m_sampleCount, m_seed, 0, 0); }
    std::string toString() const override { return fmt("Independent[sampleCount=%u]", m_sampleCount); }
};
class Stratified : public Sampler {
public:
    Stratified(const PropertyList &p) {
        m_seed = (uint64_t)p.getInteger("seed", 1);
        size_t count = (size_t)p.getInteger("sampleCount", 16);
        m_resolution = (size_t)p.getInteger("resolution", 4);
        while (m_resolution * m_resolution < count) m_resolution++;
        if (count != m_resolution * m_resolution) std::cout << "Sample count should be square and power of two, rounding to " << m_resolution * m_resolution << std::endl;
        m_sampleCount = (uint32_t)(m_resolution * m_resolution);
    }
    kz_sampler_desc describe() const override { return samplerDesc(KZ_SAMPLER_STRATIFIED, m_sampleCount, m_seed, (int)m_resolution, (int)m_resolution); }
    std::string toString() const override { return fmt("Stratified[sampleCount=%u]", m_sampleCount); }
private:
    size_t m_resolution;
};
class Correlated : public Sampler {
public:
    Correlated(const PropertyList &p) {
        m_seed = (uint64_t)p.getInteger("seed", 1);
        m_sampleCount = (uint32_t)p.getInteger("sampleCount", 16);
        m_res[1] = (int)std::sqrt((double)m_sampleCount);
        m_res[0] = (int)((m_sampleCount + (uint32_t)m_res[1] - 1) / (uint32_t)m_res[1]);
        if (m_sampleCount != (uint32_t)(m_res[0] * m_res[1])) std::cout << "Sample count rounded up to " << m_res[0] * m_res[1] << std::endl;
        m_sampleCount = (uint32_t)(m_res[0] * m_res[1]);
    }
    kz_sampler_desc describe() const override { return samplerDesc(KZ_SAMPLER_CORRELATED, m_sampleCount, m_seed, m_res[0], m_res[1]); }
    std::string toString() const override { return fmt("Correlated[sampleCount=%u]", m_sampleCount); }
private:
    int m_res[2];
};
class PMJ02BN : public Sampler {
public:
    PMJ02BN(const PropertyList &p) {
        m_seed = (uint64_t)p.getInteger("seed", 1);
        m_sampleCount = (uint32_t)p.getInteger("sampleCount", 16);
        if (m_sampleCount > 65536) m_sampleCount = 65536;
        /* optional binary blob: uint16[48*128*128] blue noise followed by uint32[5*65536*2] pmj02bn */
        m_tableFile = p.getString("tableFile", getenv("KAZEN_PMJ02BN_TABLES") ? getenv("KAZEN_PMJ02BN_TABLES") : "");
    }
    kz_sampler_desc describe() const override { return samplerDesc(KZ_SAMPLER_PMJ02BN, m_sampleCount, m_seed, 0, 0); }
    const std::string &tableFile() const { return m_tableFile; }
    std::string toString() const override { return fmt("PMJ02BN[sampleCount=%u]", m_sampleCount); }
private:
    std::string m_tableFile;
};
KAZEN_REGISTER_CLASS(Independent, "independent");
KAZEN_REGISTER_CLASS(Stratified, "stratified");
KAZEN_REGISTER_CLASS(Correlated, "correlated");
KAZEN_REGISTER_CLASS(PMJ02BN, "pmj02bn");

/* =============================================================== meshes (mesh.cpp:14-53,136-161,200-343) */
Mesh::~Mesh() { delete m_bsdf; delete m_light; }
void Mesh::addChild(Object *obj) {
    switch (obj->getClassType()) {
        case EBSDF:
            if (m_bsdf) throw Exception("Mesh: tried to register multiple BSDF instances!");
            m_bsdf = static_cast<BSDF *>(obj);
            break;
        case ELight:
            if (m_light) throw Exception("Mesh: tried to register multiple Light instances!");
            m_light = static_cast<Light *>(obj);
            break;
        default:
            throw Exception("Mesh::addChild(<" + classTypeName(obj->getClassType()) + ">) is not supported!");
    }
}
void Mesh::activate() {
    if (!m_bsdf) m_bsdf = static_cast<BSDF *>(ObjectFactory::createInstance("diffuse", PropertyList()));
}
std::string Mesh::toString() const { return fmt("Mesh[name=\"%s\", vertexCount=%zu, triangleCount=%zu]", m_name.c_str(), m_V.size() / 3, m_F.size() / 3); }

class WavefrontOBJ : public Mesh {
public:
    WavefrontOBJ(const PropertyList &props) {
        const std::string filename = resolvePath(props.getString("filename"));
        std::ifstream is(filename);
        if (is.fail()) throw Exception("Unable to open OBJ file \"" + filename + "\"!");
        const Transform trafo = props.getTransform("toWorld", Transform());
        std::vector<Vec3> positions, normals; std::vector<float> texcoords;
        struct Key { uint32_t p, n, uv; bool operator==(const Key &o) const { return p == o.p && n == o.n && uv == o.uv; } };
        struct KeyHash { size_t operator()(const Key &k) const { size_t h = std::hash<uint32_t>()(k.p); h = h * 37 + std::hash<uint32_t>()(k.uv); return h * 37 + std::hash<uint32_t>()(k.n); } };
        std::unordered_map<Key, uint32_t, KeyHash> seen;
        std::vector<Key> verts;
        auto parseVertex = [](const std::string &s) -> Key {        /* "p", "p/uv", "p//n", "p/uv/n" (1-based) */
            Key k{(uint32_t)-1, (uint32_t)-1, (uint32_t)-1};
            std::vector<std::string> tk; size_t b = 0;
            for (;;) { size_t e = s.find('/', b); tk.push_back(s.substr(b, e == std::string::npos ? e : e - b)); if (e == std::string::npos) break; b = e + 1; }
            if (tk.empty() || tk.size() > 3) throw Exception("Invalid vertex data: \"" + s + "\"");
            auto toU = [&](const std::string &t) { char *end = nullptr; unsigned long v = strtoul(t.c_str(), &end, 10); if (*end != '\0') throw Exception("Could not parse integer value \"" + t + "\""); return (uint32_t)v; };
            k.p = toU(tk[0]);
            if (tk.size() >= 2 && !tk[1].empty()) k.uv = toU(tk[1]);
            if (tk.size() >= 3 && !tk[2].empty()) k.n = toU(tk[2]);
            return k;
        };
        std::string lineStr;
        while (std::getline(is, lineStr)) {
            std::istringstream line(lineStr);
            std::string prefix; line >> prefix;
            if (prefix == "v") { Vec3 p; line >> p.x >> p.y >> p.z; positions.push_back(trafo.point(p)); }
            else if (prefix == "vt") { float u = 0, v = 0; line >> u >> v; texcoords.push_back(u); texcoords.push_back(v); }
            else if (prefix == "vn") {
                Vec3 n; line >> n.x >> n.y >> n.z;
                n = trafo.normal(n);
                /* Eigen's normalized() (mesh.cpp:244): v / sqrt(v.v) when v.v > 0, else v itself; the unrolled 3-term reduction adds a0*b0 + (a1*b1 + a2*b2) */
                const float z = n.x * n.x + (n.y * n.y + n.z * n.z);
                if (z > 0.f) { const float l = std::sqrt(z); n = Vec3{n.x / l, n.y / l, n.z / l}; }
                normals.push_back(n);
            } else if (prefix == "f") {
                std::string v1, v2, v3, v4; line >> v1 >> v2 >> v3 >> v4;
                Key f[6]; int nv = 3;
                f[0] = parseVertex(v1); f[1] = parseVertex(v2); f[2] = parseVertex(v3);
                if (!v4.empty()) { f[3] = parseVertex(v4); f[4] = f[0]; f[5] = f[2]; nv = 6; }      /* quad -> (0,1,2),(3,0,2) */
                for (int i = 0; i < nv; ++i) {
                    auto it = seen.find(f[i]);
                    if (it == seen.end()) { seen[f[i]] = (uint32_t)verts.size(); m_F.push_back((uint32_t)verts.size()); verts.push_back(f[i]); }
                    else m_F.push_back(it->second);
                }
            }
        }
        m_F.resize(m_F.size() / 3 * 3);
        auto fetch = [&](size_t idx, size_t n, const char *what) { if (idx < 1 || idx > n) throw Exception(std::string("OBJ ") + what + " index out of range in \"" + filename + "\""); return idx - 1; };
        m_V.resize(verts.size() * 3);
        for (size_t i = 0; i < verts.size(); ++i) { const Vec3 &p = positions[fetch(verts[i].p, positions.size(), "position")]; m_V[3 * i] = p.x; m_V[3 * i + 1] = p.y; m_V[3 * i + 2] = p.z; }
        if (!normals.empty()) {
            m_N.resize(verts.size() * 3);
            for (size_t i = 0; i < verts.size(); ++i) { const Vec3 &n = normals[fetch(verts[i].n, normals.size(), "normal")]; m_N[3 * i] = n.x; m_N[3 * i + 1] = n.y; m_N[3 * i + 2] = n.z; }
        }
        if (!texcoords.empty()) {
            m_UV.resize(verts.size() * 2);
            for (size_t i = 0; i < verts.size(); ++i) { const size_t k = fetch(verts[i].uv, texcoords.size() / 2, "texcoord"); m_UV[2 * i] = texcoords[2 * k]; m_UV[2 * i + 1] = texcoords[2 * k + 1]; }
        }
        m_name = filename;
    }
};
KAZEN_REGISTER_CLASS(WavefrontOBJ, "obj");

/* =============================================================== accelerator plugin */
class GpuBvh : public Accel {
public:
    GpuBvh(const PropertyList &p) {
        const std::string b = p.getString("builder", "sah");
        if (b == "sah") m_builder = KZ_BUILD_HOST_SAH; else if (b == "lbvh") m_builder = KZ_BUILD_LBVH;
        else throw Exception("gpu_bvh: unknown builder \"" + b + "\" (sah | lbvh)");
    }
    void addMesh(Mesh *mesh) override { m_meshes.push_back(mesh); }
    void build() override {}
    int builder() const override { return m_builder; }
    std::string toString() const override { return fmt("GpuBvh[builder=%s, meshes=%zu]", m_builder == KZ_BUILD_LBVH ? "lbvh" : "sah", m_meshes.size()); }
private:
    int m_builder; std::vector<Mesh *> m_meshes;
};
KAZEN_REGISTER_CLASS(GpuBvh, "gpu_bvh");

/* =============================================================== scene (scene.cpp:17-126) */
Scene::Scene(const PropertyList &props) {
    /* the reference hard-wires `new Accel()` (scene.cpp:17); here the accelerator is looked up by name */
    PropertyList ap;
    if (props.has("accelBuilder")) ap.setString("builder", props.getString("accelBuilder"));
    Object *a = ObjectFactory::createInstance(props.getString("accel", "gpu_bvh"), ap);
    if (a->getClassType() != EAccel) { delete a; throw Exception("scene: \"accel\" does not name an accelerator plugin"); }
    m_accel = static_cast<Accel *>(a);
    gpus = props.getInteger("gpus", 1);
}
Scene::~Scene() {
    for (Mesh *m : m_meshes) delete m;
    delete m_accel; delete m_sampler; delete m_camera; delete m_integrator; delete m_background;
}
void Scene::addChild(Object *obj) {
    switch (obj->getClassType()) {
        case EMesh: { Mesh *mesh = static_cast<Mesh *>(obj); m_accel->addMesh(mesh); m_meshes.push_back(mesh); } break;
        case ELight: throw Exception("Scene::addChild(): lights must be children of a mesh");
        case ESampler: if (m_sampler) throw Exception("There can only be one sampler per scene!"); m_sampler = static_cast<Sampler *>(obj); break;
        case ECamera: if (m_camera) throw Exception("There can only be one camera per scene!"); m_camera = static_cast<Camera *>(obj); break;
        case EIntegrator: if (m_integrator) throw Exception("There can only be one integrator per scene!"); m_integrator = static_cast<Integrator *>(obj); break;
        case EAccel: delete m_accel; m_accel = static_cast<Accel *>(obj); for (Mesh *m : m_meshes) m_accel->addMesh(m); break;
        case ETexture:
            if (obj->getId() == "background") { if (m_background) throw Exception("There is already a background defined!"); m_background = static_cast<Texture *>(obj); }
            else delete obj;
            break;
        default: throw Exception("Scene::addChild(<" + classTypeName(obj->getClassType()) + ">) is not supported!");
    }
}
void Scene::activate() {
    m_accel->build();
    if (!m_integrator) throw Exception("No integrator was specified!");
    if (!m_camera) throw Exception("No camera was specified!");
    if (!m_sampler) m_sampler = static_cast<Sampler *>(ObjectFactory::createInstance("independent", PropertyList()));
}
std::string Scene::toString() const {
    std::string s = "Scene[\n  integrator = " + m_integrator->toString() + ",\n  sampler = " + m_sampler->toString() + ",\n  camera = " + m_camera->toString() +
                    ",\n  accel = " + m_accel->toString() + ",\n  meshes = {\n";
    for (const Mesh *m : m_meshes) s += "    " + m->toString() + "\n";
    return s + "  }\n]";
}

const kz_scene_desc &Scene::flatten() {
    if (m_flat) return m_flat->desc;
    m_flat.reset(new FlattenCtx());
    FlattenCtx &c = *m_flat;
    for (Mesh *m : m_meshes) {
        kz_mesh_desc d; memset(&d, 0, sizeof(d));
        d.positions = m->m_V.data(); d.normals = m->m_N.empty() ? nullptr : m->m_N.data(); d.uvs = m->m_UV.empty() ? nullptr : m->m_UV.data();
        d.indices = m->m_F.data(); d.n_vertices = (uint32_t)(m->m_V.size() / 3); d.n_triangles = (uint32_t)(m->m_F.size() / 3);
        d.bsdf = m->getBSDF()->flatten(c);
        d.light = -1;
        if (m->isLight()) { c.lights.push_back(m->getLight()->describe()); d.light = (int32_t)c.lights.size() - 1; }
        c.meshes.push_back(d);
    }
    c.desc.background = m_background ? m_background->flatten(c) : -1;
    for (size_t i = 0; i < c.images.size(); ++i) c.images[i].rgb = c.image_data[i].data();
    c.desc.meshes = c.meshes.data(); c.desc.n_meshes = (uint32_t)c.meshes.size();
    c.desc.bsdfs = c.bsdfs.data(); c.desc.n_bsdfs = (uint32_t)c.bsdfs.size();
    c.desc.textures = c.textures.data(); c.desc.n_textures = (uint32_t)c.textures.size();
    c.desc.images = c.images.data(); c.desc.n_images = (uint32_t)c.images.size();
    c.desc.lights = c.lights.data(); c.desc.n_lights = (uint32_t)c.lights.size();
    c.desc.camera = m_camera->describe();
    c.desc.sampler = m_sampler->describe();
    if (c.desc.sampler.type == KZ_SAMPLER_PMJ02BN) {
        const std::string &tf = static_cast<PMJ02BN *>(m_sampler)->tableFile();
        const size_t nb = 48 * 128 * 128, np = 5 * 65536 * 2;
        if (!tf.empty()) {
            std::ifstream f(resolvePath(tf), std::ios::binary);
            c.blue_noise.resize(nb); c.pmj.resize(np);
            if (!f.read((char *)c.blue_noise.data(), (std::streamsize)(nb * 2)) || !f.read((char *)c.pmj.data(), (std::streamsize)(np * 4)))
                throw Exception("pmj02bn: cannot read the sample tables from \"" + tf + "\"");
        } else {
            std::cout << "pmj02bn: the reference's blue-noise / pmj02bn tables are not part of its public tree; using the stand-in "
                         "(0,2)-sequence tables (set tableFile / KAZEN_PMJ02BN_TABLES to supply pbrt-v4's)" << std::endl;
            fallbackPmjTables(c.blue_noise, c.pmj);
        }
        c.desc.sampler.blue_noise = c.blue_noise.data(); c.desc.sampler.pmj02bn = c.pmj.data();
    }
    c.desc.integrator = m_integrator->describe();
    c.desc.filter = m_camera->getReconstructionFilter()->tabulate();
    return c.desc;
}

/* =============================================================== the GPU integrator + render driver */
class GpuPathMisIntegrator : public Integrator {        /* integrator.cpp:185-355 behind the C ABI */
public:
    GpuPathMisIntegrator(const PropertyList &p) {
        m_desc.max_depth = std::min(512, p.getInteger("maxDepth", 5));
        m_desc.trace_bias = p.getFloat("traceBias", 0.001f);
        m_desc.regularization = p.getBoolean("regularization", false) ? 1 : 0;
        m_desc.accumulated_roughness = p.getFloat("accumulatedRoughness", 0.5f);
        m_desc.type = KZ_INTEGRATOR_PATH_MIS;
        m_desc.env_sampling = p.getBoolean("envSampling", false) ? 1 : 0;     /* the environment as a light (kz_env.h); off: the reference estimator */
        m_desc.texture_filtering = p.getBoolean("textureFiltering", false) ? 1 : 0;     /* footprint-filtered image lookups (kz_texlod.h); off: mip level 0 */
    }
    GpuPathMisIntegrator(const PropertyList &, int type) { m_desc = kz_integrator_desc{5, 0.001f, 0, 0.5f, type, 0, 0}; }
    ~GpuPathMisIntegrator() override { if (m_ctx) kzgpu_destroy(m_ctx); }
    kz_integrator_desc describe() const override { return m_desc; }

    /* renderer.cpp:75: the upload / accel-build hook */
    void preprocess(const Scene *scene_) override {
        Scene *scene = const_cast<Scene *>(scene_);
        std::vector<int> ids;
        for (int i = 0; i < std::max(1, scene->gpus); ++i) ids.push_back(i);
        int rc = kzgpu_create(ids.data(), (int)ids.size(), &m_ctx);
        if (rc != KZ_OK) throw Exception(std::string("GPU integrator: ") + kzgpu_last_error(nullptr));
        if ((rc = kzgpu_scene_upload(m_ctx, &scene->flatten())) != KZ_OK) throw Exception(std::string("GPU integrator: scene upload failed: ") + kzgpu_last_error(m_ctx));
        if ((rc = kzgpu_accel_build(m_ctx, scene->getAccel()->builder())) != KZ_OK) throw Exception(std::string("GPU integrator: accel build failed: ") + kzgpu_last_error(m_ctx));
    }
    bool renderFrame(Scene *scene, ImageBlock &result) override {
        if (!m_ctx) preprocess(scene);
        int32_t w, h, b;
        kzgpu_frame_dims(m_ctx, &w, &h, &b);
        result.width = w; result.height = h; result.border = b;
        result.data.assign((size_t)(w + 2 * b) * (h + 2 * b) * 4, 0.f);
        const int32_t total = (int32_t)scene->getSampler()->getSampleCount();
        const int32_t s0 = std::max(0, scene->sppBegin), s1 = scene->sppEnd < 0 ? total : std::min(total, scene->sppEnd);
        if (s0 >= s1) throw Exception("GPU integrator: empty sample range");
        int32_t clear = 1;
        if (!scene->resumeFrame.empty()) {      /* the frame is a sum over sample indices: keep adding to a saved one */
            std::ifstream f(scene->resumeFrame, std::ios::binary);
            int32_t hdr[3] = {0, 0, 0};
            f.read((char *)hdr, sizeof(hdr));
            if (!f || hdr[0] != w || hdr[1] != h || hdr[2] != b) throw Exception("resume frame \"" + scene->resumeFrame + "\" does not match this camera / filter");
            f.read((char *)result.data.data(), (std::streamsize)(result.data.size() * sizeof(float)));
            if (!f) throw Exception("resume frame \"" + scene->resumeFrame + "\" is truncated");
            clear = 0;
        }
        kz_render_req req{0, 0, w, h, s0, s1, clear};
        if (kzgpu_render(m_ctx, &req, result.data.data()) != KZ_OK) throw Exception(std::string("GPU integrator: render failed: ") + kzgpu_last_error(m_ctx));
        return true;
    }
    kzgpu_ctx *context() const { return m_ctx; }
    std::string toString() const override {
        static const char *names[] = {"GpuPathMisIntegrator", "GpuNormalIntegrator", "GpuAmbientOcclusionIntegrator", "GpuWhittedIntegrator", "GpuPathMatsIntegrator"};
        return fmt("%s[maxDepth=%d, traceBias=%g, regularization=%d, textureFiltering=%d, envSampling=%d]", names[m_desc.type], m_desc.max_depth, m_desc.trace_bias,
                   m_desc.regularization, m_desc.texture_filtering, m_desc.env_sampling);
    }
private:
    kz_integrator_desc m_desc; kzgpu_ctx *m_ctx = nullptr;
};
KAZEN_REGISTER_CLASS(GpuPathMisIntegrator, "path_mis");
/* SURVEY 8(f)-3: the other integrators run through the same wavefront (integrator.cpp:11-181) */
#define KZ_ALT_INTEGRATOR(cls, name, type)                                                                         \
    class cls : public GpuPathMisIntegrator { public: cls(const PropertyList &p) : GpuPathMisIntegrator(p, type) {} };   \
    KAZEN_REGISTER_CLASS(cls, name)
KZ_ALT_INTEGRATOR(GpuNormalIntegrator, "normals", KZ_INTEGRATOR_NORMALS)
KZ_ALT_INTEGRATOR(GpuAmbientOcclusionIntegrator, "ao", KZ_INTEGRATOR_AO)
KZ_ALT_INTEGRATOR(GpuWhittedIntegrator, "whitted", KZ_INTEGRATOR_WHITTED)
KZ_ALT_INTEGRATOR(GpuPathMatsIntegrator, "path_mats", KZ_INTEGRATOR_PATH_MATS)

namespace renderer {
void render(Scene *scene, const std::string &outputName, bool writeRaw) {
    Integrator *integrator = scene->getIntegrator();
    const auto t0 = std::chrono::steady_clock::now();
    integrator->preprocess(scene);
    const auto t1 = std::chrono::steady_clock::now();
    ImageBlock result;
    if (!integrator->renderFrame(scene, result))
        throw Exception("integrator \"" + integrator->toString() + "\" has no whole-frame GPU implementation and this build has no CPU tile loop");
    const auto t2 = std::chrono::steady_clock::now();
    std::cout << "Scene upload + accel build took " << std::chrono::duration<double, std::milli>(t1 - t0).count() << " ms" << std::endl;
    const double ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
    const int sppTotal = (int)scene->getSampler()->getSampleCount();
    const double paths = (double)result.width * result.height * ((scene->sppEnd < 0 ? sppTotal : std::min(sppTotal, scene->sppEnd)) - std::max(0, scene->sppBegin));
    std::cout << "Render ready. (took " << ms << " ms, " << paths / ms / 1e3 << " Mpaths/s)" << std::endl;
    GpuPathMisIntegrator *g = dynamic_cast<GpuPathMisIntegrator *>(integrator);
    std::vector<uint8_t> srgb((size_t)result.width * result.height * 3);
    std::vector<float> linear((size_t)result.width * result.height * 3, 0.f);
    if (g && g->context()) {
        if (kzgpu_resolve(g->context(), result.data.data(), linear.data(), srgb.data()) != KZ_OK) throw Exception(std::string("resolve failed: ") + kzgpu_last_error(g->context()));
        kz_stats st;
        if (kzgpu_stats(g->context(), &st) == KZ_OK)
            std::cout << "paths " << st.paths << ", extension rays " << st.rays_extension << ", shadow rays " << st.rays_shadow << ", vertices " << st.vertices
                      << ", kernel launches " << st.kernel_launches << ", trace " << st.ms_trace << " ms, shade " << st.ms_shade << " ms, frame merge over NVLink "
                      << st.ms_merge << " ms, scene upload " << st.ms_upload << " ms, accel build " << st.ms_build << " ms, accel " << st.bvh_nodes
                      << " nodes / " << st.bvh_bytes / 1048576.0 << " MiB" << std::endl;
    }
    writePNG(outputName + ".png", result.width, result.height, srgb.data());
    writeEXR(outputName + ".exr", result.width, result.height, linear.data());
    if (writeRaw) {
        std::ofstream f(outputName + ".rgbw", std::ios::binary);
        const int32_t hdr[3] = {result.width, result.height, result.border};
        f.write((const char *)hdr, sizeof(hdr));
        f.write((const char *)result.data.data(), (std::streamsize)(result.data.size() * sizeof(float)));
    }
    std::cout << "Wrote " << outputName << ".png and " << outputName << ".exr" << std::endl;
}
}  // namespace renderer

class SceneObject : public Scene { public: SceneObject(const PropertyList &p) : Scene(p) {} };
KAZEN_REGISTER_CLASS(SceneObject, "scene");

}  // namespace kazen
