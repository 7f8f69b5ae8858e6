// Test driver: the frame drop-in hvo_shim::FrameExtractorGPU (shim/FrameExtractorGPU.h) against the per-class drop-ins.  Each frame
// is built twice into the stand-in Frame (tests/cpp/standins/frame_standin.hpp):
//   (a) FrameExtractorGPU::extract, one frame call;
//   (b) the per-class shims in the reference's order: ORBextractor, hvo_shim::undistortKeyPoints, the depth lookup of
//       Frame::ComputeStereoFromRGBD and hvo_stereo_uright_from_depth; LineFrontEnd::extract + cullingLine; PlaneDetection;
//       hvo_normals_compute_batch; the hvo_proj / hvo_lproj grids with hvo_shim::computeImageBounds; BowTransformerT; LpvoNormals.
//   in.bin : int32 magic, w, h, nframes, nfeatures, nlevels, iniThFAST, minThFAST, nLSDFeature, max_planes, want_lpvo, mode,
//            n_nodes (0 = no vocabulary), voc_L ; float scaleFactor, fx, fy, cx, cy, k1, k2, p1, p2, k3, bf, depth_factor ;
//            per frame gray [h][w] u8, depth [h][w] u16 ; with a vocabulary child_start [n+1] i32, nchild i32, child_ids [nchild] i32,
//            node_desc [n][32] u8, node_weight [n] f64, node_word [n] i32.
//            mode 0: the images as given; 1: the depth handed over as CV_16SC1; 2: the gray image one column narrower.
//   out.bin: per frame int32 ok (what extract returned), frame (a), and when ok frame (b).  A frame is
//            float mnMinX, mnMaxX, mnMinY, mnMaxY, mfGridElementWidthInv, mfGridElementHeightInv ;
//            int32 N ; N x 28 B mvKeys ; N x 28 B mvKeysUn ; int32 rows, cols, type of mDescriptors ; rows x 32 B ; N float mvDepth ;
//            N float mvuRight ;
//            int32 NL ; NL x 68 B mvKeylinesUn ; int32 rows, cols, type of mLdesc ; rows x 32 B ; NL x 3 double mvKeyLineFunctions ;
//            int32 plane_num_ ; per plane 3 double normal, 3 double center, int32 N, int32 nv, nv int32 plane_vertices_,
//            nv x 3 double cloud.vertices of those pixels ;
//            int32 n ; n x {3 float normal, 3 float cameraPosition, 2 int32 FramePosition} vSurfaceNormal ;
//            mGrid, then mGridForLine: 3072 int32 cell sizes (cell = ix * 48 + iy), then the cells' entries as int32 ;
//            int32 n ; n x (uint32 word, double value) mBowVec ; int32 n ; per node uint32 node, int32 k, k uint32 features (mFeatVec) ;
//            with want_lpvo: int32 n ; n x 3 double pt_normals ; n float depth_normals.
//   With a third argument reps: frame 0 only, reps times extract and then the bare blocking frame call with the same outputs on the same
//   handle; out.bin = int32 reps, then reps doubles each of extract seconds, fill seconds (lastFillSeconds) and frame-call seconds.
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <vector>

#include "frame_standin.hpp"
#include "FrameExtractorGPU.h"
#include "LineExtractorGPU.h"
#include "ORBextractor.h"
#include "WindowedMatcherGPU.h"

using ORB_SLAM2::Frame;

float Frame::mnMinX = 0.f, Frame::mnMaxX = 0.f, Frame::mnMinY = 0.f, Frame::mnMaxY = 0.f;
float Frame::mfGridElementWidthInv = 0.f, Frame::mfGridElementHeightInv = 0.f;

// The members of DBoW2::TemplatedVocabulary that VocabularyArrays reads, loaded from the arrays hvo_bow_set_vocabulary takes.
class ArrayVocabulary {
public:
    ArrayVocabulary(int n, int L, const std::vector<int32_t>& child_start, const std::vector<int32_t>& child_ids, const std::vector<uint8_t>& desc,
                    const std::vector<double>& weight, const std::vector<int32_t>& word) {
        m_nodes.resize(n);
        for (int i = 0; i < n; ++i) {
            for (int c = child_start[i]; c < child_start[i + 1]; ++c) m_nodes[i].children.push_back((unsigned)child_ids[c]);
            if (i > 0) {
                m_nodes[i].descriptor = cv::Mat(1, 32, CV_8U);
                std::memcpy(m_nodes[i].descriptor.ptr(), &desc[(size_t)i * 32], 32);
            }
            m_nodes[i].weight = weight[i];
            m_nodes[i].word_id = word[i] >= 0 ? (unsigned)word[i] : 0u;
        }
        m_L = L;
    }

protected:
    struct Node {
        std::vector<unsigned> children;
        cv::Mat descriptor;
        double weight = 0;
        unsigned word_id = 0;
        bool isLeaf() const { return children.empty(); }
    };
    std::vector<Node> m_nodes;
    int m_L = 0;
};

template <class T>
static void put(FILE* fo, const T& v) { std::fwrite(&v, sizeof(T), 1, fo); }
static void putMat(FILE* fo, const cv::Mat& m) {
    put(fo, (int32_t)m.rows); put(fo, (int32_t)m.cols); put(fo, (int32_t)(m.empty() ? 0 : m.type()));
    for (int i = 0; i < m.rows; ++i) std::fwrite(m.ptr(i), 1, 32, fo);
}
static void putGrid(FILE* fo, const std::vector<std::size_t> (&g)[64][48]) {
    for (int ix = 0; ix < 64; ++ix)
        for (int iy = 0; iy < 48; ++iy) put(fo, (int32_t)g[ix][iy].size());
    for (int ix = 0; ix < 64; ++ix)
        for (int iy = 0; iy < 48; ++iy)
            for (std::size_t v : g[ix][iy]) put(fo, (int32_t)v);
}

static void writeFrame(FILE* fo, const Frame& F, const float bounds[6], bool lpvo, const std::vector<double>& ptNormals, const std::vector<float>& depthNormals) {
    std::fwrite(bounds, 4, 6, fo);
    put(fo, (int32_t)F.N);
    std::fwrite(F.mvKeys.data(), 28, F.mvKeys.size(), fo);
    std::fwrite(F.mvKeysUn.data(), 28, F.mvKeysUn.size(), fo);
    putMat(fo, F.mDescriptors);
    std::fwrite(F.mvDepth.data(), 4, F.mvDepth.size(), fo);
    std::fwrite(F.mvuRight.data(), 4, F.mvuRight.size(), fo);
    put(fo, (int32_t)F.NL);
    std::fwrite(F.mvKeylinesUn.data(), 68, F.mvKeylinesUn.size(), fo);
    putMat(fo, F.mLdesc);
    for (const auto& v : F.mvKeyLineFunctions) std::fwrite(v.v, 8, 3, fo);
    const PlaneDetection& P = F.planeDetector;
    put(fo, (int32_t)P.plane_num_);
    for (int i = 0; i < P.plane_num_; ++i) {
        std::fwrite(P.plane_filter.extractedPlanes[i]->normal, 8, 3, fo);
        std::fwrite(P.plane_filter.extractedPlanes[i]->center, 8, 3, fo);
        put(fo, (int32_t)P.plane_filter.extractedPlanes[i]->N);
        put(fo, (int32_t)P.plane_vertices_[i].size());
        std::fwrite(P.plane_vertices_[i].data(), 4, P.plane_vertices_[i].size(), fo);
        for (int j : P.plane_vertices_[i]) std::fwrite(P.cloud.vertices[j].v, 8, 3, fo);
    }
    put(fo, (int32_t)F.vSurfaceNormal.size());
    for (const auto& s : F.vSurfaceNormal) {
        const float e[6] = {s.normal.x, s.normal.y, s.normal.z, s.cameraPosition.x, s.cameraPosition.y, s.cameraPosition.z};
        std::fwrite(e, 4, 6, fo);
        put(fo, (int32_t)s.FramePosition.x); put(fo, (int32_t)s.FramePosition.y);
    }
    putGrid(fo, F.mGrid);
    putGrid(fo, F.mGridForLine);
    put(fo, (int32_t)F.mBowVec.size());
    for (const auto& e : F.mBowVec) { put(fo, (uint32_t)e.first); put(fo, (double)e.second); }
    put(fo, (int32_t)F.mFeatVec.size());
    for (const auto& e : F.mFeatVec) {
        put(fo, (uint32_t)e.first); put(fo, (int32_t)e.second.size());
        std::fwrite(e.second.data(), 4, e.second.size(), fo);
    }
    if (lpvo) {
        put(fo, (int32_t)depthNormals.size());
        std::fwrite(ptNormals.data(), 8, ptNormals.size(), fo);
        std::fwrite(depthNormals.data(), 4, depthNormals.size(), fo);
    }
}

int main(int argc, char** argv) {
    if (argc != 3 && argc != 4) { std::fprintf(stderr, "usage: shim_frame in.bin out.bin [reps]\n"); return 2; }
    FILE* fi = std::fopen(argv[1], "rb");
    FILE* fo = std::fopen(argv[2], "wb");
    if (!fi || !fo) return 2;
    int32_t hd[14];
    float pf[12];
    if (std::fread(hd, 4, 14, fi) != 14 || hd[0] != 0x444d5246 || std::fread(pf, 4, 12, fi) != 12) return 3;
    const int w = hd[1], h = hd[2], nf = hd[3], nfeat = hd[4], nlevels = hd[5], ini = hd[6], mn = hd[7], nlsd = hd[8], maxPlanes = hd[9];
    const bool wantLpvo = hd[10] != 0;
    const int mode = hd[11], nnodes = hd[12], vocL = hd[13];
    const float scale = pf[0], fx = pf[1], fy = pf[2], cx = pf[3], cy = pf[4], bf = pf[10], df = pf[11];
    const size_t px = (size_t)w * h;
    std::vector<uint8_t> gray(px * nf);
    std::vector<uint16_t> depth(px * nf);
    for (int f = 0; f < nf; ++f)
        if (std::fread(&gray[px * f], 1, px, fi) != px || std::fread(&depth[px * f], 2, px, fi) != px) return 4;
    std::unique_ptr<ArrayVocabulary> voc;
    if (nnodes > 0) {
        std::vector<int32_t> cs(nnodes + 1), ids, word(nnodes);
        std::vector<uint8_t> desc((size_t)nnodes * 32);
        std::vector<double> weight(nnodes);
        int32_t nchild = 0;
        if (std::fread(cs.data(), 4, cs.size(), fi) != cs.size() || std::fread(&nchild, 4, 1, fi) != 1) return 4;
        ids.resize(nchild);
        if (std::fread(ids.data(), 4, ids.size(), fi) != ids.size() || std::fread(desc.data(), 1, desc.size(), fi) != desc.size() ||
            std::fread(weight.data(), 8, weight.size(), fi) != weight.size() || std::fread(word.data(), 4, word.size(), fi) != word.size())
            return 4;
        voc.reset(new ArrayVocabulary(nnodes, vocL, cs, ids, desc, weight, word));
    }
    std::fclose(fi);

    // mK and mDistCoef as Tracking holds them (CV_32F; five coefficients)
    cv::Mat K(3, 3, CV_32F), D(5, 1, CV_32F);
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) K.at<float>(i, j) = 0.f;
    K.at<float>(0, 0) = fx; K.at<float>(1, 1) = fy; K.at<float>(0, 2) = cx; K.at<float>(1, 2) = cy; K.at<float>(2, 2) = 1.f;
    for (int i = 0; i < 5; ++i) D.at<float>(i) = pf[5 + i];

    hvo_shim::FrameExtractorGPU fe(w, h, nfeat, scale, nlevels, ini, mn, 1, 1.2f, (unsigned)nlsd, 0.125, K, D, bf, df, maxPlanes);
    if (voc) fe.setVocabulary(*voc, 4);

    if (argc == 4) {
        const int reps = std::atoi(argv[3]);
        hvo_frame* hf = fe.handle();
        if (!hf || reps < 1) return 5;
        cv::Mat img(h, w, CV_8UC1, gray.data(), (size_t)w), dimg(h, w, CV_16UC1, depth.data(), (size_t)w * 2);
        // the bare call asks for the outputs extract asks for
        int oc = 0, ml = 0, nc = 0;
        hvo_frame_capacities(hf, &oc, &ml, &nc);
        const int lgc = hvo_frame_line_grid_capacity(hf), lc = hvo_frame_lpvo_capacity(hf);
        const bool undist = pf[5] != 0.f || pf[6] != 0.f || pf[7] != 0.f || pf[8] != 0.f || pf[9] != 0.f;
        std::vector<hvo_keypoint> kps(oc), kpsun(oc);
        std::vector<uint8_t> desc((size_t)oc * 32), ldesc((size_t)ml * 32), lab8(px);
        std::vector<int32_t> lab32(maxPlanes <= 254 ? 0 : px), bw(oc), fvo(oc), nof(oc);
        std::vector<float> kd(oc), ku(oc), n3((size_t)nc * 3), ld(lc);
        std::vector<hvo_keyline> kl(ml);
        std::vector<double> lv((size_t)ml * 3), p7((size_t)maxPlanes * 7), bv(oc), ln((size_t)lc * 3);
        std::vector<uint16_t> gc(3072), gi(oc), lgcnt(3072), lgi(lgc);
        int32_t nkp = 0, nl = 0, np = 0, bc = 0, fc = 0, lcnt = 0;
        hvo_frame_outputs o;
        std::memset(&o, 0, sizeof(o));
        o.kps = kps.data(); o.desc = desc.data(); o.kp_counts = &nkp; o.kp_depth = kd.data(); o.kp_uright = ku.data(); o.kps_un = undist ? kpsun.data() : nullptr;
        o.keylines = kl.data(); o.line_desc = ldesc.data(); o.linevec3 = lv.data(); o.line_counts = &nl; o.n_planes = &np; o.planes7 = p7.data();
        if (maxPlanes <= 254) o.membership8 = lab8.data(); else o.membership = lab32.data();
        o.normals3 = n3.data();
        hvo_frame_bow_outputs b = {&bc, bw.data(), bv.data(), fvo.data(), &fc, nof.data(), nullptr};
        hvo_frame_grid_outputs g = {gc.data(), gi.data(), lgcnt.data(), lgi.data()};
        hvo_frame_lpvo_outputs lp = {ln.data(), ld.data(), nullptr, &lcnt};
        std::vector<double> te(reps), tf(reps), tc(reps);
        for (int r = 0; r < reps; ++r) {
            std::unique_ptr<Frame> F(new Frame);
            std::vector<cv::Mat> ptN;
            std::vector<float> dN;
            auto t0 = std::chrono::steady_clock::now();
            if (!fe.extract(img, dimg, *F, wantLpvo, &ptN, &dN)) return 6;
            auto t1 = std::chrono::steady_clock::now();
            if (hvo_frame_extract_batch_lpvo(hf, gray.data(), depth.data(), 1, &o, voc ? &b : nullptr, &g, wantLpvo ? &lp : nullptr) != HVO_OK) return 7;
            auto t2 = std::chrono::steady_clock::now();
            te[r] = std::chrono::duration<double>(t1 - t0).count();
            tf[r] = fe.lastFillSeconds();
            tc[r] = std::chrono::duration<double>(t2 - t1).count();
        }
        put(fo, (int32_t)reps);
        std::fwrite(te.data(), 8, reps, fo);
        std::fwrite(tf.data(), 8, reps, fo);
        std::fwrite(tc.data(), 8, reps, fo);
        std::fclose(fo);
        return 0;
    }

    // the per-class drop-ins of (b), one per Tracking as the reference holds them
    std::unique_ptr<ORB_SLAM2::ORBextractor> orb;
    std::unique_ptr<hvo_shim::LineFrontEnd> lines;
    std::unique_ptr<hvo_shim::BowTransformerT<ArrayVocabulary>> bow;
    std::unique_ptr<hvo_shim::LpvoNormals> lpvo;
    hvo_normals* nh = nullptr;
    hvo_proj* ph = nullptr;
    hvo_lproj* lh = nullptr;
    int ncount = 0;

    for (int f = 0; f < nf; ++f) {
        uint8_t* gf = &gray[px * f];
        uint16_t* dfr = &depth[px * f];
        cv::Mat img(h, w, CV_8UC1, gf, (size_t)w), dimg(h, w, CV_16UC1, dfr, (size_t)w * 2);
        const cv::Mat imgArg = mode == 2 ? cv::Mat(h, w - 1, CV_8UC1, gf, (size_t)w) : img;
        const cv::Mat depArg = mode == 1 ? cv::Mat(h, w, CV_16SC1, dfr, (size_t)w * 2) : dimg;

        // (a)
        std::unique_ptr<Frame> A(new Frame);
        std::vector<cv::Mat> ptN;
        std::vector<float> dN;
        const bool ok = fe.extract(imgArg, depArg, *A, wantLpvo, &ptN, &dN);
        std::vector<double> nrm;
        for (const cv::Mat& m : ptN) for (int k = 0; k < 3; ++k) nrm.push_back(m.at<double>(k));
        const float ba[6] = {Frame::mnMinX, Frame::mnMaxX, Frame::mnMinY, Frame::mnMaxY, Frame::mfGridElementWidthInv, Frame::mfGridElementHeightInv};
        put(fo, (int32_t)ok);
        writeFrame(fo, *A, ba, wantLpvo, nrm, dN);
        if (!ok) continue;

        // (b)
        if (!orb) {
            orb.reset(new ORB_SLAM2::ORBextractor(nfeat, scale, nlevels, ini, mn));
            lines.reset(new hvo_shim::LineFrontEnd(1, 1.2f, (unsigned)nlsd, 0.125));
            if (voc) bow.reset(new hvo_shim::BowTransformerT<ArrayVocabulary>(*voc));
            if (wantLpvo) lpvo.reset(new hvo_shim::LpvoNormals(fx, fy, cx, cy, df, w, h));
            const hvo_normals_params np = {fx, fy, cx, cy, df, 0.05f, 10.0f};   // Frame.cc:2179-2180
            if (hvo_normals_create(&np, w, h, 1, 0, &nh) != HVO_OK || hvo_proj_create(0, &ph) != HVO_OK || hvo_lproj_create(0, &lh) != HVO_OK) {
                std::fprintf(stderr, "shim_frame: %s\n", hvo_last_error());
                return 8;
            }
            ncount = hvo_normals_count(nh);
        }
        std::unique_ptr<Frame> B(new Frame);
        // thread A: ExtractORBNDepth, UndistortKeyPoints, ComputeStereoFromRGBD (Frame.cc:874-884, 1701-1731, 1940-1961)
        (*orb)(img, cv::Mat(), B->mvKeys, B->mDescriptors);
        const int N = (int)B->mvKeys.size();
        B->N = N;
        hvo_shim::undistortKeyPoints(B->mvKeys, K, D, B->mvKeysUn);
        B->mvDepth.assign(N, -1.f);
        for (int i = 0; i < N; ++i) {   // depth at the distorted keypoint, valid in (0, 7) m
            const int u = std::min((int)B->mvKeys[i].pt.x, w - 1), v = std::min((int)B->mvKeys[i].pt.y, h - 1);
            const float d = (float)dfr[(size_t)v * w + u] * df;
            if (d > 0.f && d < 7.0f) B->mvDepth[i] = d;
        }
        B->mvuRight.resize(N);
        if (hvo_stereo_uright_from_depth(reinterpret_cast<const hvo_keypoint*>(B->mvKeysUn.data()), B->mvDepth.data(), N, bf, B->mvuRight.data()) != HVO_OK) return 9;
        // thread B: ExtractLSD = LINEextractor::operator() + cullingLine (Frame.cc:895-950)
        lines->extract(img, B->mvKeylinesUn, B->mLdesc, B->mvKeyLineFunctions);
        lines->cullingLine(img, B->mvKeylinesUn, B->mLdesc, B->mvKeyLineFunctions);
        B->NL = (int)B->mvKeylinesUn.size();
        // thread C: ComputePlanes (Frame.cc:2104-2212)
        if (!B->planeDetector.readDepthImage(dimg, K, df)) return 10;
        B->planeDetector.runPlaneDetection(h, w);
        std::vector<float> out8((size_t)ncount * 8);
        if (hvo_normals_compute_batch(nh, dfr, 1, out8.data()) != HVO_OK) return 11;
        B->vSurfaceNormal.resize(ncount);
        for (int i = 0; i < ncount; ++i) hvo_shim::setSurfaceNormal(B->vSurfaceNormal[i], &out8[(size_t)i * 8]);
        // the grid threads (Frame.cc:304-307, 832-872), with ComputeImageBounds and the first frame's cell inverses (:101-107)
        float bb[6];
        hvo_shim::computeImageBounds(K, D, w, h, bb[0], bb[1], bb[2], bb[3]);
        bb[4] = static_cast<float>(FRAME_GRID_COLS) / static_cast<float>(bb[1] - bb[0]);
        bb[5] = static_cast<float>(FRAME_GRID_ROWS) / static_cast<float>(bb[3] - bb[2]);
        if (N > 0) {
            std::vector<uint8_t> desc((size_t)N * 32);
            for (int i = 0; i < N; ++i) std::memcpy(&desc[(size_t)i * 32], B->mDescriptors.ptr(i), 32);
            std::vector<int32_t> start(3073), items(N);
            if (hvo_proj_set_frame(ph, reinterpret_cast<const hvo_keypoint*>(B->mvKeysUn.data()), B->mvuRight.data(), desc.data(), N, bb[0], bb[2], bb[1],
                                   bb[3]) != HVO_OK || hvo_proj_get_grid(ph, start.data(), items.data()) != HVO_OK) return 12;
            for (int c = 0; c < 3072; ++c) B->mGrid[c / 48][c % 48].assign(items.begin() + start[c], items.begin() + start[c + 1]);
        }
        if (B->NL > 0) {
            const int nl = B->NL;
            std::vector<uint8_t> ld((size_t)nl * 32);
            std::vector<double> fn((size_t)nl * 3);
            for (int i = 0; i < nl; ++i) {
                std::memcpy(&ld[(size_t)i * 32], B->mLdesc.ptr(i), 32);
                for (int k = 0; k < 3; ++k) fn[(size_t)i * 3 + k] = B->mvKeyLineFunctions[i][k];
            }
            std::vector<int32_t> cnt(3072), items((size_t)nl * 64);
            int nitems = 0;
            if (hvo_lproj_set_frame(lh, reinterpret_cast<const hvo_keyline*>(B->mvKeylinesUn.data()), fn.data(), ld.data(), nullptr, nl, bb[0], bb[2], bb[1],
                                    bb[3]) != HVO_OK || hvo_lproj_get_grid(lh, cnt.data(), items.data(), (int)items.size(), &nitems) != HVO_OK) return 13;
            size_t o = 0;
            for (int c = 0; c < 3072; ++c) { B->mGridForLine[c / 48][c % 48].assign(items.begin() + o, items.begin() + o + cnt[c]); o += cnt[c]; }
        }
        // Frame::ComputeBoW (Frame.cc:1692-1699)
        if (bow) {
            std::vector<cv::Mat> rows;
            for (int i = 0; i < N; ++i) rows.push_back(B->mDescriptors.row(i));
            bow->transform(rows, B->mBowVec, B->mFeatVec, 4);
        }
        // thread D: Manhattan::computeNormalsLPVO
        std::vector<double> bn;
        std::vector<float> bd;
        if (lpvo) {
            std::vector<int32_t> pix;
            lpvo->compute(dfr, bn, bd, pix);
        }
        writeFrame(fo, *B, bb, wantLpvo, bn, bd);
    }
    hvo_normals_destroy(nh);
    hvo_proj_destroy(ph);
    hvo_lproj_destroy(lh);
    std::fclose(fo);
    return 0;
}
