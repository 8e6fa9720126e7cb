/* tests/gt_sampling_box_ops.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * C restatement of the two compiled CPU ops that pcdet's gt_sampling (DataBaseSampler, OpenPCDet v0.5.2) calls:
 *   iou3d_nms/src/iou3d_cpu.cpp        boxes_iou_bev_cpu -> iou_bev -> box_overlap (rotated-BEV overlap area)
 *   roiaware_pool3d/src/roiaware_pool3d.cpp  points_in_boxes_cpu -> check_pt_in_box3d_cpu
 * Built by tests/gt_sampling_oracle.py with gcc -O2 -ffp-contract=off (no FMA contraction, as the reference's ops are compiled).
 * Boxes are float32 [x, y, z, dx, dy, dz, heading].  What the restatement keeps from the reference:
 *   - every intermediate is float32, op by op, in the reference's evaluation order;
 *   - cos / sin of a heading are libm cosf / sinf of the float32 angle (cos(a) for the corners of box_overlap, cos(-a)
 *     for check_in_box2d and for the point test);
 *   - check_in_box2d: |rot| < d / 2 + 1e-2 in float32;  intersection: fast rectangle exclusion, strict cross-sign
 *     test, |s5 - s1| > 1e-8 picks the formula;  point_cmp: atan2f of the offsets from the polygon centre, and the
 *     polygon is bubble-sorted with it;  area: fan from the first sorted point, fabs(area) / 2.0;
 *   - iou_bev = overlap / fmaxf(sa + sb - overlap, 1e-8);
 *   - check_pt_in_box3d_cpu: fabsf(z - cz) > dz / 2.0 and fabs(local) < d / 2.0 + MARGIN are evaluated in double (the
 *     literals promote them), the local coordinates in float32.
 */
#include <math.h>

#define EPS 1e-8f

typedef struct { float x, y; } Point;

static Point pt(float x, float y) { Point p; p.x = x; p.y = y; return p; }
static float fmin_ref(float a, float b) { return a > b ? b : a; }
static float fmax_ref(float a, float b) { return a > b ? a : b; }
static float cross2(Point a, Point b) { return a.x * b.y - a.y * b.x; }
static float cross3(Point p1, Point p2, Point p0) { return (p1.x - p0.x) * (p2.y - p0.y) - (p2.x - p0.x) * (p1.y - p0.y); }

static int check_rect_cross(Point p1, Point p2, Point q1, Point q2) {
    return fmin_ref(p1.x, p2.x) <= fmax_ref(q1.x, q2.x) && fmin_ref(q1.x, q2.x) <= fmax_ref(p1.x, p2.x) &&
           fmin_ref(p1.y, p2.y) <= fmax_ref(q1.y, q2.y) && fmin_ref(q1.y, q2.y) <= fmax_ref(p1.y, p2.y);
}

static int check_in_box2d(const float *box, Point p) {
    const float MARGIN = 1e-2f;
    float center_x = box[0], center_y = box[1];
    float angle_cos = cosf(-box[6]), angle_sin = sinf(-box[6]);
    float rot_x = (p.x - center_x) * angle_cos + (p.y - center_y) * (-angle_sin);
    float rot_y = (p.x - center_x) * angle_sin + (p.y - center_y) * angle_cos;
    return fabsf(rot_x) < box[3] / 2 + MARGIN && fabsf(rot_y) < box[4] / 2 + MARGIN;
}

static int intersection(Point p1, Point p0, Point q1, Point q0, Point *ans) {
    if (check_rect_cross(p0, p1, q0, q1) == 0) return 0;
    float s1 = cross3(q0, p1, p0);
    float s2 = cross3(p1, q1, p0);
    float s3 = cross3(p0, q1, q0);
    float s4 = cross3(q1, p1, q0);
    if (!(s1 * s2 > 0 && s3 * s4 > 0)) return 0;
    float s5 = cross3(q1, p1, p0);
    if (fabsf(s5 - s1) > EPS) {
        ans->x = (s5 * q0.x - s1 * q1.x) / (s5 - s1);
        ans->y = (s5 * q0.y - s1 * q1.y) / (s5 - s1);
    } else {
        float a0 = p0.y - p1.y, b0 = p1.x - p0.x, c0 = p0.x * p1.y - p1.x * p0.y;
        float a1 = q0.y - q1.y, b1 = q1.x - q0.x, c1 = q0.x * q1.y - q1.x * q0.y;
        float D = a0 * b1 - a1 * b0;
        ans->x = (b0 * c1 - b1 * c0) / D;
        ans->y = (a1 * c0 - a0 * c1) / D;
    }
    return 1;
}

static void rotate_around_center(Point center, float angle_cos, float angle_sin, Point *p) {
    float new_x = (p->x - center.x) * angle_cos + (p->y - center.y) * (-angle_sin) + center.x;
    float new_y = (p->x - center.x) * angle_sin + (p->y - center.y) * angle_cos + center.y;
    *p = pt(new_x, new_y);
}

static int point_cmp(Point a, Point b, Point center) {
    return atan2f(a.y - center.y, a.x - center.x) > atan2f(b.y - center.y, b.x - center.x);
}

float box_overlap(const float *box_a, const float *box_b) {
    float a_angle = box_a[6], b_angle = box_b[6];
    float a_dx_half = box_a[3] / 2, b_dx_half = box_b[3] / 2, a_dy_half = box_a[4] / 2, b_dy_half = box_b[4] / 2;
    float a_x1 = box_a[0] - a_dx_half, a_y1 = box_a[1] - a_dy_half;
    float a_x2 = box_a[0] + a_dx_half, a_y2 = box_a[1] + a_dy_half;
    float b_x1 = box_b[0] - b_dx_half, b_y1 = box_b[1] - b_dy_half;
    float b_x2 = box_b[0] + b_dx_half, b_y2 = box_b[1] + b_dy_half;
    Point center_a = pt(box_a[0], box_a[1]), center_b = pt(box_b[0], box_b[1]);
    Point ca[5], cb[5];
    ca[0] = pt(a_x1, a_y1); ca[1] = pt(a_x2, a_y1); ca[2] = pt(a_x2, a_y2); ca[3] = pt(a_x1, a_y2);
    cb[0] = pt(b_x1, b_y1); cb[1] = pt(b_x2, b_y1); cb[2] = pt(b_x2, b_y2); cb[3] = pt(b_x1, b_y2);
    float a_cos = cosf(a_angle), a_sin = sinf(a_angle);
    float b_cos = cosf(b_angle), b_sin = sinf(b_angle);
    for (int k = 0; k < 4; k++) {
        rotate_around_center(center_a, a_cos, a_sin, &ca[k]);
        rotate_around_center(center_b, b_cos, b_sin, &cb[k]);
    }
    ca[4] = ca[0];
    cb[4] = cb[0];
    Point cross_points[16];
    Point poly_center = pt(0, 0);
    int cnt = 0;
    for (int i = 0; i < 4; i++) {
        for (int j = 0; j < 4; j++) {
            if (intersection(ca[i + 1], ca[i], cb[j + 1], cb[j], &cross_points[cnt])) {
                poly_center = pt(poly_center.x + cross_points[cnt].x, poly_center.y + cross_points[cnt].y);
                cnt++;
            }
        }
    }
    for (int k = 0; k < 4; k++) {
        if (check_in_box2d(box_a, cb[k])) {
            poly_center = pt(poly_center.x + cb[k].x, poly_center.y + cb[k].y);
            cross_points[cnt] = cb[k];
            cnt++;
        }
        if (check_in_box2d(box_b, ca[k])) {
            poly_center = pt(poly_center.x + ca[k].x, poly_center.y + ca[k].y);
            cross_points[cnt] = ca[k];
            cnt++;
        }
    }
    poly_center.x /= cnt;
    poly_center.y /= cnt;
    for (int j = 0; j < cnt - 1; j++) {
        for (int i = 0; i < cnt - j - 1; i++) {
            if (point_cmp(cross_points[i], cross_points[i + 1], poly_center)) {
                Point temp = cross_points[i];
                cross_points[i] = cross_points[i + 1];
                cross_points[i + 1] = temp;
            }
        }
    }
    float area = 0;
    for (int k = 0; k < cnt - 1; k++) {
        Point d0 = pt(cross_points[k].x - cross_points[0].x, cross_points[k].y - cross_points[0].y);
        Point d1 = pt(cross_points[k + 1].x - cross_points[0].x, cross_points[k + 1].y - cross_points[0].y);
        area += cross2(d0, d1);
    }
    return (float)(fabsf(area) / 2.0);
}

static float iou_bev(const float *box_a, const float *box_b) {
    float sa = box_a[3] * box_a[4];
    float sb = box_b[3] * box_b[4];
    float s_overlap = box_overlap(box_a, box_b);
    return s_overlap / fmaxf(sa + sb - s_overlap, EPS);
}

/* ans_iou[i * nb + j] = iou_bev(boxes_a[i], boxes_b[j]) */
void boxes_iou_bev_cpu(const float *boxes_a, int na, const float *boxes_b, int nb, float *ans_iou) {
    for (int i = 0; i < na; i++)
        for (int j = 0; j < nb; j++) ans_iou[(long)i * nb + j] = iou_bev(boxes_a + i * 7, boxes_b + j * 7);
}

static int check_pt_in_box3d_cpu(const float *p, const float *box3d) {
    const float MARGIN = 1e-2f;
    float x = p[0], y = p[1], z = p[2];
    float cx = box3d[0], cy = box3d[1], cz = box3d[2];
    float dx = box3d[3], dy = box3d[4], dz = box3d[5], rz = box3d[6];
    if (fabsf(z - cz) > dz / 2.0) return 0;
    float cosa = cosf(-rz), sina = sinf(-rz);
    float shift_x = x - cx, shift_y = y - cy;
    float local_x = shift_x * cosa + shift_y * (-sina);
    float local_y = shift_x * sina + shift_y * cosa;
    return (fabs(local_x) < dx / 2.0 + MARGIN) & (fabs(local_y) < dy / 2.0 + MARGIN);
}

/* in_boxes[i] = number of boxes that contain point i (points: n rows of `stride` floats, x, y, z first); the
 * reference's points_in_boxes_cpu writes the (boxes, points) 0/1 matrix that remove_points_in_boxes3d sums over boxes */
void points_in_boxes_cpu(const float *boxes, int nb, const float *points, long n, int stride, int *in_boxes) {
    for (long i = 0; i < n; i++) {
        int c = 0;
        for (int j = 0; j < nb; j++) c += check_pt_in_box3d_cpu(points + i * stride, boxes + j * 7);
        in_boxes[i] = c;
    }
}
