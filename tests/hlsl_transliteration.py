"""Line-by-line Python transliteration of the reference's in-tree traversal shader, written independently of oracle/:
/root/reference/src/rt_gpu/rt_gpu_software_query.hlsl — cwbvh_node_intersect (213-303), ray_get_octant_inv4 (314-326),
traverse_bvh (328-438), intersect_ray_tri (89-129) — with ONE substitution: triangles are the f32 {v0, e1, e2} records of
the CPU path instead of the shader's f16 edges (unpack_triangle).  Every float operation is a separately rounded IEEE
binary32 operation (numpy.float32 scalars), as HLSL without fast-math evaluates them; dot / cross use the association
x*x' + y*y' + z*z' and a.yzx*b.zxy - a.zxy*b.yzx.  Test infrastructure only (slow: a few hundred rays per second)."""
import numpy as np

f32 = np.float32
F32_MAX = f32(3.402823466e+38)
F32_EPSILON = f32(1.1920929e-7)          # sampling.hlsl:3


def asfloat(u):
    return np.array([u & 0xffffffff], dtype=np.uint32).view(np.float32)[0]


def asuint(f):
    return int(np.array([f], dtype=np.float32).view(np.uint32)[0])


def extract_byte(x, b):                                               # :199-202
    return (x >> (b * 8)) & 0xff


def firstbithigh(x):
    return x.bit_length() - 1


def dot(a, b):
    return f32(f32(f32(a[0] * b[0]) + f32(a[1] * b[1])) + f32(a[2] * b[2]))


def cross(a, b):
    return (f32(f32(a[1] * b[2]) - f32(a[2] * b[1])), f32(f32(a[2] * b[0]) - f32(a[0] * b[2])), f32(f32(a[0] * b[1]) - f32(a[1] * b[0])))


class Scene:
    def __init__(self, nodes_bytes, tri_bytes, tri_stride, blas_offsets=None, tlas_start=0):
        self.nodes = np.frombuffer(bytes(nodes_bytes), dtype=np.uint32).reshape(-1, 20)        # uint4 data[5]
        self.tris = np.frombuffer(bytes(tri_bytes), dtype=np.float32).reshape(-1, tri_stride // 4)
        self.blas_offsets = None if blas_offsets is None else [int(x) for x in blas_offsets]
        self.tlas_start = int(tlas_start)


def cwbvh_node_intersect(org, d, oct_inv4, max_distance, node):     # :213-303
    with np.errstate(all="ignore"):
        p = [asfloat(int(node[k])) for k in range(3)]
        e_imask = int(node[3])
        e = [extract_byte(e_imask, k) for k in range(3)]
        adjusted_ray_dir_inv = [f32(asfloat(e[k] << 23) / d[k]) for k in range(3)]            # :237-241
        adjusted_ray_origin = [f32(f32(p[k] - org[k]) / d[k]) for k in range(3)]             # :242
        hit_mask = 0
        for i in range(2):
            meta4 = int(node[6 + i])                                                          # data[1].z / .w
            is_inner4 = (meta4 & (meta4 << 1)) & 0x10101010
            inner_mask4 = ((is_inner4 >> 4) * 0xff) & 0xffffffff
            bit_index4 = (meta4 ^ (oct_inv4 & inner_mask4)) & 0x1f1f1f1f
            child_bits4 = (meta4 >> 5) & 0x07070707
            q_lo = [int(node[8 + 4 * k + i]) for k in range(3)]                              # data[2+k].x / .y
            q_hi = [int(node[8 + 4 * k + 2 + i]) for k in range(3)]                          # data[2+k].z / .w
            q_min = [q_hi[k] if d[k] < 0.0 else q_lo[k] for k in range(3)]                   # :266-273
            q_max = [q_lo[k] if d[k] < 0.0 else q_hi[k] for k in range(3)]
            EPSILON = f32(0.0001)
            for j in range(4):
                tmin3 = [f32(f32(f32(extract_byte(q_min[k], j)) * adjusted_ray_dir_inv[k]) + adjusted_ray_origin[k]) for k in range(3)]
                tmax3 = [f32(f32(f32(extract_byte(q_max[k], j)) * adjusted_ray_dir_inv[k]) + adjusted_ray_origin[k]) for k in range(3)]
                tmin = max4(tmin3[0], tmin3[1], tmin3[2], EPSILON)
                tmax = min4(tmax3[0], tmax3[1], tmax3[2], max_distance)
                if tmin <= tmax:
                    hit_mask |= (extract_byte(child_bits4, j) << extract_byte(bit_index4, j)) & 0xffffffff
        return hit_mask


def _max(a, b):          # HLSL max: a NaN operand yields the other one
    if np.isnan(a):
        return b
    if np.isnan(b):
        return a
    return a if a > b else b


def _min(a, b):
    if np.isnan(a):
        return b
    if np.isnan(b):
        return a
    return a if a < b else b


def max4(a, b, c, d):
    return _max(_max(_max(a, b), c), d)


def min4(a, b, c, d):
    return _min(_min(_min(a, b), c), d)


def ray_get_octant_inv4(d):                                           # :314-326
    return (0 if d[0] < 0.0 else 0x04040404) | (0 if d[1] < 0.0 else 0x02020202) | (0 if d[2] < 0.0 else 0x01010101)


def intersect_ray_tri(org, d, v0, e1_stored, e2, t):                  # :89-129; returns the new t or None
    with np.errstate(all="ignore"):
        e1 = e1_stored                      # the record holds e1 = v0 - v1 = -(v1 - v0): the shader's `-tri.e1` (:91)
        ng = cross(e1, e2)
        c = [f32(v0[k] - org[k]) for k in range(3)]
        r = cross(d, c)
        inv_det = f32(f32(1.0) / dot(ng, d))
        u = f32(dot(r, e2) * inv_det)
        v = f32(dot(r, e1) * inv_det)
        w = f32(f32(f32(1.0) - u) - v)
        hit = asuint(u) | asuint(v) | asuint(w)
        if inv_det != 0.0 and (hit & 0x80000000) == 0:
            tt = f32(dot(ng, c) * inv_det)
            if tt >= 0.0 and tt <= t:                                 # :119-120: an equal t replaces the earlier hit
                return tt
    return None


def traverse_bvh(scene, origin, direction, stack_peak=False):         # :328-438; returns (t, triangle_id, nodes, tris)
    """stack_peak=True: the tuple ends with the most entries the stack held at once"""
    org = [f32(x) for x in origin]
    d = [f32(x) for x in direction]
    d = [F32_EPSILON if x == 0.0 else x for x in d]                   # :334
    stack = []
    oct_inv4 = ray_get_octant_inv4(d)
    current_group = [0, 0x80000000]
    t, triangle_id = F32_MAX, -1
    n_nodes = n_tris = peak = 0
    while True:
        if current_group[1] & 0xff000000:
            hits_imask = current_group[1]
            child_index_offset = firstbithigh(hits_imask)
            child_index_base = current_group[0]
            current_group[1] &= ~(1 << child_index_offset) & 0xffffffff
            if current_group[1] & 0xff000000:
                stack.append(list(current_group))
                peak = max(peak, len(stack))
            slot_index = (child_index_offset - 24) ^ (oct_inv4 & 0xff)
            relative_index = bin(hits_imask & ~(0xffffffff << slot_index) & 0xffffffff).count("1")
            node = scene.nodes[child_index_base + relative_index]
            n_nodes += 1
            hitmask = cwbvh_node_intersect(org, d, oct_inv4, t, node)
            imask = extract_byte(int(node[3]), 3)
            current_group[0] = int(node[4])
            triangle_group = [int(node[5]), hitmask & 0x00ffffff]
            current_group[1] = (hitmask & 0xff000000) | imask
        else:
            triangle_group = list(current_group)
            current_group = [0, 0]
        while triangle_group[1] != 0:
            local = firstbithigh(triangle_group[1])
            triangle_group[1] &= ~(1 << local) & 0xffffffff
            g = triangle_group[0] + local
            rec = scene.tris[g]
            n_tris += 1
            tt = intersect_ray_tri(org, d, rec[0:3], rec[4:7], rec[8:11], t)
            if tt is not None:
                t, triangle_id = tt, g
        if (current_group[1] & 0xff000000) == 0:
            if not stack:
                break
            current_group = stack.pop()
    return (t, triangle_id, n_nodes, n_tris) + ((peak,) if stack_peak else ())


INVALID = 0xFFFFFFFF


def traverse_bvh_tlas(scene, origin, direction, stack_peak=False):
    """rt_gpu_software_query_tlas.hlsl:333-500; returns (t, triangle_id, nodes, tris, instances entered), and with
    stack_peak=True the most entries the stack held at once"""
    org = [f32(x) for x in origin]
    d = [f32(x) for x in direction]
    d = [F32_EPSILON if x == 0.0 else x for x in d]                   # :339
    stack = []
    tlas_stack_size = INVALID                                         # :343
    current_bvh_offset = scene.tlas_start                             # :344
    oct_inv4 = ray_get_octant_inv4(d)
    current_group = [0, 0x80000000]
    t, triangle_id = F32_MAX, -1
    n_nodes = n_tris = n_inst = peak = 0
    while True:
        if current_group[1] & 0xff000000:
            hits_imask = current_group[1]
            child_index_offset = firstbithigh(hits_imask)
            child_index_base = current_group[0]
            current_group[1] &= ~(1 << child_index_offset) & 0xffffffff
            if current_group[1] & 0xff000000:
                stack.append(list(current_group))
                peak = max(peak, len(stack))
            slot_index = (child_index_offset - 24) ^ (oct_inv4 & 0xff)
            relative_index = bin(hits_imask & ~(0xffffffff << slot_index) & 0xffffffff).count("1")
            node = scene.nodes[current_bvh_offset + child_index_base + relative_index]          # :383
            n_nodes += 1
            hitmask = cwbvh_node_intersect(org, d, oct_inv4, t, node)
            imask = extract_byte(int(node[3]), 3)
            current_group[0] = int(node[4])
            triangle_group = [int(node[5]), hitmask & 0x00ffffff]
            current_group[1] = (hitmask & 0xff000000) | imask
        else:
            triangle_group = list(current_group)
            current_group = [0, 0]
        while triangle_group[1] != 0:
            if tlas_stack_size == INVALID:                                                       # :410: a TLAS leaf = an instance
                local = firstbithigh(triangle_group[1])
                triangle_group[1] &= ~(1 << local) & 0xffffffff
                g = triangle_group[0] + local
                if triangle_group[1] != 0:
                    stack.append(list(triangle_group))                                           # :420-423
                if (current_group[1] & 0xff000000) != 0:
                    stack.append(list(current_group))                                            # :425-428
                peak = max(peak, len(stack))
                tlas_stack_size = len(stack)                                                     # :431
                current_bvh_offset = scene.blas_offsets[g]                                       # :439
                n_inst += 1
                current_group = [0, 0x80000000]                                                  # :443
                break
            local = firstbithigh(triangle_group[1])
            triangle_group[1] &= ~(1 << local) & 0xffffffff
            g = triangle_group[0] + local
            rec = scene.tris[g]
            n_tris += 1
            tt = intersect_ray_tri(org, d, rec[0:3], rec[4:7], rec[8:11], t)
            if tt is not None:
                t, triangle_id = tt, g
        if (current_group[1] & 0xff000000) == 0:
            if not stack:
                break
            if len(stack) == tlas_stack_size:                                                    # :480-484
                tlas_stack_size = INVALID
                current_bvh_offset = scene.tlas_start
            current_group = stack.pop()
    return (t, triangle_id, n_nodes, n_tris, n_inst) + ((peak,) if stack_peak else ())
